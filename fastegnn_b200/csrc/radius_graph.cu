// radius_graph.cu -- on-device graph construction (SURVEY.md 8 f2): radius graph + keep-shortest selection + CSR
// emission in the layout the layer kernels consume, so no edge list ever leaves the GPU and graph_prep's sort of a
// distance-ordered edge list is not needed.
//
// Replaces, per batch of graphs,
//   datasets/simulation/dataset.py:80-82,96-101   radius_graph(loc_0, r) -> cutoff_edge (torch.sort of the edge
//                                                 lengths, keep int(E (1 - cutoff_rate)) shortest) -> torch.norm
//   datasets/nbody/dataset.py:102-113             complete graph, topk shortest          (r = +inf here)
//   datasets/protein/dataset.py:146-156,208-213   10 A contact graph without self loops, same cutoff_edge
// and the CSR-by-row sort that models/FastEGNN.py's scatter chain stands for (graph_prep.cu).
//
// Semantics (restated on the CPU by oracle/radius_graph_oracle.py, bit for bit):
//   candidates  ordered pairs (i, j), i != j, same graph, d2 < r*r with
//               d2 = (dx*dx + dy*dy) + dz*dz in fp32, round-to-nearest, no fused multiply-add; dist = sqrtf(d2)
//   selection   per graph, the k_b = int(E_b * keep_frac) candidates that come first in the order
//               (dist, col, row) -- i.e. ascending length with ties in the order a stable sort of an edge list grouped
//               by target node leaves them (what torch.sort does to torch_cluster's output in cutoff_edge)
//   layout      CSR by row, inside a row ascending (dist, col) == stable sort by row of the distance-ordered list
//
// Search structure: a per-graph cell grid (<= 255 cells per axis, cell side >= r (1 + 2^-10)); nodes are sorted by
// (graph, cell key) with the radix sort of graph_prep.cu; a node scans the 9 runs of 3 x-adjacent cells found by
// binary search in the sorted key array.  Nothing here allocates or synchronises: the candidate count comes back in
// a device counter and the caller sizes the second call from it.
#include "common.cuh"

namespace fegnn {
namespace rg {

constexpr int kCellBits = 8;
constexpr int kCellMax = 255;

__device__ __forceinline__ unsigned f2ord(float f) {
  unsigned b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

struct Grid {          // one per graph
  float lo[3];
  float side[3];
  int n[3];
};

__global__ void bbox_init_kernel(int B, unsigned* __restrict__ lo, unsigned* __restrict__ hi) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 3 * B) {
    lo[i] = 0xffffffffu;
    hi[i] = 0u;
  }
}
__global__ void bbox_kernel(int N, const float* __restrict__ x, const int* __restrict__ batch, unsigned* __restrict__ lo,
                            unsigned* __restrict__ hi) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = i < N;
  const int b = valid ? batch[i] : -1;
  const int b0 = __shfl_sync(0xffffffffu, b, 0);
  const bool uniform = __all_sync(0xffffffffu, b == b0);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    unsigned v = valid ? f2ord(x[(size_t)i * 3 + k]) : 0u;
    if (uniform) {
      if (b0 < 0) continue;
      unsigned mn = v, mx = v;
      for (int o = 16; o > 0; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      }
      if ((threadIdx.x & 31) == 0) {
        atomicMin(lo + b0 * 3 + k, mn);
        atomicMax(hi + b0 * 3 + k, mx);
      }
    } else if (valid) {
      atomicMin(lo + b * 3 + k, v);
      atomicMax(hi + b * 3 + k, v);
    }
  }
}
__global__ void grid_kernel(int B, float r, const unsigned* __restrict__ lo, const unsigned* __restrict__ hi,
                            const int* __restrict__ gptr, Grid* __restrict__ grid) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  Grid g;
  const bool empty = gptr[b + 1] <= gptr[b];
  const float s0 = r * (1.f + 1.f / 1024.f);          // margin over r: cell indices are computed in fp32
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    g.lo[k] = 0.f; g.side[k] = 1.f; g.n[k] = 1;
    if (empty) continue;
    const float l = ord2f(lo[b * 3 + k]), h = ord2f(hi[b * 3 + k]);
    const float ext = h - l;
    g.lo[k] = l;
    if (!(ext > 0.f) || !(s0 < 3.0e38f) || !(ext < 3.0e38f)) continue;     // one cell along this axis
    const float q = ext / s0;
    if (q < (float)kCellMax) {
      g.n[k] = (int)q + 1;
      g.side[k] = s0;
    } else {
      g.n[k] = kCellMax;
      g.side[k] = fmaxf(s0, (ext / (float)kCellMax) * (1.f + 1.f / 1024.f));
    }
  }
  grid[b] = g;
}
__device__ __forceinline__ int cell_of(float v, float lo, float side, int n) {
  if (n <= 1) return 0;
  int c = (int)((v - lo) / side);
  return c < 0 ? 0 : (c > n - 1 ? n - 1 : c);
}
__global__ void cellkey_kernel(int N, const float* __restrict__ x, const int* __restrict__ batch,
                               const Grid* __restrict__ grid, int* __restrict__ key, int* __restrict__ iota) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const Grid g = grid[batch[i]];
  const int cx = cell_of(x[(size_t)i * 3 + 0], g.lo[0], g.side[0], g.n[0]);
  const int cy = cell_of(x[(size_t)i * 3 + 1], g.lo[1], g.side[1], g.n[1]);
  const int cz = cell_of(x[(size_t)i * 3 + 2], g.lo[2], g.side[2], g.n[2]);
  key[i] = (cz << (2 * kCellBits)) | (cy << kCellBits) | cx;
  iota[i] = i;
}
__global__ void gather_int_kernel(int n, const int* __restrict__ idx, const int* __restrict__ src, int* __restrict__ dst) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[idx[i]];
}
// sorted position t -> (x, y, z, node id) and the node's cell key
__global__ void pack_kernel(int N, const int* __restrict__ order, const float* __restrict__ x, const int* __restrict__ key,
                            float4* __restrict__ pk, int* __restrict__ ck) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= N) return;
  const int i = order[t];
  pk[t] = make_float4(x[(size_t)i * 3], x[(size_t)i * 3 + 1], x[(size_t)i * 3 + 2], __int_as_float(i));
  ck[t] = key[i];
}

__device__ __forceinline__ float dist2_rn(float4 a, float4 b) {
  const float dx = __fsub_rn(a.x, b.x), dy = __fsub_rn(a.y, b.y), dz = __fsub_rn(a.z, b.z);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}
__device__ __forceinline__ int lower_bound_int(const int* __restrict__ a, int lo, int hi, int v) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}
__device__ __forceinline__ bool key_less(float da, int ca, float db, int cb) { return da < db || (da == db && ca < cb); }

// in-place ascending (dist, col) order of one row's candidates (thread-private range of global memory)
__device__ void sort_row(float* __restrict__ d, int* __restrict__ c, int n) {
  if (n <= 48) {
    for (int i = 1; i < n; ++i) {
      const float dv = d[i];
      const int cv = c[i];
      int j = i - 1;
      while (j >= 0 && key_less(dv, cv, d[j], c[j])) {
        d[j + 1] = d[j];
        c[j + 1] = c[j];
        --j;
      }
      d[j + 1] = dv;
      c[j + 1] = cv;
    }
    return;
  }
  // heap sort (max-heap on (dist, col))
  auto sift = [&](int root, int end) {
    const float dv = d[root];
    const int cv = c[root];
    int hole = root;
    for (;;) {
      int child = 2 * hole + 1;
      if (child >= end) break;
      if (child + 1 < end && key_less(d[child], c[child], d[child + 1], c[child + 1])) ++child;
      if (!key_less(dv, cv, d[child], c[child])) break;
      d[hole] = d[child];
      c[hole] = c[child];
      hole = child;
    }
    d[hole] = dv;
    c[hole] = cv;
  };
  for (int s = n / 2 - 1; s >= 0; --s) sift(s, n);
  for (int end = n - 1; end > 0; --end) {
    const float dv = d[0];
    const int cv = c[0];
    d[0] = d[end]; c[0] = c[end];
    d[end] = dv; c[end] = cv;
    sift(0, end);
  }
}

// FILL = false: count the candidates of every node; FILL = true: write (col, dist) at the row's offset and order them.
template <bool FILL>
__global__ void __launch_bounds__(128) neighbour_kernel(int N, float r2, const float4* __restrict__ pk,
                                                        const int* __restrict__ ck, const int* __restrict__ batch,
                                                        const int* __restrict__ gptr, const Grid* __restrict__ grid,
                                                        int* __restrict__ deg, const int* __restrict__ cand_rowptr,
                                                        int cap, int* __restrict__ ccol, float* __restrict__ cdist,
                                                        int* __restrict__ crow) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= N) return;
  const float4 me = pk[t];
  const int i = __float_as_int(me.w);
  const int b = batch[i];
  const int s0 = gptr[b], s1 = gptr[b + 1];
  const Grid g = grid[b];
  const int key = ck[t];
  const int cx = key & kCellMax, cy = (key >> kCellBits) & kCellMax, cz = key >> (2 * kCellBits);
  const int x0 = cx > 0 ? cx - 1 : 0, x1 = cx + 1 < g.n[0] ? cx + 1 : g.n[0] - 1;
  int cnt = 0;
  int base = 0, room = 0;
  if (FILL) {
    base = cand_rowptr[i];
    room = cand_rowptr[i + 1] - base;
    if (base + room > cap) room = cap - base < 0 ? 0 : cap - base;       // caller's capacity too small: truncate, never overrun
  }
  for (int zz = cz - 1; zz <= cz + 1; ++zz) {
    if (zz < 0 || zz >= g.n[2]) continue;
    for (int yy = cy - 1; yy <= cy + 1; ++yy) {
      if (yy < 0 || yy >= g.n[1]) continue;
      const int klo = (zz << (2 * kCellBits)) | (yy << kCellBits) | x0;
      const int khi = (zz << (2 * kCellBits)) | (yy << kCellBits) | x1;
      int p = lower_bound_int(ck, s0, s1, klo);
      for (; p < s1 && ck[p] <= khi; ++p) {
        const float4 o = pk[p];
        const int j = __float_as_int(o.w);
        if (j == i) continue;
        const float d2 = dist2_rn(me, o);
        if (d2 < r2) {
          if (FILL) {
            if (cnt < room) {
              ccol[base + cnt] = j;
              cdist[base + cnt] = __fsqrt_rn(d2);
              crow[base + cnt] = i;
            }
          }
          ++cnt;
        }
      }
    }
  }
  if (!FILL) deg[i] = cnt;
  else sort_row(cdist + base, ccol + base, cnt < room ? cnt : room);
}

// ---------------------------------------------------------------- per-graph selection of the k_b first candidates in
// (dist, col, row) order: most-significant-digit radix select over the 96-bit key, 8 bits per pass.
struct Sel {
  unsigned prefix[3];     // digits fixed so far (dist bits, col, row)
  int krem;               // rank of the wanted element among the still-matching candidates
  int kb;                 // candidates to keep in this graph
};
__global__ void sel_init_kernel(int B, double keep_frac, const int* __restrict__ gptr, const int* __restrict__ cand_rowptr,
                                Sel* __restrict__ sel, int* __restrict__ hist) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) {
    const int eb = cand_rowptr[gptr[b + 1]] - cand_rowptr[gptr[b]];
    int kb = (int)((double)eb * keep_frac);             // int(E_b * (1 - cutoff_rate)), datasets/*/dataset.py cutoff_edge
    kb = kb < 0 ? 0 : (kb > eb ? eb : kb);
    Sel s;
    s.prefix[0] = s.prefix[1] = s.prefix[2] = 0u;
    s.krem = kb - 1;
    s.kb = kb;
    sel[b] = s;
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 256 * B; i += gridDim.x * blockDim.x) hist[i] = 0;
}
__device__ __forceinline__ bool sel_matches(const Sel& s, int pass, unsigned w0, unsigned w1, unsigned w2, unsigned& digit) {
  const unsigned w[3] = {w0, w1, w2};
  const int word = pass >> 2, sh = 24 - 8 * (pass & 3);
  for (int k = 0; k < word; ++k)
    if (w[k] != s.prefix[k]) return false;
  const unsigned hi_mask = sh == 24 ? 0u : (0xffffffffu << (sh + 8));
  if ((w[word] & hi_mask) != (s.prefix[word] & hi_mask)) return false;
  digit = (w[word] >> sh) & 255u;
  return true;
}
constexpr int kSelChunk = 2048;
__global__ void __launch_bounds__(256) sel_hist_kernel(int ncand_cap, const int* __restrict__ n_cand, int pass,
                                                       const int* __restrict__ crow, const int* __restrict__ ccol,
                                                       const float* __restrict__ cdist, const int* __restrict__ batch,
                                                       const Sel* __restrict__ sel, int* __restrict__ hist) {
  __shared__ int h[256];
  __shared__ int b0s;
  const int n = min(*n_cand, ncand_cap);
  const int base = blockIdx.x * kSelChunk;
  if (base >= n) return;
  h[threadIdx.x] = 0;
  if (threadIdx.x == 0) b0s = batch[crow[base]];
  __syncthreads();
  const int b0 = b0s;
  for (int e = base + threadIdx.x; e < min(n, base + kSelChunk); e += 256) {
    const int r = crow[e];
    const int b = batch[r];
    const Sel s = sel[b];
    if (s.kb <= 0) continue;
    unsigned digit;
    if (sel_matches(s, pass, __float_as_uint(cdist[e]), (unsigned)ccol[e], (unsigned)r, digit)) {
      if (b == b0) atomicAdd(&h[digit], 1);
      else atomicAdd(hist + b * 256 + digit, 1);
    }
  }
  __syncthreads();
  if (h[threadIdx.x] != 0) atomicAdd(hist + b0 * 256 + threadIdx.x, h[threadIdx.x]);
}
// one warp per graph: find the digit whose bucket holds rank krem, fix it in the prefix, clear the histogram
__global__ void __launch_bounds__(128) sel_pick_kernel(int B, int pass, Sel* __restrict__ sel, int* __restrict__ hist) {
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= B) return;
  int* h = hist + b * 256;
  int v[8], tot = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    v[j] = h[lane * 8 + j];
    tot += v[j];
    h[lane * 8 + j] = 0;
  }
  int inc = tot;
  for (int o = 1; o < 32; o <<= 1) {
    int u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  Sel s = sel[b];
  if (s.kb <= 0) return;
  int run = inc - tot;                       // candidates in lower digits
  int found = -1, before = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (found < 0 && s.krem >= run && s.krem < run + v[j]) {
      found = lane * 8 + j;
      before = run;
    }
    run += v[j];
  }
  const unsigned who = __ballot_sync(0xffffffffu, found >= 0);
  if (who == 0u) return;                     // cannot happen for a consistent state
  const int src = __ffs(who) - 1;
  found = __shfl_sync(0xffffffffu, found, src);
  before = __shfl_sync(0xffffffffu, before, src);
  if (lane == 0) {
    const int word = pass >> 2, sh = 24 - 8 * (pass & 3);
    s.prefix[word] |= (unsigned)found << sh;
    s.krem -= before;
    sel[b] = s;
  }
}
__device__ __forceinline__ bool kept(const Sel& s, float d, int c, int r) {
  if (s.kb <= 0) return false;
  const unsigned w0 = __float_as_uint(d), w1 = (unsigned)c, w2 = (unsigned)r;
  if (w0 != s.prefix[0]) return w0 < s.prefix[0];
  if (w1 != s.prefix[1]) return w1 < s.prefix[1];
  return w2 <= s.prefix[2];
}
// EMIT = false: kept candidates per row -> deg ; EMIT = true: compact the kept candidates into the CSR arrays
template <bool EMIT>
__global__ void compact_kernel(int N, int Fe, int select, int cap, const int* __restrict__ cand_rowptr,
                               const int* __restrict__ ccol, const float* __restrict__ cdist,
                               const int* __restrict__ batch, const Sel* __restrict__ sel, int* __restrict__ deg,
                               const int* __restrict__ rowptr, int out_cap, int* __restrict__ row, int* __restrict__ col,
                               float* __restrict__ ea, float* __restrict__ dinv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  int lo = cand_rowptr[i], hi = cand_rowptr[i + 1];
  if (hi > cap) hi = cap;
  Sel s;
  if (select) s = sel[batch[i]];
  int n = 0;
  const int out = EMIT ? rowptr[i] : 0;
  for (int e = lo; e < hi; ++e) {
    const float d = cdist[e];
    const int c = ccol[e];
    if (select && !kept(s, d, c, i)) continue;
    if (EMIT && out + n < out_cap) {
      row[out + n] = i;
      col[out + n] = c;
      for (int f = 0; f < Fe; ++f) ea[(size_t)(out + n) * Fe + f] = d;
    }
    ++n;
  }
  if (!EMIT) deg[i] = n;
  else if (dinv != nullptr) dinv[i] = 1.f / (float)(n < 1 ? 1 : n);
}

// generic LSD radix sort of (key, val) int pairs on `bits` key bits with the tile kernels of graph_prep.cu;
// returns which of the two buffer pairs holds the result
static cudaError_t sort_pairs(int n, int bits, int* keysA, int* valsA, int* keysB, int* valsB, int* hist, int* sums,
                              int** keys_out, int** vals_out, cudaStream_t st) {
  const int G = (n + kSortTile - 1) / kSortTile;
  int *kin = keysA, *vin = valsA, *kout = keysB, *vout = valsB;
  cudaError_t e;
  for (int shift = 0; shift < bits; shift += 8) {
    radix_hist_kernel<false><<<G, kSortThreads, 0, st>>>(n, shift, nullptr, kin, G, hist); ++g_launches;
    if ((e = exclusive_scan(hist, 256 * G, hist, nullptr, sums, st)) != cudaSuccess) return e;
    radix_scatter_kernel<false><<<G, kSortThreads, 0, st>>>(n, shift, nullptr, kin, vin, G, hist, kout, vout); ++g_launches;
    int* tk = kin; kin = kout; kout = tk;
    int* tv = vin; vin = vout; vout = tv;
  }
  *keys_out = kin;
  *vals_out = vin;
  return cudaGetLastError();
}

struct Workspace {
  int *key, *kA, *vA, *kB, *vB, *ck, *deg, *hist, *sums, *selhist;
  float4* pk;
  unsigned *lo, *hi;
  Grid* grid;
  Sel* sel;
  size_t bytes;
};
static inline size_t up16(size_t v) { return (v + 15) & ~(size_t)15; }
// Carves the workspace; base may be null (size query).
static Workspace carve(void* base, int N, int B) {
  Workspace w;
  uint8_t* p = reinterpret_cast<uint8_t*>(base);
  size_t off = 0;
  auto take = [&](size_t nbytes) {
    uint8_t* q = p ? p + off : nullptr;
    off += up16(nbytes);
    return q;
  };
  const size_t n = (size_t)N, G = (n + kSortTile - 1) / kSortTile;
  const size_t nscan = (256 * G > n + 1 ? 256 * G : n + 1);
  w.pk = reinterpret_cast<float4*>(take(16 * n));
  w.key = reinterpret_cast<int*>(take(4 * n));
  w.kA = reinterpret_cast<int*>(take(4 * n));
  w.vA = reinterpret_cast<int*>(take(4 * n));
  w.kB = reinterpret_cast<int*>(take(4 * n));
  w.vB = reinterpret_cast<int*>(take(4 * n));
  w.ck = reinterpret_cast<int*>(take(4 * n));
  w.deg = reinterpret_cast<int*>(take(4 * (n + 1)));
  w.hist = reinterpret_cast<int*>(take(4 * 256 * (G + 1)));
  w.sums = reinterpret_cast<int*>(take(4 * ((nscan + kScanChunk - 1) / kScanChunk + 2)));
  w.lo = reinterpret_cast<unsigned*>(take(12 * (size_t)(B + 1)));
  w.hi = reinterpret_cast<unsigned*>(take(12 * (size_t)(B + 1)));
  w.grid = reinterpret_cast<Grid*>(take(sizeof(Grid) * (size_t)(B + 1)));
  w.sel = reinterpret_cast<Sel*>(take(sizeof(Sel) * (size_t)(B + 1)));
  w.selhist = reinterpret_cast<int*>(take(4 * 256 * (size_t)(B + 1)));
  w.bytes = off + 64;
  return w;
}

// fegnn_radius_graph_fill_live: the live count out of the uncapped totals, and the sticky overflow bits
__global__ void live_status_kernel(const int* __restrict__ n_cand, int cand_cap, const int* __restrict__ n_edges, int out_cap,
                                   int* __restrict__ n_live, unsigned* __restrict__ status) {
  const int nc = *n_cand, ne = *n_edges;
  *n_live = ne < 0 ? 0 : (ne > out_cap ? out_cap : ne);
  const unsigned bits = (nc > cand_cap ? FEGNN_LIVE_CAND_OVERFLOW : 0u) | (ne > out_cap ? FEGNN_LIVE_EDGE_OVERFLOW : 0u);
  if (bits != 0u) atomicOr(status, bits);
}

}  // namespace rg

size_t radius_graph_workspace_bytes(int N, int B) { return rg::carve(nullptr, N, B).bytes; }

// pass 1: batch / gptr / inv_nb, cell sort, candidate degrees -> cand_rowptr (exclusive scan) and *n_cand
cudaError_t radius_graph_count(int N, int B, const float* x, const int64_t* data_batch, float r, int* batch, int* gptr,
                               float* inv_nb, int* cand_rowptr, int* n_cand, void* ws, cudaStream_t st) {
  using namespace rg;
  Workspace w = carve(ws, N, B);
  cudaError_t e;
  if ((e = cudaMemsetAsync(gptr, 0, sizeof(int) * ((size_t)B + 1), st)) != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(n_cand, 0, sizeof(int), st)) != cudaSuccess) return e;
  if (N > 0) { batch_kernel<<<(N + 255) / 256, 256, 0, st>>>(N, data_batch, batch, gptr); ++g_launches; }
  if ((e = exclusive_scan(gptr, B + 1, gptr, nullptr, w.sums, st)) != cudaSuccess) return e;
  if (B > 0) { recip_kernel<<<(B + 255) / 256, 256, 0, st>>>(B, gptr, inv_nb); ++g_launches; }
  if (N == 0) return cudaMemsetAsync(cand_rowptr, 0, sizeof(int), st);
  bbox_init_kernel<<<(3 * B + 255) / 256, 256, 0, st>>>(B, w.lo, w.hi); ++g_launches;
  bbox_kernel<<<(N + 255) / 256, 256, 0, st>>>(N, x, batch, w.lo, w.hi); ++g_launches;
  grid_kernel<<<(B + 127) / 128, 128, 0, st>>>(B, r, w.lo, w.hi, gptr, w.grid); ++g_launches;
  cellkey_kernel<<<(N + 255) / 256, 256, 0, st>>>(N, x, batch, w.grid, w.key, w.vA); ++g_launches;
  if ((e = cudaMemcpyAsync(w.kA, w.key, sizeof(int) * (size_t)N, cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return e;
  int *ks = nullptr, *vs = nullptr;
  if ((e = sort_pairs(N, 3 * kCellBits, w.kA, w.vA, w.kB, w.vB, w.hist, w.sums, &ks, &vs, st)) != cudaSuccess) return e;
  if (B > 1) {                     // second key: the graph id (stable, so cells stay ordered inside a graph)
    int bits = 1;
    while (bits < 31 && (1ll << bits) < (long long)B) ++bits;
    int* ko = (ks == w.kA) ? w.kB : w.kA;
    int* vo = (vs == w.vA) ? w.vB : w.vA;
    gather_int_kernel<<<(N + 255) / 256, 256, 0, st>>>(N, vs, batch, ks); ++g_launches;     // keys := graph of each node
    if ((e = sort_pairs(N, bits, ks, vs, ko, vo, w.hist, w.sums, &ks, &vs, st)) != cudaSuccess) return e;
  }
  pack_kernel<<<(N + 255) / 256, 256, 0, st>>>(N, vs, x, w.key, w.pk, w.ck); ++g_launches;
  neighbour_kernel<false><<<(N + 127) / 128, 128, 0, st>>>(N, r * r, w.pk, w.ck, batch, gptr, w.grid, cand_rowptr, nullptr, 0,
                                                           nullptr, nullptr, nullptr); ++g_launches;
  if ((e = cudaMemsetAsync(cand_rowptr + N, 0, sizeof(int), st)) != cudaSuccess) return e;
  if ((e = exclusive_scan(cand_rowptr, N + 1, cand_rowptr, n_cand, w.sums, st)) != cudaSuccess) return e;
  return cudaGetLastError();
}

// pass 2 (same workspace, untouched since pass 1): candidates -> selection -> CSR
cudaError_t radius_graph_fill(int N, int B, int Fe, float r, double keep_frac, int cap, const int* batch,
                              const int* gptr, const int* cand_rowptr, const int* n_cand, int* ccol, float* cdist,
                              int* crow, int out_cap, int* rowptr, int* row, int* col, float* edge_attr, float* dinv,
                              int* n_edges, void* ws, cudaStream_t st) {
  using namespace rg;
  Workspace w = carve(ws, N, B);
  cudaError_t e;
  if ((e = cudaMemsetAsync(n_edges, 0, sizeof(int), st)) != cudaSuccess) return e;
  if (N == 0) return cudaMemsetAsync(rowptr, 0, sizeof(int), st);
  neighbour_kernel<true><<<(N + 127) / 128, 128, 0, st>>>(N, r * r, w.pk, w.ck, batch, gptr, w.grid, nullptr, cand_rowptr, cap,
                                                          ccol, cdist, crow); ++g_launches;
  const int select = keep_frac < 1.0 ? 1 : 0;
  if (select && cap > 0) {
    sel_init_kernel<<<(B + 255) / 256, 256, 0, st>>>(B, keep_frac, gptr, cand_rowptr, w.sel, w.selhist); ++g_launches;
    const int blocks = (cap + kSelChunk - 1) / kSelChunk;
    for (int pass = 0; pass < 12; ++pass) {
      sel_hist_kernel<<<blocks, 256, 0, st>>>(cap, n_cand, pass, crow, ccol, cdist, batch, w.sel, w.selhist); ++g_launches;
      sel_pick_kernel<<<(B * 32 + 127) / 128, 128, 0, st>>>(B, pass, w.sel, w.selhist); ++g_launches;
    }
  }
  compact_kernel<false><<<(N + 255) / 256, 256, 0, st>>>(N, Fe, select, cap, cand_rowptr, ccol, cdist, batch, w.sel, rowptr,
                                                         nullptr, 0, nullptr, nullptr, nullptr, nullptr); ++g_launches;
  if ((e = cudaMemsetAsync(rowptr + N, 0, sizeof(int), st)) != cudaSuccess) return e;
  if ((e = exclusive_scan(rowptr, N + 1, rowptr, n_edges, w.sums, st)) != cudaSuccess) return e;
  compact_kernel<true><<<(N + 255) / 256, 256, 0, st>>>(N, Fe, select, cap, cand_rowptr, ccol, cdist, batch, w.sel, nullptr,
                                                        rowptr, out_cap, row, col, edge_attr, dinv); ++g_launches;
  return cudaGetLastError();
}

}  // namespace fegnn
