// graph_prep.cu -- once-per-forward integer work: CSR-by-row of the edge list.
//
// The reference re-gathers with the unsorted int64 edge_index in every layer and reduces
// with scatter_add (models/FastEGNN.py:182,210,279-294).  Here the edges are stably sorted
// by row ONCE (bit-identical to torch.sort(row, stable=True)), indices narrowed to int32,
// edge attributes gathered into sorted order, and the clamped counts of
// unsorted_segment_mean (:294) / global_mean_pool turned into reciprocal vectors.
//
// Sort: least-significant-digit radix sort, 8-bit digits, ceil(bits(N-1)/8) passes.
// Each pass = per-tile histogram -> exclusive scan (digit-major) -> stable scatter, where a
// tile is 4096 consecutive elements and the in-tile stable rank comes from warp match masks.
// Small edge lists (up to kFusedMaxTiles tiles of 2048: Water-3D has 89) take a shorter chain: smaller tiles, the scan folded into the scatter kernel (each CTA sums the tile histograms below it: 2 launches
// per pass instead of 3) and the CSR emission (perm, row, col, sorted edge_attr) folded into the last scatter.
#include "common.cuh"

namespace fegnn {

constexpr int kSortThreads = 256;
constexpr int kSortItems = 16;                             // rounds per warp
constexpr int kSortTile = kSortThreads * kSortItems;       // 4096
constexpr int kScanChunk = 4096;                           // 256 threads x 16
constexpr int kFusedItems = 8;                             // small edge lists: tiles of 2048 ...
constexpr int kFusedTile = kSortThreads * kFusedItems;
constexpr int kFusedMaxTiles = 128;                        // ... up to this many (E <= 262 144): every CTA of the scatter kernel
                                                           // reads all tile histograms (G^2 KB of L2 traffic: 8 MB at G = 89)

// ---------------------------------------------------------------- exclusive scan (int32)
__global__ void __launch_bounds__(256) scan_block_sums(const int* __restrict__ in, int n, int* __restrict__ sums) {
  __shared__ int red[8];
  const int base = blockIdx.x * kScanChunk;
  int acc = 0;
  for (int i = threadIdx.x; i < kScanChunk; i += 256) {
    int idx = base + i;
    if (idx < n) acc += in[idx];
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < 8; ++w) t += red[w];
    sums[blockIdx.x] = t;
  }
}
// single block: in-place exclusive scan of sums[0..nb)
__global__ void __launch_bounds__(1024) scan_sums(int* __restrict__ sums, int nb) {
  __shared__ int wsum[32];
  __shared__ int carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int base = 0; base < nb; base += 1024) {
    int idx = base + threadIdx.x;
    int v = idx < nb ? sums[idx] : 0;
    int inc = v;
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    if (w == 0) {
      int t = wsum[lane];
      int ti = t;
      for (int o = 1; o < 32; o <<= 1) {
        int u = __shfl_up_sync(0xffffffffu, ti, o);
        if (lane >= o) ti += u;
      }
      wsum[lane] = ti - t;   // exclusive prefix of warp sums
    }
    __syncthreads();
    const int carry = carry_s;
    if (idx < nb) sums[idx] = carry + wsum[w] + inc - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry_s = carry + wsum[w] + inc;
    __syncthreads();
  }
}
// out[i] = exclusive prefix of in (may alias); if total != null and this is the last block, *total = sum
__global__ void __launch_bounds__(256) scan_apply(const int* __restrict__ in, int n, const int* __restrict__ sums,
                                                  int* __restrict__ out, int* __restrict__ total) {
  __shared__ int wsum[8];
  const int base = blockIdx.x * kScanChunk + threadIdx.x * 16;
  int v[16];
  int tsum = 0;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    int idx = base + j;
    v[j] = idx < n ? in[idx] : 0;
    tsum += v[j];
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int inc = tsum;
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) wsum[w] = inc;
  __syncthreads();
  int woff = 0;
  for (int k = 0; k < w; ++k) woff += wsum[k];
  int run = sums[blockIdx.x] + woff + inc - tsum;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    int idx = base + j;
    if (idx < n) out[idx] = run;
    run += v[j];
  }
  if (total != nullptr && blockIdx.x == gridDim.x - 1 && threadIdx.x == 255) *total = run;
}

// One launch for small inputs (n <= 64 K: degree arrays and digit histograms of Water-3D-size graphs): thread t owns
// the contiguous chunk [t*per, (t+1)*per), the block scans the 1024 chunk sums.  in may alias out.
constexpr int kSmallScan = 65536;
__global__ void __launch_bounds__(1024) scan_small(const int* __restrict__ in, int n, int* __restrict__ out,
                                                   int* __restrict__ total) {
  __shared__ int wsum[32];
  const int per = (n + 1023) / 1024;
  const int lo = min(n, (int)threadIdx.x * per), hi = min(n, lo + per);
  int tsum = 0;
  for (int i = lo; i < hi; ++i) tsum += in[i];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int inc = tsum;
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) wsum[w] = inc;
  __syncthreads();
  if (w == 0) {
    int t = wsum[lane], ti = t;
    for (int o = 1; o < 32; o <<= 1) {
      int u = __shfl_up_sync(0xffffffffu, ti, o);
      if (lane >= o) ti += u;
    }
    wsum[lane] = ti - t;
  }
  __syncthreads();
  int run = wsum[w] + inc - tsum;
  for (int i = lo; i < hi; ++i) {       // in[i] is read before out[i] is written: safe when aliased
    const int v = in[i];
    out[i] = run;
    run += v;
  }
  if (total != nullptr && threadIdx.x == 1023) *total = run;
}

// Arrays that fit shared memory (n <= 12 K: the degree array and the digit histograms of a Water-3D-size graph, the
// per-graph counts of any batch): coalesced load into shared memory, per-thread chunk scan there, coalesced store.
constexpr int kSmemScan = 12160;                      // 47.5 KB of static shared memory
__global__ void __launch_bounds__(1024) scan_smem(const int* __restrict__ in, int n, int* __restrict__ out,
                                                  int* __restrict__ total) {
  __shared__ int buf[kSmemScan];
  __shared__ int wsum[32];
  for (int i = threadIdx.x; i < n; i += 1024) buf[i] = in[i];
  __syncthreads();
  const int per = (n + 1023) / 1024;
  const int lo = min(n, (int)threadIdx.x * per), hi = min(n, lo + per);
  int tsum = 0;
  for (int i = lo; i < hi; ++i) tsum += buf[i];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int inc = tsum;
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) wsum[w] = inc;
  __syncthreads();
  if (w == 0) {
    int t = wsum[lane], ti = t;
    for (int o = 1; o < 32; o <<= 1) {
      int u = __shfl_up_sync(0xffffffffu, ti, o);
      if (lane >= o) ti += u;
    }
    wsum[lane] = ti - t;
  }
  __syncthreads();
  int run = wsum[w] + inc - tsum;
  for (int i = lo; i < hi; ++i) {
    const int v = buf[i];
    buf[i] = run;
    run += v;
  }
  if (total != nullptr && threadIdx.x == 1023) *total = run;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += 1024) out[i] = buf[i];
}

static cudaError_t exclusive_scan(const int* in, int n, int* out, int* total, int* sums, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  if (n <= kSmemScan) {
    scan_smem<<<1, 1024, 0, st>>>(in, n, out, total); ++g_launches;
    return cudaGetLastError();
  }
  if (n <= kSmallScan) {
    scan_small<<<1, 1024, 0, st>>>(in, n, out, total); ++g_launches;
    return cudaGetLastError();
  }
  int nb = (n + kScanChunk - 1) / kScanChunk;
  scan_block_sums<<<nb, 256, 0, st>>>(in, n, sums); ++g_launches;
  scan_sums<<<1, 1024, 0, st>>>(sums, nb); ++g_launches;
  scan_apply<<<nb, 256, 0, st>>>(in, n, sums, out, total); ++g_launches;
  return cudaGetLastError();
}

// ---------------------------------------------------------------- counting
__global__ void count_rows_kernel(int E, const int64_t* __restrict__ row64, int* __restrict__ deg) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < E) atomicAdd(deg + (int)row64[e], 1);
}
__global__ void batch_kernel(int N, const int64_t* __restrict__ b64, int* __restrict__ batch, int* __restrict__ cnt) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = i < N ? (int)b64[i] : -1;
  if (i < N) batch[i] = b;
  // data_batch is non-decreasing: a warp usually holds one graph id -> one atomic per run of equal ids, not per node
  const unsigned same = __match_any_sync(0xffffffffu, b);
  if (b >= 0 && (int)(__ffs(same) - 1) == (int)(threadIdx.x & 31)) atomicAdd(cnt + b, __popc(same));
}
__global__ void recip_kernel(int n, const int* __restrict__ ptr, float* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    int c = ptr[i + 1] - ptr[i];
    out[i] = 1.f / (float)(c < 1 ? 1 : c);
  }
}

// ---------------------------------------------------------------- small graphs: the counts chain in two launches
// (1) degree counts and the int32 batch vector + per-graph node counts in one grid; (2) both exclusive scans (rowptr, gptr)
// with their clamped reciprocals (unsorted_segment_mean's count.clamp(min=1), models/FastEGNN.py:294 / global_mean_pool) in
// one two-block launch.  Replaces count_rows, batch, scan, scan, recip, recip (6 launches of a few microseconds each on the
// critical path of the first edge kernel).
__global__ void count_rows_batch_kernel(int E, int N, const int64_t* __restrict__ row64, const int64_t* __restrict__ b64,
                                        int* __restrict__ deg, int* __restrict__ batch, int* __restrict__ cnt) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < E) atomicAdd(deg + (int)row64[i], 1);
  if (i < (N + 31) / 32 * 32) {                  // whole warps: the match below is warp-wide
    const int b = i < N ? (int)b64[i] : -1;
    if (i < N) batch[i] = b;
    // a warp usually holds one graph id -> one atomic per group of equal ids, not per node
    const unsigned same = __match_any_sync(0xffffffffu, b);
    if (b >= 0 && (int)(__ffs(same) - 1) == (int)(threadIdx.x & 31)) atomicAdd(cnt + b, __popc(same));
  }
}
__global__ void __launch_bounds__(1024) scan2_recip_kernel(int* __restrict__ p0, int n0, float* __restrict__ r0,
                                                            int* __restrict__ p1, int n1, float* __restrict__ r1) {
  __shared__ int buf[kSmemScan];
  __shared__ int wsum[32];
  int* io = blockIdx.x == 0 ? p0 : p1;
  const int n = blockIdx.x == 0 ? n0 : n1;
  float* rc = blockIdx.x == 0 ? r0 : r1;
  for (int i = threadIdx.x; i < n; i += 1024) buf[i] = io[i];
  __syncthreads();
  const int per = (n + 1023) / 1024;
  const int lo = min(n, (int)threadIdx.x * per), hi = min(n, lo + per);
  int tsum = 0;
  for (int i = lo; i < hi; ++i) tsum += buf[i];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int inc = tsum;
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) wsum[w] = inc;
  __syncthreads();
  if (w == 0) {
    int t = wsum[lane], ti = t;
    for (int o = 1; o < 32; o <<= 1) {
      int u = __shfl_up_sync(0xffffffffu, ti, o);
      if (lane >= o) ti += u;
    }
    wsum[lane] = ti - t;
  }
  __syncthreads();
  int run = wsum[w] + inc - tsum;
  for (int i = lo; i < hi; ++i) {
    const int v = buf[i];
    buf[i] = run;
    run += v;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += 1024) {
    io[i] = buf[i];
    if (i + 1 < n) {
      const int c = buf[i + 1] - buf[i];
      rc[i] = 1.f / (float)(c < 1 ? 1 : c);
    }
  }
}

// ---------------------------------------------------------------- radix passes
// keys come from the int64 row vector in the first pass (vals implicit = index)
template <bool FIRST>
__global__ void __launch_bounds__(kSortThreads) radix_hist_kernel(int E, int shift, const int64_t* __restrict__ row64,
                                                                  const int* __restrict__ keys, int G,
                                                                  int* __restrict__ hist) {
  __shared__ int h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int base = blockIdx.x * kSortTile;
  for (int i = threadIdx.x; i < kSortTile; i += kSortThreads) {
    int idx = base + i;
    if (idx < E) {
      int k = FIRST ? (int)row64[idx] : keys[idx];
      atomicAdd(&h[(k >> shift) & 255], 1);
    }
  }
  __syncthreads();
  hist[threadIdx.x * G + blockIdx.x] = h[threadIdx.x];
}

template <bool FIRST>
__global__ void __launch_bounds__(kSortThreads) radix_scatter_kernel(int E, int shift,
                                                                     const int64_t* __restrict__ row64,
                                                                     const int* __restrict__ keys,
                                                                     const int* __restrict__ vals, int G,
                                                                     const int* __restrict__ hist_scan,
                                                                     int* __restrict__ keys_out,
                                                                     int* __restrict__ vals_out) {
  __shared__ int wcount[8][256];    // per-warp digit counts, later running offsets
  __shared__ int goff[256];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  for (int i = tid; i < 8 * 256; i += kSortThreads) (&wcount[0][0])[i] = 0;
  goff[tid] = hist_scan[tid * G + blockIdx.x];
  __syncthreads();
  const int wbase = blockIdx.x * kSortTile + w * (kSortItems * 32);
  int k[kSortItems];
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    int idx = wbase + r * 32 + lane;
    k[r] = idx < E ? (FIRST ? (int)row64[idx] : keys[idx]) : -1;
  }
  // phase 1: per-warp digit counts
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    int idx = wbase + r * 32 + lane;
    if (idx < E) atomicAdd(&wcount[w][(k[r] >> shift) & 255], 1);
  }
  __syncthreads();
  // phase 2: exclusive prefix over warps per digit (thread tid owns digit tid)
  {
    int run = 0;
    for (int ww = 0; ww < 8; ++ww) {
      int c = wcount[ww][tid];
      wcount[ww][tid] = run;
      run += c;
    }
  }
  __syncthreads();
  // phase 3: in-order stable ranking, 32 elements per round
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    int idx = wbase + r * 32 + lane;
    const bool valid = idx < E;
    const int d = valid ? ((k[r] >> shift) & 255) : 256 + lane;   // invalid lanes never match
    unsigned m = __match_any_sync(0xffffffffu, d);
    int rank = __popc(m & ((1u << lane) - 1u));
    int pos = 0;
    if (valid) pos = goff[d] + wcount[w][d] + rank;
    __syncwarp();
    if (valid && rank == 0) wcount[w][d] += __popc(m);
    __syncwarp();
    if (valid) {
      keys_out[pos] = k[r];
      vals_out[pos] = FIRST ? idx : vals[idx];
    }
  }
}

// ---------------------------------------------------------------- small edge lists: 2 launches per pass
// histogram of tile b in hist[b * 256 + digit] (tile-major: the scatter kernel's column sums are coalesced)
template <bool FIRST>
__global__ void __launch_bounds__(kSortThreads) radix_hist_fused_kernel(int E, int shift, const int64_t* __restrict__ row64,
                                                                        const int* __restrict__ keys, int* __restrict__ hist) {
  __shared__ int h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int base = blockIdx.x * kFusedTile;
#pragma unroll
  for (int r = 0; r < kFusedItems; ++r) {
    const int idx = base + r * kSortThreads + threadIdx.x;
    if (idx < E) {
      const int k = FIRST ? (int)row64[idx] : keys[idx];
      atomicAdd(&h[(k >> shift) & 255], 1);
    }
  }
  __syncthreads();
  hist[blockIdx.x * 256 + threadIdx.x] = h[threadIdx.x];
}

struct CsrOut {            // last pass: the CSR arrays instead of (key, value) pairs
  const int64_t* col64;
  const float* ea;
  int *perm, *row, *col;
  float* ea_sorted;
  int Fe;
};

template <bool FIRST, bool LAST>
__global__ void __launch_bounds__(kSortThreads) radix_scatter_fused_kernel(int E, int shift, const int64_t* __restrict__ row64,
                                                                           const int* __restrict__ keys,
                                                                           const int* __restrict__ vals, int G,
                                                                           const int* __restrict__ hist,
                                                                           int* __restrict__ keys_out, int* __restrict__ vals_out,
                                                                           CsrOut o) {
  __shared__ int wcount[8][256];    // per-warp digit counts, later running offsets
  __shared__ int goff[256];
  __shared__ int wtot[8];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  for (int i = tid; i < 8 * 256; i += kSortThreads) (&wcount[0][0])[i] = 0;
  const int wbase = blockIdx.x * kFusedTile + w * (kFusedItems * 32);
  // every global load of the thread goes out first: keys, values and -- last pass -- the gathers of the CSR emission
  // (col64[v], edge_attr[v]); they travel under the column sums and the ranking instead of two dependent round trips per round
  int k[kFusedItems], vv[kFusedItems];
#pragma unroll
  for (int r = 0; r < kFusedItems; ++r) {
    const int idx = wbase + r * 32 + lane;
    k[r] = idx < E ? (FIRST ? (int)row64[idx] : keys[idx]) : -1;
    vv[r] = idx < E ? (FIRST ? idx : vals[idx]) : 0;
  }
  constexpr int kEaRegs = 4;                       // edge_attr columns carried in registers (wider: gathered at the store)
  int cc[kFusedItems];
  float ee[kFusedItems][kEaRegs];
  if (LAST) {
#pragma unroll
    for (int r = 0; r < kFusedItems; ++r) {
      const int idx = wbase + r * 32 + lane;
      cc[r] = idx < E ? (int)o.col64[vv[r]] : 0;
#pragma unroll
      for (int f = 0; f < kEaRegs; ++f) ee[r][f] = (idx < E && f < o.Fe) ? o.ea[(size_t)vv[r] * o.Fe + f] : 0.f;
    }
  }
  // the scan, inline: digit `tid` starts at (all smaller digits of every tile) + (this digit in the tiles below).  The column
  // sums over the G tile histograms are split four ways (64 threads x int4 per histogram row, rows b = q mod 4) with 16 loads
  // in flight per thread: the plain one-digit-per-thread walk was G dependent-latency batches, 8 us at Water-3D.
  {
    __shared__ int part[2][4][256];
    const int q = tid >> 6, c4 = tid & 63;
    int4 tot4 = make_int4(0, 0, 0, 0), bel4 = make_int4(0, 0, 0, 0);
    const int4* h4 = reinterpret_cast<const int4*>(hist);
    // Every CTA reads the same G histogram rows: walked in the same order they all hit the same few L2 lines at the same
    // time (65 % of the kernel's samples sat on the first add behind these loads).  Each CTA starts at its own row instead.
    constexpr int kBatch = 16;                     // loads issued back to back before the first add
    const int n4 = (G + 3) / 4, rot = (int)((blockIdx.x * 11u) % (unsigned)n4);
    for (int j0 = 0; j0 < n4; j0 += kBatch) {
      int4 c[kBatch];
      int bb[kBatch];
#pragma unroll
      for (int j = 0; j < kBatch; ++j) {
        int jj = j0 + j + rot;
        jj -= jj >= n4 ? n4 : 0;
        bb[j] = j0 + j < n4 ? q + 4 * jj : G;
        c[j] = bb[j] < G ? __ldcg(h4 + bb[j] * 64 + c4) : make_int4(0, 0, 0, 0);
      }
#pragma unroll
      for (int j = 0; j < kBatch; ++j) {
        const int m = bb[j] < (int)blockIdx.x ? -1 : 0;
        tot4.x += c[j].x; tot4.y += c[j].y; tot4.z += c[j].z; tot4.w += c[j].w;
        bel4.x += c[j].x & m; bel4.y += c[j].y & m; bel4.z += c[j].z & m; bel4.w += c[j].w & m;
      }
    }
    *reinterpret_cast<int4*>(&part[0][q][4 * c4]) = tot4;
    *reinterpret_cast<int4*>(&part[1][q][4 * c4]) = bel4;
    __syncthreads();
    const int tot = part[0][0][tid] + part[0][1][tid] + part[0][2][tid] + part[0][3][tid];
    const int below = part[1][0][tid] + part[1][1][tid] + part[1][2][tid] + part[1][3][tid];
    int inc = tot;
#pragma unroll
    for (int o_ = 1; o_ < 32; o_ <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, inc, o_);
      if (lane >= o_) inc += u;
    }
    if (lane == 31) wtot[w] = inc;
    __syncthreads();
    int wpre = 0;
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) wpre += ww < w ? wtot[ww] : 0;
    goff[tid] = wpre + inc - tot + below;
  }
  // phase 1: per-warp digit counts
#pragma unroll
  for (int r = 0; r < kFusedItems; ++r) {
    const int idx = wbase + r * 32 + lane;
    if (idx < E) atomicAdd(&wcount[w][(k[r] >> shift) & 255], 1);
  }
  __syncthreads();
  // phase 2: exclusive prefix over warps per digit (thread tid owns digit tid)
  {
    int run = 0;
    for (int ww = 0; ww < 8; ++ww) {
      const int c = wcount[ww][tid];
      wcount[ww][tid] = run;
      run += c;
    }
  }
  __syncthreads();
  // phase 3: in-order stable ranking, 32 elements per round
#pragma unroll
  for (int r = 0; r < kFusedItems; ++r) {
    const int idx = wbase + r * 32 + lane;
    const bool valid = idx < E;
    const int d = valid ? ((k[r] >> shift) & 255) : 256 + lane;   // invalid lanes never match
    const unsigned m = __match_any_sync(0xffffffffu, d);
    const int rank = __popc(m & ((1u << lane) - 1u));
    int pos = 0;
    if (valid) pos = goff[d] + wcount[w][d] + rank;
    __syncwarp();
    if (valid && rank == 0) wcount[w][d] += __popc(m);
    __syncwarp();
    if (valid) {
      const int v = vv[r];
      if (LAST) {
        o.perm[pos] = v;
        o.row[pos] = k[r];
        o.col[pos] = cc[r];
#pragma unroll
        for (int f = 0; f < kEaRegs; ++f)
          if (f < o.Fe) o.ea_sorted[(size_t)pos * o.Fe + f] = ee[r][f];
        for (int f = kEaRegs; f < o.Fe; ++f) o.ea_sorted[(size_t)pos * o.Fe + f] = o.ea[(size_t)v * o.Fe + f];
      } else {
        keys_out[pos] = k[r];
        vals_out[pos] = v;
      }
    }
  }
}

__global__ void iota_copy_kernel(int E, const int64_t* __restrict__ row64, int* __restrict__ keys, int* __restrict__ vals) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < E) {
    keys[e] = (int)row64[e];
    vals[e] = e;
  }
}

// ---------------------------------------------------------------- live edge count (fegnn_graph_prep_live)
// The edge list is padded to the capacity E; *n_in is the caller's live count, clamped to [0, E].  Edges past it are never
// read as indices: the live path counts only live rows and sorts from the keys below instead of from the int64 rows.
__device__ __forceinline__ int live_count(int E, const int* n_in) {
  const int n = *n_in;
  return n < 0 ? 0 : (n > E ? E : n);
}
__global__ void count_live_rows_kernel(int E, const int* __restrict__ n_in, const int64_t* __restrict__ row64,
                                       int* __restrict__ deg) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < live_count(E, n_in)) atomicAdd(deg + (int)row64[e], 1);
}
// the first pass's (key, value) pairs: a live edge its row, a padding edge the key N (it sorts after every row); thread 0
// also writes the clamped count (the graph's own word) and flags a count outside [0, E] in the sticky status word
__global__ void live_keys_kernel(int N, int E, const int* __restrict__ n_in, const int64_t* __restrict__ row64,
                                 int* __restrict__ keys, int* __restrict__ vals, int* __restrict__ n_out,
                                 unsigned* __restrict__ status) {
  const int live = live_count(E, n_in);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < E) {
    keys[e] = e < live ? (int)row64[e] : N;
    vals[e] = e;
  }
  if (e == 0) {
    *n_out = live;
    if (*n_in != live) atomicOr(status, FEGNN_LIVE_BAD_COUNT);
  }
}

__global__ void finalize_kernel(int E, int Fe, const int* __restrict__ keys, const int* __restrict__ vals,
                                const int64_t* __restrict__ col64, const float* __restrict__ ea,
                                int* __restrict__ perm, int* __restrict__ row, int* __restrict__ col,
                                float* __restrict__ ea_sorted) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < E) {
    int p = vals[i];
    perm[i] = p;
    row[i] = keys[i];
    col[i] = (int)col64[p];
    for (int f = 0; f < Fe; ++f) ea_sorted[(size_t)i * Fe + f] = ea[(size_t)p * Fe + f];
  }
}

size_t graph_prep_workspace_bytes(int N, int E) {
  size_t G = ((size_t)E + kSortTile - 1) / kSortTile;
  const size_t Gf = ((size_t)E + kFusedTile - 1) / kFusedTile;
  if (Gf <= (size_t)kFusedMaxTiles) G = Gf;                 // the short chain's tile histograms
  size_t nscan = 256 * G > (size_t)N + 1 ? 256 * G : (size_t)N + 1;
  size_t sums = (nscan + kScanChunk - 1) / kScanChunk + 1;
  return ((size_t)4 * E + 256 * G + 2 * sums + 64) * sizeof(int);      // two scan scratch areas: the two chains overlap
}

// n_live_in != nullptr: the live path of fegnn_graph_prep_live (E is the capacity; n_live_out / status as documented there)
cudaError_t graph_prep(int N, int E, int B, int Fe, const int64_t* edge_index, const int64_t* data_batch,
                       const float* edge_attr, int* perm, int* rowptr, int* row, int* col, int* batch, int* gptr,
                       float* ea_sorted, float* dinv, float* inv_nb, void* ws, cudaStream_t st, cudaStream_t st_counts,
                       const int* n_live_in = nullptr, int* n_live_out = nullptr, unsigned* status = nullptr) {
  const bool live = n_live_in != nullptr;
  const int G = (E + kSortTile - 1) / kSortTile;
  const int Gf = (E + kFusedTile - 1) / kFusedTile;
  static const bool fused_ok = getenv("FEGNN_SORT_FUSED") == nullptr || atoi(getenv("FEGNN_SORT_FUSED")) != 0;   // experiment switch
  const int Gh = Gf <= kFusedMaxTiles ? Gf : G;             // tiles whose histograms the workspace holds (as sized above)
  int* keysA = reinterpret_cast<int*>(ws);
  int* keysB = keysA + E;
  int* valsA = keysB + E;
  int* valsB = valsA + E;
  int* hist = valsB + E;
  int* sums = hist + (size_t)256 * Gh;
  cudaError_t e;
  {
    // counts -> rowptr, gptr, reciprocals (stream st_counts, own scan scratch)
    size_t nscan = 256 * (size_t)Gh > (size_t)N + 1 ? 256 * (size_t)Gh : (size_t)N + 1;
    int* sums2 = sums + (nscan + kScanChunk - 1) / kScanChunk + 1;
    cudaStream_t sc = st_counts;
    if ((e = cudaMemsetAsync(rowptr, 0, sizeof(int) * ((size_t)N + 1), sc)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(gptr, 0, sizeof(int) * ((size_t)B + 1), sc)) != cudaSuccess) return e;
    if (fused_ok && N > 0 && B > 0 && N + 1 <= kSmemScan && B + 1 <= kSmemScan) {
      if (live) {       // rows up to the live count; the fused kernel does the batch part alone (E = 0)
        if (E > 0) { count_live_rows_kernel<<<(E + 255) / 256, 256, 0, sc>>>(E, n_live_in, edge_index, rowptr); ++g_launches; }
        count_rows_batch_kernel<<<(N + 255) / 256, 256, 0, sc>>>(0, N, edge_index, data_batch, rowptr, batch, gptr); ++g_launches;
      } else {
        const int n = E > N ? E : N;
        count_rows_batch_kernel<<<(n + 255) / 256, 256, 0, sc>>>(E, N, edge_index, data_batch, rowptr, batch, gptr); ++g_launches;
      }
      scan2_recip_kernel<<<2, 1024, 0, sc>>>(rowptr, N + 1, dinv, gptr, B + 1, inv_nb); ++g_launches;
    } else {
      if (E > 0 && live) { count_live_rows_kernel<<<(E + 255) / 256, 256, 0, sc>>>(E, n_live_in, edge_index, rowptr); ++g_launches; }
      else if (E > 0) { count_rows_kernel<<<(E + 255) / 256, 256, 0, sc>>>(E, edge_index, rowptr); ++g_launches; }
      if (N > 0) { batch_kernel<<<(N + 255) / 256, 256, 0, sc>>>(N, data_batch, batch, gptr); ++g_launches; }
      if ((e = exclusive_scan(rowptr, N + 1, rowptr, nullptr, sums2, sc)) != cudaSuccess) return e;
      if ((e = exclusive_scan(gptr, B + 1, gptr, nullptr, sums2, sc)) != cudaSuccess) return e;
      if (N > 0) { recip_kernel<<<(N + 255) / 256, 256, 0, sc>>>(N, rowptr, dinv); ++g_launches; }
      if (B > 0) { recip_kernel<<<(B + 255) / 256, 256, 0, sc>>>(B, gptr, inv_nb); ++g_launches; }
    }
  }
  // live: the first pass's keys (padding -> N) into keysA / valsA, the clamped count and the status bit; the passes then
  // all read keys from the workspace, on enough bits for the key N
  if (live) {
    live_keys_kernel<<<E > 0 ? (E + 255) / 256 : 1, 256, 0, st>>>(N, E, n_live_in, edge_index, keysA, valsA, n_live_out,
                                                                  status); ++g_launches;
  }
  if (E == 0) return cudaGetLastError();
  // radix sort (row, edge id)
  int bits = 1;
  while (bits < 31 && (1ll << bits) < (long long)(live ? N + 1 : N)) ++bits;
  const int passes = (bits + 7) / 8;
  const int* kin = live ? keysA : nullptr;
  const int* vin = live ? valsA : nullptr;
  int* kout = live ? keysB : keysA;
  int* vout = live ? valsB : valsA;
  if (Gf <= kFusedMaxTiles && fused_ok) {
    // short chain: per pass one histogram launch and one scatter launch that scans for itself; the last one emits the CSR
    const CsrOut o{edge_index + E, edge_attr, perm, row, col, ea_sorted, Fe};
    for (int p = 0; p < passes; ++p) {
      const int shift = 8 * p;
      const bool first = p == 0 && !live, lastp = p == passes - 1;
      if (first) radix_hist_fused_kernel<true><<<Gf, kSortThreads, 0, st>>>(E, shift, edge_index, nullptr, hist);
      else radix_hist_fused_kernel<false><<<Gf, kSortThreads, 0, st>>>(E, shift, nullptr, kin, hist);
      ++g_launches;
      if (first && lastp)
        radix_scatter_fused_kernel<true, true><<<Gf, kSortThreads, 0, st>>>(E, shift, edge_index, nullptr, nullptr, Gf, hist, kout, vout, o);
      else if (first)
        radix_scatter_fused_kernel<true, false><<<Gf, kSortThreads, 0, st>>>(E, shift, edge_index, nullptr, nullptr, Gf, hist, kout, vout, o);
      else if (lastp)
        radix_scatter_fused_kernel<false, true><<<Gf, kSortThreads, 0, st>>>(E, shift, nullptr, kin, vin, Gf, hist, kout, vout, o);
      else
        radix_scatter_fused_kernel<false, false><<<Gf, kSortThreads, 0, st>>>(E, shift, nullptr, kin, vin, Gf, hist, kout, vout, o);
      ++g_launches;
      kin = kout;
      vin = vout;
      kout = (kout == keysA) ? keysB : keysA;
      vout = (vout == valsA) ? valsB : valsA;
    }
    return cudaGetLastError();
  }
  for (int p = 0; p < passes; ++p) {
    const int shift = 8 * p;
    if (p == 0 && !live) radix_hist_kernel<true><<<G, kSortThreads, 0, st>>>(E, shift, edge_index, nullptr, G, hist);
    else radix_hist_kernel<false><<<G, kSortThreads, 0, st>>>(E, shift, nullptr, kin, G, hist);
    ++g_launches;
    if ((e = exclusive_scan(hist, 256 * G, hist, nullptr, sums, st)) != cudaSuccess) return e;
    if (p == 0 && !live)
      radix_scatter_kernel<true><<<G, kSortThreads, 0, st>>>(E, shift, edge_index, nullptr, nullptr, G, hist, kout, vout);
    else
      radix_scatter_kernel<false><<<G, kSortThreads, 0, st>>>(E, shift, nullptr, kin, vin, G, hist, kout, vout);
    ++g_launches;
    kin = kout;
    vin = vout;
    kout = (kout == keysA) ? keysB : keysA;
    vout = (vout == valsA) ? valsB : valsA;
  }
  finalize_kernel<<<(E + 255) / 256, 256, 0, st>>>(E, Fe, kin, vin, edge_index + E, edge_attr, perm, row, col,
                                                    ea_sorted); ++g_launches;
  return cudaGetLastError();
}

}  // namespace fegnn
