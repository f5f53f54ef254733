// node_kernels.cu -- per-node phases (fp32 FMA formulation).
//
//  node_pre   the h-dependent half of every first Linear whose input the reference builds
//             with torch.cat (models/FastEGNN.py:103,114,159) plus the phi_v / phi_g heads
//             (:139,:142):  P = Ws h + b1, Q = Wt h, Av = V1h h + c1, Uh = U1h h + e1.
//  node_h     phi_h (:153-166) with the first Linear split per source block.
//  embed      embedding_in (:271); graph_xsum feeds xbar of the first layer (:212).
// Spec: oracle/staged.py node_pre / node_pre_bwd / node_h_fwd / node_h_bwd.
#include "common.cuh"

namespace fegnn {

// ------------------------------------------------------------------------------------------- embed
__global__ void embed_fwd_kernel(int N, int Fin, const float* __restrict__ nf, const float* __restrict__ w,
                                 const float* __restrict__ b, float* __restrict__ h) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)N * kH) return;
  int i = (int)(idx >> 6), n = (int)(idx & 63);
  float acc = b[n];
  for (int f = 0; f < Fin; ++f) acc = fmaf(nf[(size_t)i * Fin + f], w[n * Fin + f], acc);
  h[idx] = acc;
}

// A block owns `chunk` consecutive nodes; its four row groups are summed in shared memory before the 64 x (1 + Fin)
// atomics.  The kernel is bound by the latency of its strided row loop, not by the atomics (measured: 16 blocks of 512
// nodes took 72 us on Water-3D, 63 blocks of 128 nodes 26 us), so chunks are SMALL (>= 64 nodes, ~4 blocks per SM).
__global__ void __launch_bounds__(kThreads) embed_bwd_kernel(int N, int Fin, int chunk, const float* __restrict__ nf,
                                                             const float* __restrict__ w,
                                                             const float* __restrict__ gh, float* __restrict__ gw,
                                                             float* __restrict__ gb, float* __restrict__ gnf) {
  __shared__ float red[3][17][kH];
  const int n = threadIdx.x & 63, grp = threadIdx.x >> 6;
  const int i0 = blockIdx.x * chunk, i1 = min(N, i0 + chunk);
  float aw[16];
#pragma unroll
  for (int f = 0; f < 16; ++f) aw[f] = 0.f;
  float ab = 0.f;
#pragma unroll 16                                // a chunk of 64 nodes = 16 rows per thread: every load in flight at once
  for (int i = i0 + grp; i < i1; i += 4) {
    float g = gh[(size_t)i * kH + n];
    ab += g;
#pragma unroll
    for (int f = 0; f < 16; ++f)
      if (f < Fin) aw[f] = fmaf(g, nf[(size_t)i * Fin + f], aw[f]);
  }
  if (grp > 0) {
    red[grp - 1][16][n] = ab;
#pragma unroll
    for (int f = 0; f < 16; ++f)
      if (f < Fin) red[grp - 1][f][n] = aw[f];
  }
  __syncthreads();
  if (grp == 0) {
    atomicAdd(gb + n, ab + red[0][16][n] + red[1][16][n] + red[2][16][n]);
#pragma unroll
    for (int f = 0; f < 16; ++f)
      if (f < Fin) atomicAdd(gw + n * Fin + f, aw[f] + red[0][f][n] + red[1][f][n] + red[2][f][n]);
  }
  if (gnf != nullptr) {
    for (int idx = threadIdx.x; idx < (i1 - i0) * Fin; idx += kThreads) {
      int i = i0 + idx / Fin, f = idx % Fin;
      float acc = 0.f;
      for (int k = 0; k < kH; ++k) acc = fmaf(gh[(size_t)i * kH + k], w[k * Fin + f], acc);
      gnf[(size_t)i * Fin + f] = acc;
    }
  }
}

__global__ void graph_xsum_kernel(int N, const float* __restrict__ x, const int* __restrict__ batch,
                                  float* __restrict__ xsum) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  int key = i < N ? batch[i] : -1;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float v = i < N ? x[(size_t)i * 3 + k] : 0.f;
    bool tail;
    float tot = warp_segsum(v, key, lane, tail);
    if (tail && key >= 0) atomicAdd(xsum + (size_t)key * 3 + k, tot);
  }
}

// ---- per-graph sums of the deterministic forward: out_m[b][w] = sum over the nodes i of graph b of X_m[i][w], for up to
// three row-major matrices in one pair of launches (graph_xsum; Usum, Dsum and xsum_new of the virtual forward).  The nodes
// are cut into chunks of K rows, K a function of N alone.  Pass 1, one CTA per chunk, sums each column of the chunk in node
// order per graph run: a graph that lies inside the chunk gets its total stored; a run that continues into the previous or
// next chunk goes to the chunk's slot 0 (run at its first row) or 1 (run at its last).  Pass 2 adds the slots of each graph
// that spans chunks in chunk order -- 8 fixed parts of its chunk range per column, then the 8 part sums in part order -- and
// stores the total.  Graphs without nodes get nothing: the caller zero-fills out.
struct DetSegArgs {
  int N, K, n, Wtot;               // nodes, rows per chunk, matrices, their total width
  const int* batch;                // [N] non-decreasing
  const float* X[3];               // [N][W[m]]
  int W[3];
  float* out[3];                   // [B][W[m]]; remapC[m] = C > 0: column w = 3 c + k goes to [B][3][C] position k C + c
  int remapC[3];
  float* slab;                     // [nchunks][2][Wtot]
};
inline int det_chunk_rows(int N) { return N <= 262144 ? 256 : (N + 1023) / 1024; }     // at most 1 024 chunks
inline size_t det_graph_slab_floats(int N, int Wtot) {
  const int K = det_chunk_rows(N);
  return (size_t)((N + K - 1) / K) * 2 * Wtot;
}
__device__ __forceinline__ void det_graph_store(const DetSegArgs& a, int m, int b, int w, float v) {
  const int C = a.remapC[m];
  a.out[m][(size_t)b * a.W[m] + (C > 0 ? (w % 3) * C + w / 3 : w)] = v;
}
__global__ void __launch_bounds__(256) det_graph_sums_chunk_kernel(DetSegArgs a) {
  pdl_trigger();
  const int j = blockIdx.x, i0 = j * a.K, i1 = min(a.N, i0 + a.K);
  pdl_wait();
  const bool cin = i0 > 0 && a.batch[i0 - 1] == a.batch[i0], cout = i1 < a.N && a.batch[i1] == a.batch[i1 - 1];
  int wbase = 0;
  for (int m = 0; m < a.n; ++m) {
    const int W = a.W[m];
    const float* __restrict__ X = a.X[m];
    for (int w = threadIdx.x; w < W; w += blockDim.x) {
      for (int r0 = i0, r1; r0 < i1; r0 = r1) {
        const int b = a.batch[r0];
        for (r1 = r0 + 1; r1 < i1 && a.batch[r1] == b; ++r1) {}
        float acc = 0.f;
        for (int i = r0; i < r1; ++i) acc += X[(size_t)i * W + w];
        if ((r0 == i0 && cin) || (r1 == i1 && cout)) a.slab[((size_t)j * 2 + (r0 == i0 ? 0 : 1)) * a.Wtot + wbase + w] = acc;
        else det_graph_store(a, m, b, w, acc);
      }
    }
    wbase += W;
  }
}
// grid (chunks - 1, ceil(Wtot / 32)): block (j - 1, y) serves the graph that crosses the boundary in front of chunk j if
// that is its first crossing; thread (col, part) sums part `part` of the graph's slot list in column 32 y + col
__global__ void __launch_bounds__(256) det_graph_sums_fix_kernel(DetSegArgs a) {
  pdl_trigger();
  __shared__ float red[8][32];
  const int j = blockIdx.x + 1, i = j * a.K, s = i - a.K;
  pdl_wait();
  const int b = a.batch[i];
  if (a.batch[i - 1] != b) return;
  if (s > 0 && a.batch[s] == b && a.batch[s - 1] == b) return;     // the graph starts before chunk j - 1
  const int slot = a.batch[s] == b ? 0 : 1;                        // its run in chunk j - 1 starts at that chunk's first row
  int lo = i, hi = a.N;                                             // last node of the graph: batch is non-decreasing
  while (hi - lo > 1) {
    const int mid = lo + (hi - lo) / 2;
    if (a.batch[mid] == b) lo = mid; else hi = mid;
  }
  const int n = lo / a.K - j + 2;                                   // slots: chunk j - 1, then chunks j .. lo / K
  const int col = threadIdx.x & 31, part = threadIdx.x >> 5, w = blockIdx.y * 32 + col;
  float acc = 0.f;
  if (w < a.Wtot) {
    for (int e = part * n / 8; e < (part + 1) * n / 8; ++e) {
      const size_t sl = e == 0 ? (size_t)(j - 1) * 2 + slot : (size_t)(j - 1 + e) * 2;
      acc += a.slab[sl * a.Wtot + w];
    }
  }
  red[part][col] = acc;
  __syncthreads();
  if (part == 0 && w < a.Wtot) {
    float tot = 0.f;
#pragma unroll
    for (int p = 0; p < 8; ++p) tot += red[p][col];
    int m = 0, wl = w;
    while (wl >= a.W[m]) wl -= a.W[m++];
    det_graph_store(a, m, b, wl, tot);
  }
}
// a.slab must hold det_graph_slab_floats(N, Wtot) floats
inline cudaError_t launch_det_graph_sums(DetSegArgs a, cudaStream_t st) {
  if (a.N == 0) return cudaSuccess;
  a.K = det_chunk_rows(a.N);
  a.Wtot = 0;
  for (int m = 0; m < a.n; ++m) a.Wtot += a.W[m];
  const int nch = (a.N + a.K - 1) / a.K;
  if (cudaError_t e_ = launch_pdl(det_graph_sums_chunk_kernel, nch, 256, 0, st, a)) return e_;
  if (nch > 1)
    if (cudaError_t e_ = launch_pdl(det_graph_sums_fix_kernel, dim3(nch - 1, (a.Wtot + 31) / 32), 256, 0, st, a)) return e_;
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------- node_pre
struct NodePreArgs {
  int N, ld1, ldv, ldn;
  unsigned flags;
  const float* h;
  const float *edge_w0, *edge_b0, *edgev_w0, *edgev_b0, *node_w0, *node_b0;
  const float *vel_w0, *vel_b0, *vel_w2, *vel_b2, *grav_w0, *grav_b0, *grav_w2, *grav_b2;
  float *P, *Q, *Av, *Uh, *sv, *sg;
  // backward
  const float *gP, *gQ, *gAv, *gUh, *gsv, *gsg;
  float* gh;
  float *g_edge_w0, *g_edge_b0, *g_edgev_w0, *g_edgev_b0, *g_node_w0, *g_node_b0;
  float *g_vel_w0, *g_vel_b0, *g_vel_w2, *g_vel_b2, *g_grav_w0, *g_grav_b0, *g_grav_w2, *g_grav_b2;
};

// Node attributes (Fa = node_attr_nf > 0): Uh gains the rank-Fa term U1att a_i (columns [off, off + Fa) of node_w0, row
// stride ldn) and the backward adds dU1att = sum_i gUh_i a_i^T.  Only the attribute instantiations of the node_pre kernels
// do anything with these arguments: the <false> kernels are the Fa = 0 code, unchanged.
struct NodeAttrArgs {
  int Fa, ldn;
  const float* a;    // [N, Fa]
  const float* w;    // node_w0 + off
  float* gw;         // g node_w0 + off, or nullptr
};
constexpr int kMaxFa = FEGNN_MAX_FA;
constexpr size_t kAttrWBytes = kMaxFa * kH * sizeof(float);                   // U1att transposed: [f][n]
constexpr size_t kAttrGBytes = (kTM * kMaxFa + kMaxFa * kH) * sizeof(float);  // a tile [128][Fa] + dU1att partials [f][n]

// sW[f * 64 + n] = U1att[n][f]
__device__ __forceinline__ void attr_stage_w(float* __restrict__ sW, const NodeAttrArgs& at, int nt) {
  for (int i = threadIdx.x; i < at.Fa * kH; i += nt) sW[i] = at.w[(size_t)(i & 63) * at.ldn + (i >> 6)];
}
// sum_f a[row][f] * U1att[n][f], fp32 FMA
__device__ __forceinline__ float attr_dot(const NodeAttrArgs& at, const float* __restrict__ sW, int row, int n) {
  float s = 0.f;
  const float* ar = at.a + (size_t)row * at.Fa;
  for (int f = 0; f < at.Fa; ++f) s = fmaf(ar[f], sW[f * kH + n], s);
  return s;
}
// a rows i0 .. i0 + 127 -> sA[r * Fa + f], zero past the end (the gradient rows there are zero, the product must be too)
__device__ __forceinline__ void attr_load_tile(float* __restrict__ sA, const NodeAttrArgs& at, int i0, int nvalid, int nt) {
  for (int i = threadIdx.x; i < kTM * at.Fa; i += nt) sA[i] = i < nvalid * at.Fa ? at.a[(size_t)i0 * at.Fa + i] : 0.f;
}
// dU1att partials over one tile: thread (col = tid & 63, part = tid >> 6) walks rows 32 part .. 32 part + 31 of column col
// of the gradient tile (g(rr, col)); 256 threads
template <typename G>
__device__ __forceinline__ void attr_wgrad_walk(float (&sa)[kMaxFa], const float* __restrict__ sA, int Fa, G g) {
  const int col = threadIdx.x & 63, part = threadIdx.x >> 6;
  for (int rr = part * 32; rr < part * 32 + 32; ++rr) {
    const float x = g(rr, col);
#pragma unroll
    for (int f = 0; f < kMaxFa; ++f)
      if (f < Fa) sa[f] = fmaf(x, sA[rr * Fa + f], sa[f]);
  }
}
// the four row parts add in shared memory (red: [f][64], zeroed by the caller before a barrier), then one atomic per weight
// and CTA.  All threads call.
__device__ __forceinline__ void attr_wgrad_flush(const float (&sa)[kMaxFa], float* __restrict__ red, const NodeAttrArgs& at) {
  const int col = threadIdx.x & 63;
#pragma unroll
  for (int f = 0; f < kMaxFa; ++f)
    if (f < at.Fa) atomicAdd(&red[f * kH + col], sa[f]);
  __syncthreads();
  if (at.gw != nullptr)
    for (int i = threadIdx.x; i < at.Fa * kH; i += blockDim.x) atomicAdd(at.gw + (size_t)(i & 63) * at.ldn + (i >> 6), red[i]);
}

constexpr int kNodePreBlocks = 6;   // P, Q, Av, Uh, vel, grav
constexpr size_t kNodePreFwdSmem = (kWFloats + kTileFloats + 2 * kH) * sizeof(float);

// Work item = (node tile, weight block).  The grid is a multiple of the number of active blocks, so a
// CTA always meets the same block and stages its 64x64 weight once; small N still fills the GPU
// (N = 8000 -> 63 tiles x 6 blocks = 378 CTAs instead of 63; three CTAs per SM hold them in one wave).
__device__ __forceinline__ int node_pre_block_id(int k, bool last, bool grav, bool rf = false) {
  // k-th ACTIVE block -> block id (0 P, 1 Q, 2 Av, 3 Uh, 4 vel, 5 grav)
  if (last && k >= 3) ++k;
  if (rf && k >= 4) ++k;       // FastRF: phi_v acts on |v| (rf_vel_* kernels), not on h
  (void)grav;
  return k;
}

template <bool kAttr>
__global__ void __launch_bounds__(kThreads, 3) node_pre_fwd_kernel(NodePreArgs a, int nactive, NodeAttrArgs at) {
  extern __shared__ __align__(16) float smem[];
  float* Ws = smem;
  float* T0 = Ws + kWFloats;
  float* vec = T0 + kTileFloats;     // head blocks: [0] first-layer bias, [1] output weight
  float* sWa = vec + 2 * kH;         // attribute instantiation: U1att, [f][n]
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const bool grav = a.flags & FEGNN_F_GRAVITY, last = a.flags & FEGNN_F_LAST;
  const int blk = node_pre_block_id(blockIdx.x % nactive, last, grav, a.flags & FEGNN_F_RF);
  const int cta = blockIdx.x / nactive, nctas = gridDim.x / nactive;
  const float* wsrc = blk <= 1 ? a.edge_w0 : blk == 2 ? a.edgev_w0 : blk == 3 ? a.node_w0 : blk == 4 ? a.vel_w0 : a.grav_w0;
  const int ld = blk <= 1 ? a.ld1 : blk == 2 ? a.ldv : blk == 3 ? a.ldn : kH;
  pdl_trigger();
  stage_weight(Ws, wsrc, ld, blk == 1 ? kH : 0, 1);
  if (blk >= 4) {
    stage_vec(vec, blk == 4 ? a.vel_b0 : a.grav_b0, kH);
    stage_vec(vec + kH, blk == 4 ? a.vel_w2 : a.grav_w2, kH);
  }
  if constexpr (kAttr) {
    if (blk == 3) attr_stage_w(sWa, at, kThreads);
  }
  pdl_wait();
  const int ntiles = (a.N + kTM - 1) / kTM;
  for (int tile = cta; tile < ntiles; tile += nctas) {
    const int i0 = tile * kTM, nvalid = min(kTM, a.N - i0);
    __syncthreads();
    load_tile(T0, a.h + (size_t)i0 * kH, kH, nvalid);
    __syncthreads();
    float acc[kRT][4];
    zero_acc(acc);
    gemm_nt(acc, T0, Ws, ty, tx);
    if constexpr (kAttr) {
      if (blk == 3) {
#pragma unroll
        for (int i = 0; i < kRT; ++i) {
          const int r = ty * kRT + i;
          if (r < nvalid) {
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] += attr_dot(at, sWa, i0 + r, tx * 4 + j);
          }
        }
      }
    }
    if (blk < 4) {
      const float* bias = blk == 0 ? a.edge_b0 : blk == 2 ? a.edgev_b0 : blk == 3 ? a.node_b0 : nullptr;
      float* out = blk == 0 ? a.P : blk == 1 ? a.Q : blk == 2 ? a.Av : a.Uh;
      float4 bb = make_float4(0, 0, 0, 0);
      if (bias != nullptr) bb = *reinterpret_cast<const float4*>(bias + tx * 4);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int r = ty * kRT + i;
        if (r < nvalid)
          *reinterpret_cast<float4*>(out + (size_t)(i0 + r) * kH + tx * 4) =
              make_float4(acc[i][0] + bb.x, acc[i][1] + bb.y, acc[i][2] + bb.z, acc[i][3] + bb.w);
      }
    } else {
      const float4 bb = *reinterpret_cast<const float4*>(vec + tx * 4);
      const float4 w = *reinterpret_cast<const float4*>(vec + kH + tx * 4);
      const float b2 = blk == 4 ? a.vel_b2[0] : a.grav_b2[0];
      float* out = blk == 4 ? a.sv : a.sg;
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int r = ty * kRT + i;
        float s = rowsum16(silu_f(acc[i][0] + bb.x) * w.x + silu_f(acc[i][1] + bb.y) * w.y +
                           silu_f(acc[i][2] + bb.z) * w.z + silu_f(acc[i][3] + bb.w) * w.w);
        if (tx == 0 && r < nvalid) out[i0 + r] = s + b2;
      }
    }
  }
}

// dW += G^T A with the column sums of G (bias gradient) on the side.
__device__ __forceinline__ void wgrad_acc_bias(float (&wg)[4][4], float (&bs)[4], const float* __restrict__ G,
                                               const float* __restrict__ A, int nrows) {
  const int tn = threadIdx.x >> 4, tk = threadIdx.x & 15;
#pragma unroll 4
  for (int r = 0; r < nrows; ++r) {
    float4 g = *reinterpret_cast<const float4*>(G + r * kH + tn * 4);
    float4 a = *reinterpret_cast<const float4*>(A + r * kH + tk * 4);
    bs[0] += g.x; bs[1] += g.y; bs[2] += g.z; bs[3] += g.w;
    wg[0][0] = fmaf(g.x, a.x, wg[0][0]); wg[0][1] = fmaf(g.x, a.y, wg[0][1]);
    wg[0][2] = fmaf(g.x, a.z, wg[0][2]); wg[0][3] = fmaf(g.x, a.w, wg[0][3]);
    wg[1][0] = fmaf(g.y, a.x, wg[1][0]); wg[1][1] = fmaf(g.y, a.y, wg[1][1]);
    wg[1][2] = fmaf(g.y, a.z, wg[1][2]); wg[1][3] = fmaf(g.y, a.w, wg[1][3]);
    wg[2][0] = fmaf(g.z, a.x, wg[2][0]); wg[2][1] = fmaf(g.z, a.y, wg[2][1]);
    wg[2][2] = fmaf(g.z, a.z, wg[2][2]); wg[2][3] = fmaf(g.z, a.w, wg[2][3]);
    wg[3][0] = fmaf(g.w, a.x, wg[3][0]); wg[3][1] = fmaf(g.w, a.y, wg[3][1]);
    wg[3][2] = fmaf(g.w, a.z, wg[3][2]); wg[3][3] = fmaf(g.w, a.w, wg[3][3]);
  }
}
__device__ __forceinline__ void bias_flush(const float (&bs)[4], float* __restrict__ dst) {
  if (dst == nullptr) return;
  const int tn = threadIdx.x >> 4, tk = threadIdx.x & 15;
  if (tk == 0) {
#pragma unroll
    for (int j = 0; j < 4; ++j) atomicAdd(dst + tn * 4 + j, bs[j]);
  }
}

constexpr size_t kNodePreBwdSmem = (kWFloats + 2 * kTileFloats + 2 * kH) * sizeof(float);

// gh (in: dL/dh' of the residual, out: dL/dh) += G_blk W_blk ; dW_blk += G_blk^T h.
// Work item = (node tile, block) as in the forward; gh is accumulated with red.global.add.v4.f32.
template <bool kAttr>
__global__ void __launch_bounds__(kThreads, 2) node_pre_bwd_kernel(NodePreArgs a, int nactive, NodeAttrArgs at) {
  extern __shared__ __align__(16) float smem[];
  float* Ws = smem;
  float* Th = Ws + kWFloats;
  float* TG = Th + kTileFloats;
  float* vec = TG + kTileFloats;   // [0] = first-layer bias of a head, [1] = its output weight
  float* sA = vec + 2 * kH;        // attribute instantiation: a tile [128][Fa], then the dU1att partials [f][64]
  float* sRed = sA + kTM * kMaxFa;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const bool grav = a.flags & FEGNN_F_GRAVITY, last = a.gUh == nullptr;
  const int blk = node_pre_block_id(blockIdx.x % nactive, last, grav, a.flags & FEGNN_F_RF);
  const int cta = blockIdx.x / nactive, nctas = gridDim.x / nactive;
  const int ntiles = (a.N + kTM - 1) / kTM;
  const float* G = blk == 0 ? a.gP : blk == 1 ? a.gQ : blk == 2 ? a.gAv : blk == 3 ? a.gUh : nullptr;
  const bool head = blk >= 4;
  const float* wsrc = blk <= 1 ? a.edge_w0 : blk == 2 ? a.edgev_w0 : blk == 3 ? a.node_w0 : blk == 4 ? a.vel_w0 : a.grav_w0;
  const int ld = blk <= 1 ? a.ld1 : blk == 2 ? a.ldv : blk == 3 ? a.ldn : kH;
  const int off = blk == 1 ? kH : 0;
  float* gw = blk <= 1 ? a.g_edge_w0 : blk == 2 ? a.g_edgev_w0 : blk == 3 ? a.g_node_w0 : blk == 4 ? a.g_vel_w0 : a.g_grav_w0;
  float* gb = blk == 0 ? a.g_edge_b0 : blk == 2 ? a.g_edgev_b0 : blk == 3 ? a.g_node_b0
              : blk == 4 ? a.g_vel_b0 : blk == 5 ? a.g_grav_b0 : nullptr;
  const float* gs = blk == 4 ? a.gsv : a.gsg;
  pdl_trigger();
  stage_weight(Ws, wsrc, ld, off, 1);
  if (head) {
    stage_vec(vec, blk == 4 ? a.vel_b0 : a.grav_b0, kH);
    stage_vec(vec + kH, blk == 4 ? a.vel_w2 : a.grav_w2, kH);
  }
  pdl_wait();
  float wg[4][4], bs[4] = {0, 0, 0, 0}, cw2[4] = {0, 0, 0, 0};
  float cb2 = 0.f;
  zero_wg(wg);
  [[maybe_unused]] float sa[kMaxFa];
  if constexpr (kAttr) {
#pragma unroll
    for (int f = 0; f < kMaxFa; ++f) sa[f] = 0.f;
    for (int i = tid; i < kMaxFa * kH; i += kThreads) sRed[i] = 0.f;
  }
  for (int tile = cta; tile < ntiles; tile += nctas) {
    const int i0 = tile * kTM, nvalid = min(kTM, a.N - i0);
    __syncthreads();
    load_tile(Th, a.h + (size_t)i0 * kH, kH, nvalid);
    if (!head) load_tile(TG, G + (size_t)i0 * kH, kH, nvalid);
    if constexpr (kAttr) {
      if (blk == 3) attr_load_tile(sA, at, i0, nvalid, kThreads);
    }
    __syncthreads();
    if constexpr (kAttr) {
      if (blk == 3) attr_wgrad_walk(sa, sA, at.Fa, [&](int rr, int c) { return TG[rr * kH + c]; });
    }
    float acc[kRT][4];
    if (head) {
      // recompute z = W h + b ; G = gs_i * w2 * silu'(z)
      zero_acc(acc);
      gemm_nt(acc, Th, Ws, ty, tx);
      const float4 bb = *reinterpret_cast<const float4*>(vec + tx * 4);
      const float4 w2 = *reinterpret_cast<const float4*>(vec + kH + tx * 4);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int r = ty * kRT + i;
        const float g = r < nvalid ? gs[i0 + r] : 0.f;
        float av[4], dv[4];
        silu_grad_f(acc[i][0] + bb.x, av[0], dv[0]); silu_grad_f(acc[i][1] + bb.y, av[1], dv[1]);
        silu_grad_f(acc[i][2] + bb.z, av[2], dv[2]); silu_grad_f(acc[i][3] + bb.w, av[3], dv[3]);
        *reinterpret_cast<float4*>(TG + r * kH + tx * 4) =
            make_float4(g * w2.x * dv[0], g * w2.y * dv[1], g * w2.z * dv[2], g * w2.w * dv[3]);
        cw2[0] = fmaf(g, av[0], cw2[0]); cw2[1] = fmaf(g, av[1], cw2[1]);
        cw2[2] = fmaf(g, av[2], cw2[2]); cw2[3] = fmaf(g, av[3], cw2[3]);
        if (tx == 0) cb2 += g;
      }
      __syncthreads();
    }
    zero_acc(acc);
    gemm_nn(acc, TG, Ws, ty, tx);
#pragma unroll
    for (int i = 0; i < kRT; ++i) {
      const int r = ty * kRT + i;
      if (r < nvalid)
        atomicAdd(reinterpret_cast<float4*>(a.gh + (size_t)(i0 + r) * kH + tx * 4),
                  make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
    }
    wgrad_acc_bias(wg, bs, TG, Th, kTM);
  }
  wgrad_flush(wg, gw, ld, off, 1);
  bias_flush(bs, gb);
  if (head) {
    colsum_flush(cw2, blk == 4 ? a.g_vel_w2 : a.g_grav_w2, 1, tx);
    float* gb2 = blk == 4 ? a.g_vel_b2 : a.g_grav_b2;
    if (tx == 0 && gb2 != nullptr) atomicAdd(gb2, cb2);
  }
  if constexpr (kAttr) {
    if (blk == 3) attr_wgrad_flush(sa, sRed, at);      // uniform over the CTA
  }
}

// ------------------------------------------------------------------------------------------- node_h
struct NodeHArgs {
  int N, C, ldn;
  const float *h, *Uh, *msum, *dinv, *u;
  const float *node_w0, *node_w2, *node_b2;
  float *zh1, *h_new;
  float* wimg;               // tensor-core forward: operand-tile images of the weight blocks (node_tc.cu)
  // backward
  const float* gh_new;
  float *gzh1, *gm, *gu;
  float *g_node_w0, *g_node_w2, *g_node_b2;
};

// tile of A = rowscale * g[rows] (row stride ld)
__device__ __forceinline__ void load_tile_rowscaled(float* __restrict__ T, const float* __restrict__ g, size_t ld,
                                                    int nvalid, const float* __restrict__ rowscale) {
  for (int i = threadIdx.x; i < kTM * 16; i += kThreads) {
    int r = i >> 4, c4 = i & 15;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < nvalid) {
      v = *reinterpret_cast<const float4*>(g + (size_t)r * ld + c4 * 4);
      float s = rowscale != nullptr ? rowscale[r] : 1.f;       // nullptr: plain sums (FEGNN_F_NODE_SUM)
      v.x *= s; v.y *= s; v.z *= s; v.w *= s;
    }
    *reinterpret_cast<float4*>(T + r * kH + c4 * 4) = v;
  }
}

constexpr size_t kNodeHSmem = (kWFloats + 2 * kTileFloats) * sizeof(float);

// zh1 += [Uh +] W_blk A_blk for one (node tile, K-block) work item; zh1 is zero-filled by the launcher and
// accumulated with red.global.add.v4.f32 (block 0 = message mean + the h term Uh, block 1+c = u[:,c,:]).
// kDet: one CTA per node tile walks the K-blocks in block order, adds each block's product to a running total in
// registers and stores zh1 once (the same terms, in block order).
template <bool kDet>
__global__ void __launch_bounds__(kThreads, 2) node_h_z_kernel(NodeHArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* Ws = smem;
  float* T0 = Ws + kWFloats;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int nblk = a.C + 1;
  const int ntiles = (a.N + kTM - 1) / kTM;
  if constexpr (kDet) {
    pdl_trigger();
    pdl_wait();
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int i0 = tile * kTM, nvalid = min(kTM, a.N - i0);
      float tot[kRT][4];
      for (int blk = 0; blk < nblk; ++blk) {
        __syncthreads();
        if (blk == 0) {
          stage_weight(Ws, a.node_w0, a.ldn, kH, 1);
          load_tile_rowscaled(T0, a.msum + (size_t)i0 * kH, kH, nvalid, a.dinv != nullptr ? a.dinv + i0 : nullptr);
        } else {
          stage_weight(Ws, a.node_w0, a.ldn, 2 * kH + (blk - 1), a.C);
          load_tile(T0, a.u + ((size_t)i0 * a.C + (blk - 1)) * kH, (size_t)a.C * kH, nvalid);
        }
        __syncthreads();
        float acc[kRT][4];
#pragma unroll
        for (int i = 0; i < kRT; ++i) {
          const int r = ty * kRT + i;
          float4 g0 = make_float4(0, 0, 0, 0);
          if (blk == 0 && r < nvalid) g0 = *reinterpret_cast<const float4*>(a.Uh + (size_t)(i0 + r) * kH + tx * 4);
          acc[i][0] = g0.x; acc[i][1] = g0.y; acc[i][2] = g0.z; acc[i][3] = g0.w;
        }
        gemm_nt(acc, T0, Ws, ty, tx);
#pragma unroll
        for (int i = 0; i < kRT; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) tot[i][j] = blk == 0 ? acc[i][j] : tot[i][j] + acc[i][j];
      }
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int r = ty * kRT + i;
        if (r < nvalid)
          *reinterpret_cast<float4*>(a.zh1 + (size_t)(i0 + r) * kH + tx * 4) = make_float4(tot[i][0], tot[i][1], tot[i][2], tot[i][3]);
      }
    }
    return;
  }
  const int blk = blockIdx.x % nblk, cta = blockIdx.x / nblk, nctas = gridDim.x / nblk;
  pdl_trigger();
  if (blk == 0) stage_weight(Ws, a.node_w0, a.ldn, kH, 1);
  else stage_weight(Ws, a.node_w0, a.ldn, 2 * kH + (blk - 1), a.C);
  pdl_wait();
  for (int tile = cta; tile < ntiles; tile += nctas) {
    const int i0 = tile * kTM, nvalid = min(kTM, a.N - i0);
    __syncthreads();
    if (blk == 0) load_tile_rowscaled(T0, a.msum + (size_t)i0 * kH, kH, nvalid, a.dinv != nullptr ? a.dinv + i0 : nullptr);
    else load_tile(T0, a.u + ((size_t)i0 * a.C + (blk - 1)) * kH, (size_t)a.C * kH, nvalid);
    __syncthreads();
    float acc[kRT][4];
#pragma unroll
    for (int i = 0; i < kRT; ++i) {
      const int r = ty * kRT + i;
      float4 g0 = make_float4(0, 0, 0, 0);
      if (blk == 0 && r < nvalid) g0 = *reinterpret_cast<const float4*>(a.Uh + (size_t)(i0 + r) * kH + tx * 4);
      acc[i][0] = g0.x; acc[i][1] = g0.y; acc[i][2] = g0.z; acc[i][3] = g0.w;
    }
    gemm_nt(acc, T0, Ws, ty, tx);
#pragma unroll
    for (int i = 0; i < kRT; ++i) {
      const int r = ty * kRT + i;
      if (r < nvalid)
        atomicAdd(reinterpret_cast<float4*>(a.zh1 + (size_t)(i0 + r) * kH + tx * 4),
                  make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
    }
  }
}

// h' = h + U2 silu(zh1) + e2
__global__ void __launch_bounds__(kThreads, 2) node_h_out_kernel(NodeHArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* Ws = smem;
  float* T0 = Ws + kWFloats;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int ntiles = (a.N + kTM - 1) / kTM;
  pdl_trigger();
  stage_weight(Ws, a.node_w2, kH, 0, 1);
  pdl_wait();
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int i0 = tile * kTM, nvalid = min(kTM, a.N - i0);
    __syncthreads();
    for (int i = tid; i < kTM * 16; i += kThreads) {
      int r = i >> 4, c4 = i & 15;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < nvalid) {
        v = *reinterpret_cast<const float4*>(a.zh1 + (size_t)(i0 + r) * kH + c4 * 4);
        v.x = silu_f(v.x); v.y = silu_f(v.y); v.z = silu_f(v.z); v.w = silu_f(v.w);
      }
      *reinterpret_cast<float4*>(T0 + r * kH + c4 * 4) = v;
    }
    __syncthreads();
    float acc[kRT][4];
    zero_acc(acc);
    gemm_nt(acc, T0, Ws, ty, tx);
    const float4 bb = *reinterpret_cast<const float4*>(a.node_b2 + tx * 4);
#pragma unroll
    for (int i = 0; i < kRT; ++i) {
      const int r = ty * kRT + i;
      if (r < nvalid) {
        float4 hh = *reinterpret_cast<const float4*>(a.h + (size_t)(i0 + r) * kH + tx * 4);
        *reinterpret_cast<float4*>(a.h_new + (size_t)(i0 + r) * kH + tx * 4) =
            make_float4(hh.x + acc[i][0] + bb.x, hh.y + acc[i][1] + bb.y, hh.z + acc[i][2] + bb.z,
                        hh.w + acc[i][3] + bb.w);
      }
    }
  }
}

// backward pass 1: gzh1 = (gh' U2) * silu'(zh1) ; dU2 += gh'^T silu(zh1) ; de2 += sum gh'
__global__ void __launch_bounds__(kThreads, 2) node_h_bwd1_kernel(NodeHArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* Ws = smem;
  float* T0 = Ws + kWFloats;
  float* T1 = T0 + kTileFloats;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int ntiles = (a.N + kTM - 1) / kTM;
  pdl_trigger();
  stage_weight(Ws, a.node_w2, kH, 0, 1);
  pdl_wait();
  float wg[4][4], bs[4] = {0, 0, 0, 0};
  zero_wg(wg);
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int i0 = tile * kTM, nvalid = min(kTM, a.N - i0);
    __syncthreads();
    load_tile(T0, a.gh_new + (size_t)i0 * kH, kH, nvalid);
    for (int i = tid; i < kTM * 16; i += kThreads) {
      int r = i >> 4, c4 = i & 15;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < nvalid) {
        v = *reinterpret_cast<const float4*>(a.zh1 + (size_t)(i0 + r) * kH + c4 * 4);
        v.x = silu_f(v.x); v.y = silu_f(v.y); v.z = silu_f(v.z); v.w = silu_f(v.w);
      }
      *reinterpret_cast<float4*>(T1 + r * kH + c4 * 4) = v;
    }
    __syncthreads();
    float acc[kRT][4];
    zero_acc(acc);
    gemm_nn(acc, T0, Ws, ty, tx);
#pragma unroll
    for (int i = 0; i < kRT; ++i) {
      const int r = ty * kRT + i;
      if (r < nvalid) {
        float4 z = *reinterpret_cast<const float4*>(a.zh1 + (size_t)(i0 + r) * kH + tx * 4);
        float av, d0, d1, d2, d3;
        silu_grad_f(z.x, av, d0); silu_grad_f(z.y, av, d1); silu_grad_f(z.z, av, d2); silu_grad_f(z.w, av, d3);
        *reinterpret_cast<float4*>(a.gzh1 + (size_t)(i0 + r) * kH + tx * 4) =
            make_float4(acc[i][0] * d0, acc[i][1] * d1, acc[i][2] * d2, acc[i][3] * d3);
      }
    }
    wgrad_acc_bias(wg, bs, T0, T1, kTM);
  }
  wgrad_flush(wg, a.g_node_w2, kH, 0, 1);
  bias_flush(bs, a.g_node_b2);
}

// backward pass 2, one (node tile, K-block) work item: block 0 -> gm and dU1a, block 1+c -> gu[:,c,:] and dU1u_c
__global__ void __launch_bounds__(kThreads, 2) node_h_bwd2_kernel(NodeHArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* Ws = smem;
  float* T0 = Ws + kWFloats;
  float* T1 = T0 + kTileFloats;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int nblk = a.C + 1;
  const int blk = blockIdx.x % nblk, cta = blockIdx.x / nblk, nctas = gridDim.x / nblk;
  const int ntiles = (a.N + kTM - 1) / kTM;
  pdl_trigger();
  if (blk == 0) stage_weight(Ws, a.node_w0, a.ldn, kH, 1);
  else stage_weight(Ws, a.node_w0, a.ldn, 2 * kH + (blk - 1), a.C);
  pdl_wait();
  float wg[4][4];
  zero_wg(wg);
  for (int tile = cta; tile < ntiles; tile += nctas) {
    const int i0 = tile * kTM, nvalid = min(kTM, a.N - i0);
    __syncthreads();
    load_tile(T0, a.gzh1 + (size_t)i0 * kH, kH, nvalid);
    if (blk == 0) load_tile_rowscaled(T1, a.msum + (size_t)i0 * kH, kH, nvalid, a.dinv != nullptr ? a.dinv + i0 : nullptr);
    else load_tile(T1, a.u + ((size_t)i0 * a.C + (blk - 1)) * kH, (size_t)a.C * kH, nvalid);
    __syncthreads();
    float acc[kRT][4];
    zero_acc(acc);
    gemm_nn(acc, T0, Ws, ty, tx);
#pragma unroll
    for (int i = 0; i < kRT; ++i) {
      const int r = ty * kRT + i;
      if (r < nvalid) {
        if (blk == 0) {
          const float sc = a.dinv != nullptr ? a.dinv[i0 + r] : 1.f;
          *reinterpret_cast<float4*>(a.gm + (size_t)(i0 + r) * kH + tx * 4) =
              make_float4(acc[i][0] * sc, acc[i][1] * sc, acc[i][2] * sc, acc[i][3] * sc);
        } else {
          *reinterpret_cast<float4*>(a.gu + ((size_t)(i0 + r) * a.C + (blk - 1)) * kH + tx * 4) =
              make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        }
      }
    }
    wgrad_acc(wg, T0, T1, kTM);
  }
  if (blk == 0) wgrad_flush(wg, a.g_node_w0, a.ldn, kH, 1);
  else wgrad_flush(wg, a.g_node_w0, a.ldn, 2 * kH + (blk - 1), a.C);
}

// ------------------------------------------------------------------------------------------- launchers
static inline int persistent_grid(int ntiles, int sms) { return ntiles < sms ? ntiles : sms; }

cudaError_t launch_embed_fwd(int N, int Fin, const float* nf, const float* w, const float* b, float* h,
                             cudaStream_t st) {
  if (N == 0) return cudaSuccess;
  size_t total = (size_t)N * kH;
  embed_fwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(N, Fin, nf, w, b, h); ++g_launches;
  return cudaGetLastError();
}
cudaError_t launch_embed_bwd(int N, int Fin, const float* nf, const float* w, const float* gh, float* gw, float* gb,
                             float* gnf, cudaStream_t st) {
  if (N == 0) return cudaSuccess;
  int chunk = (N + 4 * 148 - 1) / (4 * 148);
  if (chunk < 64) chunk = 64;
  embed_bwd_kernel<<<(N + chunk - 1) / chunk, kThreads, 0, st>>>(N, Fin, chunk, nf, w, gh, gw, gb, gnf); ++g_launches;
  return cudaGetLastError();
}
cudaError_t launch_graph_xsum(int N, const float* x, const int* batch, float* xsum, cudaStream_t st) {
  if (N == 0) return cudaSuccess;
  graph_xsum_kernel<<<(N + 255) / 256, 256, 0, st>>>(N, x, batch, xsum); ++g_launches;
  return cudaGetLastError();
}

#define FEGNN_SET_SMEM(kernel, bytes)                                                                        \
  do {                                                                                                       \
    static DevOnce done_;                                                                               \
    if (!done_.get()) {                                                                                            \
      cudaError_t e_ = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes)); \
      if (e_ != cudaSuccess) return e_;                                                                      \
      done_.set();                                                                                          \
    }                                                                                                        \
  } while (0)

static inline int node_pre_grid(int ntiles, int nactive, int sms, int ctas_per_sm = 2) {
  int per = (ctas_per_sm * sms) / nactive;  // CTAs per block id
  if (per < 1) per = 1;
  if (per > ntiles) per = ntiles;
  return per * nactive;
}
// at != nullptr: the attribute instantiation (Fa > 0 and a Uh block: not the last layer)
cudaError_t launch_node_pre_fwd(const NodePreArgs& a, int sms, cudaStream_t st, const NodeAttrArgs* at = nullptr) {
  FEGNN_SET_SMEM(node_pre_fwd_kernel<false>, kNodePreFwdSmem);
  int ntiles = (a.N + kTM - 1) / kTM;
  if (ntiles == 0) return cudaSuccess;
  const bool grav = a.flags & FEGNN_F_GRAVITY, last = a.flags & FEGNN_F_LAST;
  const int nactive = 4 + (grav ? 2 : 1) - (last ? 1 : 0) - ((a.flags & FEGNN_F_RF) ? 1 : 0);
  if (at != nullptr) {
    FEGNN_SET_SMEM(node_pre_fwd_kernel<true>, kNodePreFwdSmem + kAttrWBytes);
    if (cudaError_t e_ = launch_pdl(node_pre_fwd_kernel<true>, node_pre_grid(ntiles, nactive, sms, 3), kThreads,
                                    kNodePreFwdSmem + kAttrWBytes, st, a, nactive, *at)) return e_;
    return cudaGetLastError();
  }
  if (cudaError_t e_ = launch_pdl(node_pre_fwd_kernel<false>, node_pre_grid(ntiles, nactive, sms, 3), kThreads, kNodePreFwdSmem, st, a, nactive,
                                  NodeAttrArgs{})) return e_;
  return cudaGetLastError();
}
cudaError_t launch_node_pre_bwd(const NodePreArgs& a, int sms, cudaStream_t st, const NodeAttrArgs* at = nullptr) {
  FEGNN_SET_SMEM(node_pre_bwd_kernel<false>, kNodePreBwdSmem);
  int ntiles = (a.N + kTM - 1) / kTM;
  if (ntiles == 0) return cudaSuccess;
  const bool grav = a.flags & FEGNN_F_GRAVITY, last = a.gUh == nullptr;
  const int nactive = 4 + (grav ? 2 : 1) - (last ? 1 : 0) - ((a.flags & FEGNN_F_RF) ? 1 : 0);
  if (at != nullptr) {
    FEGNN_SET_SMEM(node_pre_bwd_kernel<true>, kNodePreBwdSmem + kAttrGBytes);
    if (cudaError_t e_ = launch_pdl(node_pre_bwd_kernel<true>, node_pre_grid(ntiles, nactive, sms), kThreads,
                                    kNodePreBwdSmem + kAttrGBytes, st, a, nactive, *at)) return e_;
    return cudaGetLastError();
  }
  if (cudaError_t e_ = launch_pdl(node_pre_bwd_kernel<false>, node_pre_grid(ntiles, nactive, sms), kThreads, kNodePreBwdSmem, st, a, nactive,
                                  NodeAttrArgs{})) return e_;
  return cudaGetLastError();
}
// kSaved: the saved-only form of a backward's recompute (FEGNN_F_RECOMPUTE): zh1 only -- h' is already in the next layer's
// state, so the write-out kernel (U2 silu(zh1) + e2 and the residual add) does not run
template <bool kDet = false, bool kSaved = false>
cudaError_t launch_node_h_fwd(const NodeHArgs& a, int sms, cudaStream_t st, bool zero = true) {
  FEGNN_SET_SMEM(node_h_z_kernel<kDet>, kNodeHSmem);
  {
    static DevOnce done2_;
    if (!done2_.get()) {
      cudaError_t e_ = cudaFuncSetAttribute(node_h_out_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kNodeHSmem);
      if (e_ != cudaSuccess) return e_;
      done2_.set();
    }
  }
  int ntiles = (a.N + kTM - 1) / kTM;
  if (ntiles == 0) return cudaSuccess;
  cudaError_t e = zero && !kDet ? cudaMemsetAsync(a.zh1, 0, sizeof(float) * kH * (size_t)a.N, st) : cudaSuccess;
  if (e != cudaSuccess) return e;
  const int zgrid = kDet ? persistent_grid(ntiles, 2 * sms) : node_pre_grid(ntiles, a.C + 1, sms);
  if (cudaError_t e_ = launch_pdl(node_h_z_kernel<kDet>, zgrid, kThreads, kNodeHSmem, st, a)) return e_;
  if constexpr (kSaved) return cudaGetLastError();
  if (cudaError_t e_ = launch_pdl(node_h_out_kernel, persistent_grid(ntiles, 2 * sms), kThreads, kNodeHSmem, st, a)) return e_;
  return cudaGetLastError();
}
cudaError_t launch_node_h_bwd(const NodeHArgs& a, int sms, cudaStream_t st) {
  FEGNN_SET_SMEM(node_h_bwd1_kernel, kNodeHSmem);
  {
    static DevOnce done2_;
    if (!done2_.get()) {
      cudaError_t e_ = cudaFuncSetAttribute(node_h_bwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kNodeHSmem);
      if (e_ != cudaSuccess) return e_;
      done2_.set();
    }
  }
  int ntiles = (a.N + kTM - 1) / kTM;
  if (ntiles == 0) return cudaSuccess;
  if (cudaError_t e_ = launch_pdl(node_h_bwd1_kernel, persistent_grid(ntiles, 2 * sms), kThreads, kNodeHSmem, st, a)) return e_;
  if (cudaError_t e_ = launch_pdl(node_h_bwd2_kernel, node_pre_grid(ntiles, a.C + 1, sms), kThreads, kNodeHSmem, st, a)) return e_;
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------- FastRF velocity head
// models/FastRF.py:76-80,135,165: sv_i = w2 . silu(w0 n_i + b0) + b2, n_i = |v_i| (torch.norm, detached), w0 [H,1].
__global__ void __launch_bounds__(256) rf_vel_fwd_kernel(int N, const float* __restrict__ v, const float* __restrict__ w0,
                                                         const float* __restrict__ b0, const float* __restrict__ w2,
                                                         const float* __restrict__ b2, float* __restrict__ sv) {
  __shared__ float sw0[kH], sb0[kH], sw2[kH];
  if (threadIdx.x < kH) {
    sw0[threadIdx.x] = w0[threadIdx.x];
    sb0[threadIdx.x] = b0[threadIdx.x];
    sw2[threadIdx.x] = w2[threadIdx.x];
  }
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const float vx = v[(size_t)i * 3], vy = v[(size_t)i * 3 + 1], vz = v[(size_t)i * 3 + 2];
  const float n = sqrtf(vx * vx + vy * vy + vz * vz);
  float s = b2[0];
#pragma unroll 8
  for (int k = 0; k < kH; ++k) s = fmaf(silu_f(fmaf(sw0[k], n, sb0[k])), sw2[k], s);
  sv[i] = s;
}
// thread (k = tid & 63, lane group = tid >> 6) accumulates column k over a strided subset of the nodes
__global__ void __launch_bounds__(256) rf_vel_bwd_kernel(int N, const float* __restrict__ v, const float* __restrict__ w0,
                                                         const float* __restrict__ b0, const float* __restrict__ w2,
                                                         const float* __restrict__ gsv, float* __restrict__ g_w0,
                                                         float* __restrict__ g_b0, float* __restrict__ g_w2,
                                                         float* __restrict__ g_b2) {
  __shared__ float red[4][3][kH];
  __shared__ float redb[4];
  const int k = threadIdx.x & 63, grp = threadIdx.x >> 6;
  const float wk = w0[k], bk = b0[k], w2k = w2[k];
  float a_w0 = 0.f, a_b0 = 0.f, a_w2 = 0.f, a_b2 = 0.f;
  for (int i = blockIdx.x * 4 + grp; i < N; i += gridDim.x * 4) {
    const float vx = v[(size_t)i * 3], vy = v[(size_t)i * 3 + 1], vz = v[(size_t)i * 3 + 2];
    const float n = sqrtf(vx * vx + vy * vy + vz * vz);
    const float g = gsv[i];
    float act, der;
    silu_grad_f(fmaf(wk, n, bk), act, der);
    a_w2 = fmaf(g, act, a_w2);
    const float t = g * w2k * der;
    a_b0 += t;
    a_w0 = fmaf(t, n, a_w0);
    a_b2 += g;
  }
  red[grp][0][k] = a_w0; red[grp][1][k] = a_b0; red[grp][2][k] = a_w2;
  if (k == 0) redb[grp] = a_b2;
  __syncthreads();
  if (grp == 0) {
    const float s0 = red[0][0][k] + red[1][0][k] + red[2][0][k] + red[3][0][k];
    const float s1 = red[0][1][k] + red[1][1][k] + red[2][1][k] + red[3][1][k];
    const float s2 = red[0][2][k] + red[1][2][k] + red[2][2][k] + red[3][2][k];
    if (g_w0 != nullptr) atomicAdd(g_w0 + k, s0);
    if (g_b0 != nullptr) atomicAdd(g_b0 + k, s1);
    if (g_w2 != nullptr) atomicAdd(g_w2 + k, s2);
    if (k == 0 && g_b2 != nullptr) atomicAdd(g_b2, redb[0] + redb[1] + redb[2] + redb[3]);
  }
}
cudaError_t launch_rf_vel_fwd(int N, const float* v, const float* w0, const float* b0, const float* w2, const float* b2,
                              float* sv, cudaStream_t st) {
  if (N == 0) return cudaSuccess;
  rf_vel_fwd_kernel<<<(N + 255) / 256, 256, 0, st>>>(N, v, w0, b0, w2, b2, sv); ++g_launches;
  return cudaGetLastError();
}
cudaError_t launch_rf_vel_bwd(int N, const float* v, const float* w0, const float* b0, const float* w2, const float* gsv,
                              float* g_w0, float* g_b0, float* g_w2, float* g_b2, int sms, cudaStream_t st) {
  if (N == 0) return cudaSuccess;
  int grid = (N + 3) / 4;
  if (grid > 2 * sms) grid = 2 * sms;
  rf_vel_bwd_kernel<<<grid, 256, 0, st>>>(N, v, w0, b0, w2, gsv, g_w0, g_b0, g_w2, g_b2); ++g_launches;
  return cudaGetLastError();
}

}  // namespace fegnn
