// edge_kernels.cu -- fused real-edge phase (fp32 FMA formulation).
//
// Replaces models/FastEGNN.py:102-108 (edge_model), :125-129 (phi_x + segment mean
// numerator) and :156 (message aggregation) of the reference, plus their autograd.
// Per-edge tensors never reach HBM: a persistent CTA walks tiles of 128 CSR-sorted
// edges, gathers P[row] / Q[col] / x, runs phi_e and phi_x out of shared memory and
// segment-reduces the results by row.  Backward recomputes the forward per tile.
// Spec: oracle/staged.py edge_fwd / edge_bwd.
#include "common.cuh"

namespace fegnn {

struct EdgeArgs {
  int N, Nl, E, Fe, ld1;
  unsigned flags;
  unsigned exp;      // timing experiments only (env FEGNN_EXP; 0 in production): 1 no gQ scatter, 2 no gP / gx tail, 4 no P / Q gathers
  float eps;
  const int *row, *col;
  const float *ea, *x, *P, *Q;
  const float *w1, *W2, *b2, *W3, *b3, *w4, *wa, *ba;   // w1 = edge_mlp.0.weight (for wq / Wa columns)
  // forward outputs.  The backward writes neither: its edge_attr-gradient instantiations (kEa) take their output and the
  // CSR -> caller edge order map in the same two slots, so the default backward launches keep their argument block.
  // A backward kernel must never read msum / tsum (it would get g_ea / perm), nor a forward kernel g_ea / perm.
  union { float* msum; float* g_ea; };       // g_ea: [E,Fe] dL/d edge_attr in the caller's order, += (one owner per edge)
  union { float* tsum; const int* perm; };   // perm: [E] caller index of CSR edge e, or nullptr (CSR order is the caller's)
  // backward inputs / outputs
  const float *gm, *gt;
  // slab: the deterministic forward's (kDet) tile-boundary row sums, [ntiles][2][kDetSlot] (edge_det_msum); a forward
  // kernel never reads gP
  union { float* gP; float* slab; };
  float *gQ, *gx;
  float *g_w1, *g_W2, *g_b2, *g_W3, *g_b3, *g_w4, *g_wa, *g_ba;
  const int* n_edges;   // FEGNN_F_LIVE_EDGES: the live edge count (device word); E is then the capacity.  Read by kLive only
};

// The live edge count of a kLive kernel, clamped to [0, capacity].  An earlier kernel of the stream may have written the
// word (graph prep, the radius graph): it is not weight-only data, so a kernel reads it once per CTA AFTER pdl_wait(), and
// through L2 (ld.global.cg: no non-coherent load the compiler could hoist above the wait).  The kLive forms then overwrite
// their copy of a.E with it, so every bound below (tile counts, e < a.E, the dynamic tile claim, the deterministic
// boundaries) is the live one, and no row / col / edge_attr entry at or past the live count is read.
__device__ __forceinline__ int live_edges(const EdgeArgs& a) {
  const int n = __ldcg(a.n_edges);
  return n < 0 ? 0 : (n > a.E ? a.E : n);
}

// ---- deterministic forward (kDet): msum / tsum without arrival-order float sums
// Each tile sums its runs of equal row ids in row order.  A run that stays inside the tile is the row's only contribution:
// ONE add into the zero-filled msum / tsum.  A run that continues into the previous or next tile goes to the tile's
// boundary slab instead -- slot 0 for the run that starts at the tile's first edge, slot 1 for the one that ends at its
// last -- and edge_det_fixup_kernel adds the slots of such a row in tile order and stores the total.
constexpr int kDetSlot = 68;      // floats per slot: 64 msum columns, 3 tsum columns, 1 pad (16-byte slots)
inline size_t edge_det_slab_floats(int E) { return (size_t)((E + kTM - 1) / kTM) * 2 * kDetSlot; }

// does the row of this tile's first (last) edge continue from the previous (into the next) tile?
__device__ __forceinline__ bool edge_det_cont_in(const EdgeArgs& a, const int* srow, int tile) {
  return tile > 0 && a.row[tile * kTM - 1] == srow[0];
}
__device__ __forceinline__ bool edge_det_cont_out(const EdgeArgs& a, const int* srow, int tile) {
  const int e1 = (tile + 1) * kTM;
  return e1 < a.E && a.row[e1] == srow[kTM - 1];
}
// msum: thread (c4 = tid & 15, grp = tid >> 4) takes the runs that START in rows 8 grp .. 8 grp + 7 and walks each to its
// end in row order over column quad c4.  mget(rr, c4) = float4 of columns 4 c4 .. 4 c4 + 3 of edge row rr's message.
template <typename MGet>
__device__ __forceinline__ void edge_det_msum(const EdgeArgs& a, const int* srow, int tile, MGet mget) {
  const int c4 = threadIdx.x & 15, grp = threadIdx.x >> 4;
  const bool cin = edge_det_cont_in(a, srow, tile), cout = edge_det_cont_out(a, srow, tile);
  for (int r0 = grp * 8; r0 < grp * 8 + 8; ++r0) {
    const int k = srow[r0];
    if (k < 0 || (r0 > 0 && srow[r0 - 1] == k)) continue;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int r = r0;
    for (; r < kTM && srow[r] == k; ++r) {
      const float4 m = mget(r, c4);
      acc.x += m.x; acc.y += m.y; acc.z += m.z; acc.w += m.w;
    }
    if ((r0 == 0 && cin) || (r == kTM && cout))
      *reinterpret_cast<float4*>(a.slab + ((size_t)tile * 2 + (r0 == 0 ? 0 : 1)) * kDetSlot + c4 * 4) = acc;
    else
      atomicAdd(reinterpret_cast<float4*>(a.msum + (size_t)k * kH + c4 * 4), acc);
  }
}
// tsum: thread t < 128 takes the run that starts at row t, if any.  tget(rr, k) = coordinate k of edge row rr's term.
template <typename TGet>
__device__ __forceinline__ void edge_det_tsum(const EdgeArgs& a, const int* srow, int tile, TGet tget) {
  const int r0 = threadIdx.x;
  if (r0 >= kTM) return;
  const int k = srow[r0];
  if (k < 0 || (r0 > 0 && srow[r0 - 1] == k)) return;
  float acc[3] = {0.f, 0.f, 0.f};
  int r = r0;
  for (; r < kTM && srow[r] == k; ++r) {
#pragma unroll
    for (int j = 0; j < 3; ++j) acc[j] += tget(r, j);
  }
  const bool cross = (r0 == 0 && edge_det_cont_in(a, srow, tile)) || (r == kTM && edge_det_cont_out(a, srow, tile));
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    if (cross) a.slab[((size_t)tile * 2 + (r0 == 0 ? 0 : 1)) * kDetSlot + kH + j] = acc[j];
    else atomicAdd(a.tsum + (size_t)k * 3 + j, acc[j]);
  }
}
// One warp per tile boundary b (between tiles b - 1 and b): if a row r crosses it and b is r's first crossing, r's sums are
// its slot in tile b - 1 plus slot 0 of every following tile it reaches, added in tile order.  Nothing else adds into r.
// kLive: the boundaries of the live count (FEGNN_F_LIVE_EDGES); the grid covers those of the capacity.
template <bool kLive = false>
__global__ void __launch_bounds__(256) edge_det_fixup_kernel(EdgeArgs a) {
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int b = (int)((blockIdx.x * 256u + threadIdx.x) >> 5) + 1;
  int ntiles = (a.E + kTM - 1) / kTM;
  pdl_wait();
  if constexpr (kLive) {
    a.E = live_edges(a);
    ntiles = (a.E + kTM - 1) / kTM;
  }
  if (b >= ntiles) return;
  const int e = b * kTM, s = e - kTM, r = a.row[e];
  if (a.row[e - 1] != r) return;
  if (s > 0 && a.row[s] == r && a.row[s - 1] == r) return;      // r starts before tile b - 1: an earlier boundary's warp
  const int slot = a.row[s] == r ? 0 : 1;                        // r's run in tile b - 1 starts at its first edge
  for (int j = lane; j < kH + 3; j += 32) {
    float acc = a.slab[((size_t)(b - 1) * 2 + slot) * kDetSlot + j];
    for (int t = b;; ++t) {
      acc += a.slab[(size_t)t * 2 * kDetSlot + j];
      if ((t + 1) * kTM >= a.E || a.row[(t + 1) * kTM] != r) break;
    }
    if (j < kH) a.msum[(size_t)r * kH + j] = acc;
    else a.tsum[(size_t)r * 3 + (j - kH)] = acc;
  }
}
template <bool kLive = false>
inline cudaError_t launch_edge_det_fixup(const EdgeArgs& a, cudaStream_t st) {
  const int nb = (a.E + kTM - 1) / kTM - 1;      // tile boundaries
  if (nb <= 0) return cudaSuccess;
  if (cudaError_t e_ = launch_pdl(edge_det_fixup_kernel<kLive>, (nb + 7) / 8, 256, 0, st, a)) return e_;
  return cudaGetLastError();
}

struct EdgeSmemVec {
  float wq[kH], Wa[FEGNN_MAX_FE * kH], b2[kH], b3[kH], w4[kH], wa[kH];
  float ba;
  int srow[kTM], scol[kTM];
  float sq[kTM], snrm[kTM], sd[kTM * 3], sdn[kTM * 3], ss[kTM], sea[kTM * FEGNN_MAX_FE];
  // backward only
  float sgte[kTM * 3], sgs[kTM], sgq[kTM], sgate[kTM];
};

__device__ __forceinline__ void edge_stage_common(const EdgeArgs& a, EdgeSmemVec* v, float* W2s, float* W3s) {
  stage_weight(W2s, a.W2, kH, 0, 1);
  stage_weight(W3s, a.W3, kH, 0, 1);
  stage_vec(v->wq, a.w1 + 2 * kH, kH, a.ld1);
  for (int f = 0; f < a.Fe; ++f) stage_vec(v->Wa + f * kH, a.w1 + 2 * kH + 1 + f, kH, a.ld1);
  stage_vec(v->b2, a.b2, kH);
  stage_vec(v->b3, a.b3, kH);
  stage_vec(v->w4, a.w4, kH);
  if (a.flags & FEGNN_F_ATTENTION) {
    stage_vec(v->wa, a.wa, kH);
    if (threadIdx.x == 0) v->ba = a.ba[0];
  }
}

// Step 1: one thread per edge of the tile -- indices, geometry, edge attributes.
template <bool BWD>
__device__ __forceinline__ void edge_load_geometry(const EdgeArgs& a, EdgeSmemVec* v, int tile) {
  const int t = threadIdx.x;
  if (t < kTM) {
    int e = tile * kTM + t;
    int r = -1, c = 0;
    float d0 = 0, d1 = 0, d2 = 0, q = 0, nrm = 1.f;
    if (e < a.E) {
      r = a.row[e];
      c = a.col[e];
      d0 = a.x[(size_t)r * 3 + 0] - a.x[(size_t)c * 3 + 0];
      d1 = a.x[(size_t)r * 3 + 1] - a.x[(size_t)c * 3 + 1];
      d2 = a.x[(size_t)r * 3 + 2] - a.x[(size_t)c * 3 + 2];
      q = d0 * d0 + d1 * d1 + d2 * d2;
      for (int f = 0; f < a.Fe; ++f) v->sea[t * FEGNN_MAX_FE + f] = a.ea[(size_t)e * a.Fe + f];
    } else {
      for (int f = 0; f < a.Fe; ++f) v->sea[t * FEGNN_MAX_FE + f] = 0.f;   // padded rows multiply into column sums
    }
    v->srow[t] = r;
    v->scol[t] = c;
    v->sq[t] = q;
    v->sd[t * 3 + 0] = d0; v->sd[t * 3 + 1] = d1; v->sd[t * 3 + 2] = d2;
    if (a.flags & FEGNN_F_NORMALIZE) {
      nrm = sqrtf(q) + a.eps;
      float inv = 1.f / nrm;
      d0 *= inv; d1 *= inv; d2 *= inv;
    }
    v->snrm[t] = nrm;
    v->sdn[t * 3 + 0] = d0; v->sdn[t * 3 + 1] = d1; v->sdn[t * 3 + 2] = d2;
    if (BWD) {
      float g0 = 0, g1 = 0, g2 = 0;
      if (r >= 0) {
        g0 = a.gt[(size_t)r * 3 + 0]; g1 = a.gt[(size_t)r * 3 + 1]; g2 = a.gt[(size_t)r * 3 + 2];
      }
      v->sgte[t * 3 + 0] = g0; v->sgte[t * 3 + 1] = g1; v->sgte[t * 3 + 2] = g2;
      v->sgs[t] = d0 * g0 + d1 * g1 + d2 * g2;
    }
  }
}

// Step 2: z1 = P[row] + Q[col] + q wq + Wa a_e ; a1 = silu(z1) (and silu'(z1) for backward).
template <bool BWD>
__device__ __forceinline__ void edge_assemble(const EdgeArgs& a, const EdgeSmemVec* v, float* TA1, float* TD1) {
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float2 wq = *reinterpret_cast<const float2*>(v->wq + 2 * lane);
#pragma unroll 4
  for (int i = 0; i < 16; ++i) {
    const int rr = w * 16 + i;
    const int r = v->srow[rr];
    float2 o = make_float2(0.f, 0.f), od = make_float2(0.f, 0.f);
    if (r >= 0) {
      const int c = v->scol[rr];
      float2 p = *reinterpret_cast<const float2*>(a.P + (size_t)r * kH + 2 * lane);
      float2 qv = *reinterpret_cast<const float2*>(a.Q + (size_t)c * kH + 2 * lane);
      const float q = v->sq[rr];
      float z0 = p.x + qv.x + q * wq.x, z1 = p.y + qv.y + q * wq.y;
      for (int f = 0; f < a.Fe; ++f) {
        float eaf = v->sea[rr * FEGNN_MAX_FE + f];
        float2 wf = *reinterpret_cast<const float2*>(v->Wa + f * kH + 2 * lane);
        z0 = fmaf(eaf, wf.x, z0);
        z1 = fmaf(eaf, wf.y, z1);
      }
      if (BWD) {
        silu_grad_f(z0, o.x, od.x);
        silu_grad_f(z1, o.y, od.y);
      } else {
        o.x = silu_f(z0);
        o.y = silu_f(z1);
      }
    }
    *reinterpret_cast<float2*>(TA1 + rr * kH + 2 * lane) = o;
    if (BWD) *reinterpret_cast<float2*>(TD1 + rr * kH + 2 * lane) = od;
  }
}

constexpr size_t kEdgeFwdSmem = (2 * kWFloats + 2 * kTileFloats) * sizeof(float) + sizeof(EdgeSmemVec);
constexpr size_t kEdgeBwdSmem = (2 * kWFloats + 5 * kTileFloats) * sizeof(float) + sizeof(EdgeSmemVec);

// kDet: msum / tsum through edge_det_msum / edge_det_tsum and the boundary slab (same terms, summed in row order)
// kLive: the live edge count (live_edges) bounds the tiles instead of the capacity a.E
template <bool kDet, bool kLive = false>
__global__ void __launch_bounds__(kThreads, 2) edge_fwd_kernel(EdgeArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* W2s = smem;
  float* W3s = W2s + kWFloats;
  float* T1 = W3s + kWFloats;
  float* T2 = T1 + kTileFloats;
  EdgeSmemVec* v = reinterpret_cast<EdgeSmemVec*>(T2 + kTileFloats);
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15, lane = tid & 31;
  const bool att = a.flags & FEGNN_F_ATTENTION, use_tanh = a.flags & FEGNN_F_TANH;
  edge_stage_common(a, v, W2s, W3s);
  if constexpr (kLive) {
    pdl_wait();
    a.E = live_edges(a);
  }
  const int ntiles = (a.E + kTM - 1) / kTM;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    __syncthreads();   // previous iteration's readers of v / tiles are done; weights staged
    edge_load_geometry<false>(a, v, tile);
    __syncthreads();
    edge_assemble<false>(a, v, T1, nullptr);
    __syncthreads();
    float acc[kRT][4];
    zero_acc(acc);
    gemm_nt(acc, T1, W2s, ty, tx);
    {
      const float4 bb = *reinterpret_cast<const float4*>(v->b2 + tx * 4);
      const float4 wa = att ? *reinterpret_cast<const float4*>(v->wa + tx * 4) : make_float4(0, 0, 0, 0);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        float4 m;
        m.x = silu_f(acc[i][0] + bb.x); m.y = silu_f(acc[i][1] + bb.y);
        m.z = silu_f(acc[i][2] + bb.z); m.w = silu_f(acc[i][3] + bb.w);
        if (att) {
          float part = m.x * wa.x + m.y * wa.y + m.z * wa.z + m.w * wa.w;
          float gate = sigmoid_f(rowsum16(part) + v->ba);
          m.x *= gate; m.y *= gate; m.z *= gate; m.w *= gate;
        }
        *reinterpret_cast<float4*>(T2 + (ty * kRT + i) * kH + tx * 4) = m;
      }
    }
    __syncthreads();
    if constexpr (kDet) edge_det_msum(a, v->srow, tile, [&](int rr, int c4) {
      return *reinterpret_cast<const float4*>(T2 + rr * kH + c4 * 4);
    });
    else tile_segsum_rows(T2, v->srow, a.msum);
    zero_acc(acc);
    gemm_nt(acc, T2, W3s, ty, tx);
    {
      const float4 bb = *reinterpret_cast<const float4*>(v->b3 + tx * 4);
      const float4 w4 = *reinterpret_cast<const float4*>(v->w4 + tx * 4);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        float part = silu_f(acc[i][0] + bb.x) * w4.x + silu_f(acc[i][1] + bb.y) * w4.y +
                     silu_f(acc[i][2] + bb.z) * w4.z + silu_f(acc[i][3] + bb.w) * w4.w;
        float s = rowsum16(part);
        if (use_tanh) s = tanhf(s);
        if (tx == 0) v->ss[ty * kRT + i] = s;
      }
    }
    __syncthreads();
    if constexpr (kDet) {
      edge_det_tsum(a, v->srow, tile, [&](int rr, int k) { return v->sdn[rr * 3 + k] * v->ss[rr]; });
    } else if (tid < kTM) {
      const int r = v->srow[tid];
      const float s = v->ss[tid];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        bool tail;
        float tot = warp_segsum(v->sdn[tid * 3 + c] * s, r, lane, tail);
        if (tail && r >= 0) atomicAdd(a.tsum + (size_t)r * 3 + c, tot);
      }
    }
  }
}

// kEa: also g_ea[perm[e]][f] += sum_k gz1[e][k] Wa[f][k] (edge_attr enters phi_e's first Linear only)
// kLive: the live edge count (live_edges) bounds the tiles instead of the capacity a.E
template <bool kEa, bool kLive = false>
__global__ void __launch_bounds__(kThreads, 1) edge_bwd_kernel(EdgeArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* W2s = smem;
  float* W3s = W2s + kWFloats;
  float* TA1 = W3s + kWFloats;      // a1 = silu(z1)
  float* TD1 = TA1 + kTileFloats;   // silu'(z1), later gz1 in place
  float* TM = TD1 + kTileFloats;    // m (gated), later gz2
  float* TZ2 = TM + kTileFloats;    // z2 pre-activation
  float* TG = TZ2 + kTileFloats;    // gz3
  EdgeSmemVec* v = reinterpret_cast<EdgeSmemVec*>(TG + kTileFloats);
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15, lane = tid & 31, warp = tid >> 5;
  const bool att = a.flags & FEGNN_F_ATTENTION, use_tanh = a.flags & FEGNN_F_TANH,
             norm = a.flags & FEGNN_F_NORMALIZE;
  edge_stage_common(a, v, W2s, W3s);

  float wgW2[4][4], wgW3[4][4];
  zero_wg(wgW2);
  zero_wg(wgW3);
  float cw4[4] = {0, 0, 0, 0}, cb3[4] = {0, 0, 0, 0}, cb2[4] = {0, 0, 0, 0}, cwq[4] = {0, 0, 0, 0},
        cwa[4] = {0, 0, 0, 0};
  float cWa[FEGNN_MAX_FE][4];
#pragma unroll
  for (int f = 0; f < FEGNN_MAX_FE; ++f)
#pragma unroll
    for (int j = 0; j < 4; ++j) cWa[f][j] = 0.f;
  float cba = 0.f;

  if constexpr (kLive) {
    pdl_wait();
    a.E = live_edges(a);
  }
  const int ntiles = (a.E + kTM - 1) / kTM;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    __syncthreads();
    edge_load_geometry<true>(a, v, tile);
    __syncthreads();
    edge_assemble<true>(a, v, TA1, TD1);
    __syncthreads();
    float acc[kRT][4];
    // ---- recompute phi_e second layer
    zero_acc(acc);
    gemm_nt(acc, TA1, W2s, ty, tx);
    {
      const float4 bb = *reinterpret_cast<const float4*>(v->b2 + tx * 4);
      const float4 wa = att ? *reinterpret_cast<const float4*>(v->wa + tx * 4) : make_float4(0, 0, 0, 0);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int rr = ty * kRT + i;
        float4 z = make_float4(acc[i][0] + bb.x, acc[i][1] + bb.y, acc[i][2] + bb.z, acc[i][3] + bb.w);
        float4 m = make_float4(silu_f(z.x), silu_f(z.y), silu_f(z.z), silu_f(z.w));
        if (att) {
          float part = m.x * wa.x + m.y * wa.y + m.z * wa.z + m.w * wa.w;
          float gate = sigmoid_f(rowsum16(part) + v->ba);
          if (tx == 0) v->sgate[rr] = gate;
          m.x *= gate; m.y *= gate; m.z *= gate; m.w *= gate;
        }
        *reinterpret_cast<float4*>(TM + rr * kH + tx * 4) = m;
        *reinterpret_cast<float4*>(TZ2 + rr * kH + tx * 4) = z;
      }
    }
    __syncthreads();
    // ---- recompute phi_x, form gz3
    zero_acc(acc);
    gemm_nt(acc, TM, W3s, ty, tx);
    {
      const float4 bb = *reinterpret_cast<const float4*>(v->b3 + tx * 4);
      const float4 w4 = *reinterpret_cast<const float4*>(v->w4 + tx * 4);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int rr = ty * kRT + i;
        float a3[4], d3[4];
        silu_grad_f(acc[i][0] + bb.x, a3[0], d3[0]);
        silu_grad_f(acc[i][1] + bb.y, a3[1], d3[1]);
        silu_grad_f(acc[i][2] + bb.z, a3[2], d3[2]);
        silu_grad_f(acc[i][3] + bb.w, a3[3], d3[3]);
        float s = rowsum16(a3[0] * w4.x + a3[1] * w4.y + a3[2] * w4.z + a3[3] * w4.w);
        float gs = v->sgs[rr];
        if (use_tanh) {
          s = tanhf(s);
          gs *= (1.f - s * s);
        }
        if (tx == 0) v->ss[rr] = s;
        float4 g;
        g.x = gs * w4.x * d3[0]; g.y = gs * w4.y * d3[1]; g.z = gs * w4.z * d3[2]; g.w = gs * w4.w * d3[3];
        *reinterpret_cast<float4*>(TG + rr * kH + tx * 4) = g;
        cw4[0] = fmaf(gs, a3[0], cw4[0]); cw4[1] = fmaf(gs, a3[1], cw4[1]);
        cw4[2] = fmaf(gs, a3[2], cw4[2]); cw4[3] = fmaf(gs, a3[3], cw4[3]);
        cb3[0] += g.x; cb3[1] += g.y; cb3[2] += g.z; cb3[3] += g.w;
      }
    }
    __syncthreads();
    // ---- dW3 += gz3^T m ; gmm = gm[row] + gz3 W3
    wgrad_acc(wgW3, TG, TM, kTM);
#pragma unroll
    for (int i = 0; i < kRT; ++i) {
      const int r = v->srow[ty * kRT + i];
      float4 g0 = make_float4(0, 0, 0, 0);
      if (r >= 0 && a.gm != nullptr) g0 = *reinterpret_cast<const float4*>(a.gm + (size_t)r * kH + tx * 4);
      acc[i][0] = g0.x; acc[i][1] = g0.y; acc[i][2] = g0.z; acc[i][3] = g0.w;
    }
    gemm_nn(acc, TG, W3s, ty, tx);
    __syncthreads();   // every thread is done reading TM (wgrad) before it is overwritten with gz2
    {
      const float4 wa = att ? *reinterpret_cast<const float4*>(v->wa + tx * 4) : make_float4(0, 0, 0, 0);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int rr = ty * kRT + i;
        const float4 z = *reinterpret_cast<const float4*>(TZ2 + rr * kH + tx * 4);
        float m0[4], d2[4];
        silu_grad_f(z.x, m0[0], d2[0]); silu_grad_f(z.y, m0[1], d2[1]);
        silu_grad_f(z.z, m0[2], d2[2]); silu_grad_f(z.w, m0[3], d2[3]);
        float g[4] = {acc[i][0], acc[i][1], acc[i][2], acc[i][3]};
        if (att) {
          const bool valid = v->srow[rr] >= 0;
          float ggate = rowsum16(g[0] * m0[0] + g[1] * m0[1] + g[2] * m0[2] + g[3] * m0[3]);
          float gate = v->sgate[rr];
          float gpre = valid ? ggate * gate * (1.f - gate) : 0.f;
          g[0] = g[0] * gate + gpre * wa.x; g[1] = g[1] * gate + gpre * wa.y;
          g[2] = g[2] * gate + gpre * wa.z; g[3] = g[3] * gate + gpre * wa.w;
          cwa[0] = fmaf(gpre, m0[0], cwa[0]); cwa[1] = fmaf(gpre, m0[1], cwa[1]);
          cwa[2] = fmaf(gpre, m0[2], cwa[2]); cwa[3] = fmaf(gpre, m0[3], cwa[3]);
          if (tx == 0) cba += gpre;
        }
        float4 o = make_float4(g[0] * d2[0], g[1] * d2[1], g[2] * d2[2], g[3] * d2[3]);
        *reinterpret_cast<float4*>(TM + rr * kH + tx * 4) = o;
        cb2[0] += o.x; cb2[1] += o.y; cb2[2] += o.z; cb2[3] += o.w;
      }
    }
    __syncthreads();
    // ---- dW2 += gz2^T a1 ; gz1 = (gz2 W2) * silu'(z1)
    wgrad_acc(wgW2, TM, TA1, kTM);
    zero_acc(acc);
    gemm_nn(acc, TM, W2s, ty, tx);
    {
      const float4 wq = *reinterpret_cast<const float4*>(v->wq + tx * 4);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int rr = ty * kRT + i;
        float4 d1 = *reinterpret_cast<const float4*>(TD1 + rr * kH + tx * 4);
        float4 g = make_float4(acc[i][0] * d1.x, acc[i][1] * d1.y, acc[i][2] * d1.z, acc[i][3] * d1.w);
        *reinterpret_cast<float4*>(TD1 + rr * kH + tx * 4) = g;
        const float q = v->sq[rr];
        cwq[0] = fmaf(g.x, q, cwq[0]); cwq[1] = fmaf(g.y, q, cwq[1]);
        cwq[2] = fmaf(g.z, q, cwq[2]); cwq[3] = fmaf(g.w, q, cwq[3]);
#pragma unroll
        for (int f = 0; f < FEGNN_MAX_FE; ++f) {
          if (f < a.Fe) {
            const float ef = v->sea[rr * FEGNN_MAX_FE + f];
            cWa[f][0] = fmaf(g.x, ef, cWa[f][0]); cWa[f][1] = fmaf(g.y, ef, cWa[f][1]);
            cWa[f][2] = fmaf(g.z, ef, cWa[f][2]); cWa[f][3] = fmaf(g.w, ef, cWa[f][3]);
          }
        }
        float gq = rowsum16(g.x * wq.x + g.y * wq.y + g.z * wq.z + g.w * wq.w);
        if (tx == 0) v->sgq[rr] = gq;
      }
    }
    __syncthreads();
    // ---- outputs: gP (row segments), gQ (scatter by col), gx (both ends)
    tile_segsum_rows(TD1, v->srow, a.gP);
    {
      const int half = lane >> 4, l16 = lane & 15;
#pragma unroll 2
      for (int i = 0; i < 8; ++i) {
        const int rr = warp * 16 + i * 2 + half;
        if (v->srow[rr] >= 0) {
          float4 g = *reinterpret_cast<const float4*>(TD1 + rr * kH + l16 * 4);
          atomicAdd(reinterpret_cast<float4*>(a.gQ + (size_t)v->scol[rr] * kH + l16 * 4), g);
        }
      }
    }
    if (tid < kTM) {
      const int r = v->srow[tid], c = v->scol[tid];
      const float s = v->ss[tid], gq2 = 2.f * v->sgq[tid];
      const float inv = norm ? 1.f / v->snrm[tid] : 1.f;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        // a self-loop adds +gd and -gd to the same node: skip both (with normalize, 1/nrm is 1e8 there and
        // the two halves would only cancel to rounding)
        float gd = r == c ? 0.f : s * v->sgte[tid * 3 + k] * inv + gq2 * v->sd[tid * 3 + k];
        if (r >= 0 && r != c) atomicAdd(a.gx + (size_t)c * 3 + k, -gd);
        bool tail;
        float tot = warp_segsum(r >= 0 ? gd : 0.f, r, lane, tail);
        if (tail && r >= 0) atomicAdd(a.gx + (size_t)r * 3 + k, tot);
      }
    }
    if constexpr (kEa) {
      const int e = tile * kTM + tid;
      if (tid < kTM && e < a.E) {
        const float* gz = TD1 + tid * kH;
        float* dst = a.g_ea + (size_t)(a.perm != nullptr ? a.perm[e] : e) * a.Fe;
        for (int f = 0; f < a.Fe; ++f) {
          float s = 0.f;
          for (int j = 0; j < kH; ++j) {
            const int k = (j + tid) & (kH - 1);        // rotated start: the 128 row walks hit different banks
            s = fmaf(gz[k], v->Wa[f * kH + k], s);
          }
          dst[f] += s;
        }
      }
    }
  }
  // ---- per-CTA weight-gradient partials -> reference-layout gradients
  wgrad_flush(wgW3, a.g_W3, kH, 0, 1);
  wgrad_flush(wgW2, a.g_W2, kH, 0, 1);
  colsum_flush(cw4, a.g_w4, 1, tx);
  colsum_flush(cb3, a.g_b3, 1, tx);
  colsum_flush(cb2, a.g_b2, 1, tx);
  if (a.g_w1 != nullptr) {
    colsum_flush(cwq, a.g_w1 + 2 * kH, a.ld1, tx);
#pragma unroll
    for (int f = 0; f < FEGNN_MAX_FE; ++f)
      if (f < a.Fe) colsum_flush(cWa[f], a.g_w1 + 2 * kH + 1 + f, a.ld1, tx);
  }
  if (att) {
    colsum_flush(cwa, a.g_wa, 1, tx);
    if (tx == 0 && a.g_ba != nullptr) atomicAdd(a.g_ba, cba);
  }
}

// ---------------------------------------------------------------------------- host side
// kLive: grid from the capacity a.E; the kernel reads the live count
template <bool kDet = false, bool kLive = false>
cudaError_t launch_edge_fwd(const EdgeArgs& a, int sms, cudaStream_t st) {
  static DevOnce attr;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(edge_fwd_kernel<kDet, kLive>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEdgeFwdSmem);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  int ntiles = (a.E + kTM - 1) / kTM;
  if (ntiles == 0) return cudaSuccess;
  int grid = ntiles < 2 * sms ? ntiles : 2 * sms;
  edge_fwd_kernel<kDet, kLive><<<grid, kThreads, kEdgeFwdSmem, st>>>(a); ++g_launches;
  if (cudaError_t e_ = cudaGetLastError()) return e_;
  return kDet ? launch_edge_det_fixup<kLive>(a, st) : cudaSuccess;
}
template <bool kEa = false, bool kLive = false>
cudaError_t launch_edge_bwd(const EdgeArgs& a, int sms, cudaStream_t st) {
  static DevOnce attr;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(edge_bwd_kernel<kEa, kLive>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEdgeBwdSmem);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  int ntiles = (a.E + kTM - 1) / kTM;
  if (ntiles == 0) return cudaSuccess;
  int grid = ntiles < sms ? ntiles : sms;
  edge_bwd_kernel<kEa, kLive><<<grid, kThreads, kEdgeBwdSmem, st>>>(a); ++g_launches;
  return cudaGetLastError();
}

}  // namespace fegnn
