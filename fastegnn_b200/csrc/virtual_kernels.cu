// virtual_kernels.cu -- dense N x C real<->virtual phase (fp32 FMA formulation).
//
// Replaces models/FastEGNN.py:111-119 (edge_mode_virtual), :133-144 (virtual / velocity /
// gravity terms of coord_model_vel), :146-150 (coord_model_virtual) and the pooled sums
// that feed :168-177, plus their autograd.  Rows of a tile are (node, channel) pairs,
// channel fastest, so a tile holds TN = 128 / C whole nodes.  Per-graph partial sums are
// kept in shared memory while a CTA stays inside one graph and flushed with one atomic
// per value when it leaves it.  Spec: oracle/staged.py virtual_fwd / virtual_bwd.
#include "common.cuh"

namespace fegnn {

struct VirtArgs {
  int N, B, C, ldv;            // ldv = 2H+1+C (row stride of edge_mlp_virtual.0.weight)
  unsigned flags;
  float grav[3];
  const int* batch;
  const float *x, *v, *Z, *Av, *G1, *tsum, *dinv, *sv, *sg;
  const float *wv1, *V2, *c2, *Wxv, *bxv, *wxv, *WX, *bX, *wX, *wav, *bav;
  // forward outputs.  The deterministic forward kernels (kDet) form no per-graph sum: Dsum then carries the [N, C, 3] rows
  // D sX that det_graph_sums adds per graph (with u into Usum and x_new into xsum_new)
  float *u, *x_new, *Dsum, *Usum, *xsum_new;
  // backward inputs
  const float *gx_new, *gxsum_next, *gDsum, *gUsum, *gu;
  float* gu_work;              // tensor-core backward: [N,C,H] scratch (total dL/du between its two kernels)
  unsigned* stats;             // tensor-core backward: bound statistics of the edge backward (max|gt| in [0], max|x - x_0| in [2]) or nullptr
  // backward outputs
  float *gAv, *gG1, *gx, *gZ, *gsv, *gsg, *gt;
  float *g_wv1, *g_V2, *g_c2, *g_Wxv, *g_bxv, *g_wxv, *g_WX, *g_bX, *g_wX, *g_wav, *g_bav;
};

struct VirtSmem {
  float vr[kH], c2[kH], bxv[kH], wxv[kH], bX[kH], wX[kH], wav[kH];
  float bav;
  int skey[kTM];     // b*C + c, or -1
  int snode[kTM];    // global node id, or -1
  int sb[kTM];       // graph id of tile-local node jn (first TN entries)
  float sD[kTM * 3], srho[kTM], ssxv[kTM], ssX[kTM];
  float sgxn[kTM * 3], sgsxv[kTM], sgsX[kTM], sgrho[kTM], sgD[kTM * 3], sgate[kTM];
  int b_first, b_last;
  float accBig[FEGNN_MAX_C * kH];     // Usum (fwd) / gG1 (bwd) of the current graph
  float accSmall[3 * FEGNN_MAX_C];    // Dsum (fwd) / gZ (bwd)
  float accX[3];                      // xsum_new (fwd)
};

__device__ __forceinline__ void virt_stage(const VirtArgs& a, VirtSmem* s, float* V2s, float* Wxvs, float* WXs) {
  stage_weight(V2s, a.V2, kH, 0, 1);
  stage_weight(Wxvs, a.Wxv, kH, 0, 1);
  stage_weight(WXs, a.WX, kH, 0, 1);
  stage_vec(s->vr, a.wv1 + 2 * kH, kH, a.ldv);
  stage_vec(s->c2, a.c2, kH);
  stage_vec(s->bxv, a.bxv, kH);
  stage_vec(s->wxv, a.wxv, kH);
  stage_vec(s->bX, a.bX, kH);
  stage_vec(s->wX, a.wX, kH);
  if (a.flags & FEGNN_F_ATTENTION) {
    stage_vec(s->wav, a.wav, kH);
    if (threadIdx.x == 0) s->bav = a.bav[0];
  }
  for (int i = threadIdx.x; i < FEGNN_MAX_C * kH; i += kThreads) s->accBig[i] = 0.f;
  if (threadIdx.x < 3 * FEGNN_MAX_C) s->accSmall[threadIdx.x] = 0.f;
  if (threadIdx.x < 3) s->accX[threadIdx.x] = 0.f;
}

// Flush the per-graph shared accumulators of graph b (if any) and clear them.  All threads.
__device__ __forceinline__ void virt_flush(VirtSmem* s, int b, int C, float* dstBig, float* dstSmall, float* dstX) {
  __syncthreads();
  if (b >= 0) {
    for (int i = threadIdx.x; i < C * kH; i += kThreads) {
      atomicAdd(dstBig + (size_t)b * C * kH + i, s->accBig[i]);
      s->accBig[i] = 0.f;
    }
    if (threadIdx.x < 3 * C) {
      atomicAdd(dstSmall + (size_t)b * 3 * C + threadIdx.x, s->accSmall[threadIdx.x]);
      s->accSmall[threadIdx.x] = 0.f;
    }
    if (dstX != nullptr && threadIdx.x < 3) {
      atomicAdd(dstX + (size_t)b * 3 + threadIdx.x, s->accX[threadIdx.x]);
      s->accX[threadIdx.x] = 0.f;
    }
  }
  __syncthreads();
}

// Geometry of a tile: D = Z[b,:,c] - x_i, rho = |D|, keys.  One thread per (node, channel) row.
template <bool BWD>
__device__ __forceinline__ void virt_geometry(const VirtArgs& a, VirtSmem* s, int tile, int TN) {
  const int t = threadIdx.x, C = a.C;
  if (t < kTM) {
    const int jn = t / C, c = t - jn * C;
    const int i = tile * TN + jn;
    const bool valid = jn < TN && i < a.N;
    int key = -1, node = -1;
    float D0 = 0, D1 = 0, D2 = 0, rho = 0;
    if (valid) {
      const int b = a.batch[i];
      key = b * C + c;
      node = i;
      D0 = a.Z[((size_t)b * 3 + 0) * C + c] - a.x[(size_t)i * 3 + 0];
      D1 = a.Z[((size_t)b * 3 + 1) * C + c] - a.x[(size_t)i * 3 + 1];
      D2 = a.Z[((size_t)b * 3 + 2) * C + c] - a.x[(size_t)i * 3 + 2];
      rho = sqrtf(D0 * D0 + D1 * D1 + D2 * D2);
      if (c == 0) s->sb[jn] = b;
      if (t == 0) s->b_first = b;
      if (c == 0 && (jn == TN - 1 || i == a.N - 1)) s->b_last = b;
      if (BWD) {
        float g0 = a.gx_new[(size_t)i * 3 + 0], g1 = a.gx_new[(size_t)i * 3 + 1], g2 = a.gx_new[(size_t)i * 3 + 2];
        if (a.gxsum_next != nullptr) {
          g0 += a.gxsum_next[(size_t)b * 3 + 0]; g1 += a.gxsum_next[(size_t)b * 3 + 1];
          g2 += a.gxsum_next[(size_t)b * 3 + 2];
        }
        if (c == 0) { s->sgxn[jn * 3 + 0] = g0; s->sgxn[jn * 3 + 1] = g1; s->sgxn[jn * 3 + 2] = g2; }
        s->sgsxv[t] = -(D0 * g0 + D1 * g1 + D2 * g2) / (float)C;
        s->sgsX[t] = D0 * a.gDsum[((size_t)b * 3 + 0) * C + c] + D1 * a.gDsum[((size_t)b * 3 + 1) * C + c] +
                     D2 * a.gDsum[((size_t)b * 3 + 2) * C + c];
      }
    } else if (BWD) {
      s->sgsxv[t] = 0.f;
      s->sgsX[t] = 0.f;
    }
    s->skey[t] = key;
    s->snode[t] = node;
    s->sD[t * 3 + 0] = D0; s->sD[t * 3 + 1] = D1; s->sD[t * 3 + 2] = D2;
    s->srho[t] = rho;
  }
}

// zv1 = Av_i + G1[b,c] + rho vr ; WHAT: 0 -> a1 only, 1 -> a1 and d1, 2 -> d1 only
template <int WHAT>
__device__ __forceinline__ void virt_assemble(const VirtArgs& a, const VirtSmem* s, float* TA1, float* TD1) {
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float2 vr = *reinterpret_cast<const float2*>(s->vr + 2 * lane);
#pragma unroll 4
  for (int i = 0; i < 16; ++i) {
    const int rr = w * 16 + i;
    const int key = s->skey[rr];
    float2 o = make_float2(0.f, 0.f), od = make_float2(0.f, 0.f);
    if (key >= 0) {
      const int node = s->snode[rr];
      float2 p = *reinterpret_cast<const float2*>(a.Av + (size_t)node * kH + 2 * lane);
      float2 g = *reinterpret_cast<const float2*>(a.G1 + (size_t)key * kH + 2 * lane);
      const float rho = s->srho[rr];
      float z0 = p.x + g.x + rho * vr.x, z1 = p.y + g.y + rho * vr.y;
      if (WHAT == 0) {
        o.x = silu_f(z0);
        o.y = silu_f(z1);
      } else {
        silu_grad_f(z0, o.x, od.x);
        silu_grad_f(z1, o.y, od.y);
      }
    }
    if (WHAT != 2) *reinterpret_cast<float2*>(TA1 + rr * kH + 2 * lane) = o;
    if (WHAT != 0) *reinterpret_cast<float2*>(TD1 + rr * kH + 2 * lane) = od;
  }
}

// Add the rows of tile T into the per-(graph,channel) [C][64] sums.
// single == true: the whole tile lies in one graph -> shared accumulator;
// otherwise one global atomic per key run.
__device__ __forceinline__ void virt_rows_to_graph(const float* __restrict__ T, VirtSmem* s, int C, int TN, bool single,
                                                   float* __restrict__ dst) {
  const int col = threadIdx.x & 63, grp = threadIdx.x >> 6;
  const int per = (TN + 3) >> 2;
  const int j0 = grp * per, j1 = min(TN, j0 + per);
  for (int c = 0; c < C; ++c) {
    if (single) {
      float acc = 0.f;
      for (int jn = j0; jn < j1; ++jn) {
        const int r = jn * C + c;
        if (s->skey[r] >= 0) acc += T[r * kH + col];
      }
      if (j1 > j0) atomicAdd(&s->accBig[c * kH + col], acc);
    } else {
      int cur = -1;
      float acc = 0.f;
      for (int jn = j0; jn < j1; ++jn) {
        const int r = jn * C + c;
        const int k = s->skey[r];
        if (k != cur) {
          if (cur >= 0) atomicAdd(dst + (size_t)cur * kH + col, acc);
          cur = k;
          acc = 0.f;
        }
        if (k >= 0) acc += T[r * kH + col];
      }
      if (cur >= 0) atomicAdd(dst + (size_t)cur * kH + col, acc);
    }
  }
}

constexpr size_t kVirtFwdSmem = (3 * kWFloats + 2 * kTileFloats) * sizeof(float) + sizeof(VirtSmem);
constexpr size_t kVirtBwdSmem = (3 * kWFloats + 5 * kTileFloats) * sizeof(float) + sizeof(VirtSmem);

// kSaved: the saved-only form of a backward's recompute (FEGNN_F_RECOMPUTE): u, Dsum and Usum only -- x' and its per-graph
// sum are already in the next layer's state, and adding xsum_new again would double it
template <bool kDet, bool kSaved = false>
__global__ void __launch_bounds__(kThreads, 1) virtual_fwd_kernel(VirtArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* V2s = smem;
  float* Wxvs = V2s + kWFloats;
  float* WXs = Wxvs + kWFloats;
  float* T1 = WXs + kWFloats;
  float* T2 = T1 + kTileFloats;
  VirtSmem* s = reinterpret_cast<VirtSmem*>(T2 + kTileFloats);
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int C = a.C, TN = kTM / C;
  const bool att = a.flags & FEGNN_F_ATTENTION, use_tanh = a.flags & FEGNN_F_TANH, grav = a.flags & FEGNN_F_GRAVITY;
  virt_stage(a, s, V2s, Wxvs, WXs);
  const int ntiles = (a.N + TN - 1) / TN;
  int cur_b = -1;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    __syncthreads();
    virt_geometry<false>(a, s, tile, TN);
    __syncthreads();
    const bool single = s->b_first == s->b_last;
    if (!kDet && (!single || s->b_first != cur_b)) {
      const int nb = single ? s->b_first : -1;
      if constexpr (kSaved) virt_flush(s, cur_b, C, a.Usum, a.Dsum, nullptr);
      else virt_flush(s, cur_b, C, a.Usum, a.Dsum, a.xsum_new);
      cur_b = nb;
    }
    virt_assemble<0>(a, s, T1, nullptr);
    __syncthreads();
    float acc[kRT][4];
    zero_acc(acc);
    gemm_nt(acc, T1, V2s, ty, tx);
    {
      const float4 bb = *reinterpret_cast<const float4*>(s->c2 + tx * 4);
      const float4 wa = att ? *reinterpret_cast<const float4*>(s->wav + tx * 4) : make_float4(0, 0, 0, 0);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int rr = ty * kRT + i;
        float4 m;
        m.x = silu_f(acc[i][0] + bb.x); m.y = silu_f(acc[i][1] + bb.y);
        m.z = silu_f(acc[i][2] + bb.z); m.w = silu_f(acc[i][3] + bb.w);
        if (att) {
          float gate = sigmoid_f(rowsum16(m.x * wa.x + m.y * wa.y + m.z * wa.z + m.w * wa.w) + s->bav);
          m.x *= gate; m.y *= gate; m.z *= gate; m.w *= gate;
        }
        *reinterpret_cast<float4*>(T2 + rr * kH + tx * 4) = m;
        if (s->skey[rr] >= 0)
          *reinterpret_cast<float4*>(a.u + ((size_t)tile * TN * C + rr) * kH + tx * 4) = m;
      }
    }
    __syncthreads();
    if (!kDet) virt_rows_to_graph(T2, s, C, TN, single, a.Usum);
    // phi_xv head
    zero_acc(acc);
    gemm_nt(acc, T2, Wxvs, ty, tx);
    {
      const float4 bb = *reinterpret_cast<const float4*>(s->bxv + tx * 4);
      const float4 w = *reinterpret_cast<const float4*>(s->wxv + tx * 4);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        float sv_ = rowsum16(silu_f(acc[i][0] + bb.x) * w.x + silu_f(acc[i][1] + bb.y) * w.y +
                             silu_f(acc[i][2] + bb.z) * w.z + silu_f(acc[i][3] + bb.w) * w.w);
        if (use_tanh) sv_ = tanhf(sv_);
        if (tx == 0) s->ssxv[ty * kRT + i] = sv_;
      }
    }
    // phi_X head
    zero_acc(acc);
    gemm_nt(acc, T2, WXs, ty, tx);
    {
      const float4 bb = *reinterpret_cast<const float4*>(s->bX + tx * 4);
      const float4 w = *reinterpret_cast<const float4*>(s->wX + tx * 4);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        float sv_ = rowsum16(silu_f(acc[i][0] + bb.x) * w.x + silu_f(acc[i][1] + bb.y) * w.y +
                             silu_f(acc[i][2] + bb.z) * w.z + silu_f(acc[i][3] + bb.w) * w.w);
        if (use_tanh) sv_ = tanhf(sv_);
        if (tx == 0) s->ssX[ty * kRT + i] = sv_;
      }
    }
    __syncthreads();
    // per-row: Dsum[b,:,c] += D * sX
    if (tid < kTM) {
      const int key = s->skey[tid];
      if (key >= 0) {
        const int b = key / C, c = key - b * C;
        const float sX = s->ssX[tid];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          float val = s->sD[tid * 3 + k] * sX;
          if (kDet) a.Dsum[((size_t)tile * TN * C + tid) * 3 + k] = val;
          else if (single) atomicAdd(&s->accSmall[k * C + c], val);
          else atomicAdd(a.Dsum + ((size_t)b * 3 + k) * C + c, val);
        }
      }
    }
    // per-node: x' (models/FastEGNN.py:133-142) and its per-graph sum
    if constexpr (kSaved) continue;
    if (tid < TN) {
      const int i = tile * TN + tid;
      if (i < a.N) {
        const int b = s->sb[tid];
        const float di = a.dinv != nullptr ? a.dinv[i] : 1.f, svi = a.sv[i];
        const float sgi = grav ? a.sg[i] : 0.f;
        const float invC = 1.f / (float)C;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          float vsum = 0.f;
          for (int c = 0; c < C; ++c) vsum += s->sD[(tid * C + c) * 3 + k] * s->ssxv[tid * C + c];
          float xn = a.x[(size_t)i * 3 + k] + a.tsum[(size_t)i * 3 + k] * di - vsum * invC +
                     svi * a.v[(size_t)i * 3 + k];
          if (grav) xn += sgi * a.grav[k];
          a.x_new[(size_t)i * 3 + k] = xn;
          if (kDet) continue;
          if (single) atomicAdd(&s->accX[k], xn);
          else atomicAdd(a.xsum_new + (size_t)b * 3 + k, xn);
        }
      }
    }
  }
  if constexpr (kSaved) virt_flush(s, cur_b, C, a.Usum, a.Dsum, nullptr);
  else if (!kDet) virt_flush(s, cur_b, C, a.Usum, a.Dsum, a.xsum_new);
}

__global__ void __launch_bounds__(kThreads, 1) virtual_bwd_kernel(VirtArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* V2s = smem;
  float* Wxvs = V2s + kWFloats;
  float* WXs = Wxvs + kWFloats;
  float* T0 = WXs + kWFloats;      // a1
  float* T1 = T0 + kTileFloats;    // z2, later silu'(z1), later gzv1
  float* T2 = T1 + kTileFloats;    // u
  float* T3 = T2 + kTileFloats;    // head gradients gzxv / gzX
  float* T4 = T3 + kTileFloats;    // running du, later gzv2
  VirtSmem* s = reinterpret_cast<VirtSmem*>(T4 + kTileFloats);
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int C = a.C, TN = kTM / C;
  const bool att = a.flags & FEGNN_F_ATTENTION, use_tanh = a.flags & FEGNN_F_TANH, grav = a.flags & FEGNN_F_GRAVITY;
  virt_stage(a, s, V2s, Wxvs, WXs);

  float wgV2[4][4], wgWxv[4][4], wgWX[4][4];
  zero_wg(wgV2); zero_wg(wgWxv); zero_wg(wgWX);
  float cwxv[4] = {0, 0, 0, 0}, cbxv[4] = {0, 0, 0, 0}, cwX[4] = {0, 0, 0, 0}, cbX[4] = {0, 0, 0, 0},
        cc2[4] = {0, 0, 0, 0}, cvr[4] = {0, 0, 0, 0}, cwav[4] = {0, 0, 0, 0};
  float cbav = 0.f;

  const int ntiles = (a.N + TN - 1) / TN;
  int cur_b = -1;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    __syncthreads();
    virt_geometry<true>(a, s, tile, TN);
    __syncthreads();
    const bool single = s->b_first == s->b_last;
    if (!single || s->b_first != cur_b) {
      const int nb = single ? s->b_first : -1;
      virt_flush(s, cur_b, C, a.gG1, a.gZ, nullptr);
      cur_b = nb;
    }
    virt_assemble<0>(a, s, T0, nullptr);
    __syncthreads();
    float acc[kRT][4];
    // ---- recompute u
    zero_acc(acc);
    gemm_nt(acc, T0, V2s, ty, tx);
    {
      const float4 bb = *reinterpret_cast<const float4*>(s->c2 + tx * 4);
      const float4 wa = att ? *reinterpret_cast<const float4*>(s->wav + tx * 4) : make_float4(0, 0, 0, 0);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int rr = ty * kRT + i;
        float4 z = make_float4(acc[i][0] + bb.x, acc[i][1] + bb.y, acc[i][2] + bb.z, acc[i][3] + bb.w);
        float4 m = make_float4(silu_f(z.x), silu_f(z.y), silu_f(z.z), silu_f(z.w));
        if (att) {
          float gate = sigmoid_f(rowsum16(m.x * wa.x + m.y * wa.y + m.z * wa.z + m.w * wa.w) + s->bav);
          if (tx == 0) s->sgate[rr] = gate;
          m.x *= gate; m.y *= gate; m.z *= gate; m.w *= gate;
        }
        *reinterpret_cast<float4*>(T2 + rr * kH + tx * 4) = m;
        *reinterpret_cast<float4*>(T1 + rr * kH + tx * 4) = z;
      }
    }
    __syncthreads();
    // ---- the two coordinate heads: head 0 = phi_xv, head 1 = phi_X
#pragma unroll 1
    for (int head = 0; head < 2; ++head) {
      const float* Ws = head == 0 ? Wxvs : WXs;
      const float* bvec = head == 0 ? s->bxv : s->bX;
      const float* wvec = head == 0 ? s->wxv : s->wX;
      const float* gsv_ = head == 0 ? s->sgsxv : s->sgsX;
      float* sout = head == 0 ? s->ssxv : s->ssX;
      zero_acc(acc);
      gemm_nt(acc, T2, Ws, ty, tx);
      float cw[4] = {0, 0, 0, 0}, cb[4] = {0, 0, 0, 0};
      {
        const float4 bb = *reinterpret_cast<const float4*>(bvec + tx * 4);
        const float4 w = *reinterpret_cast<const float4*>(wvec + tx * 4);
#pragma unroll
        for (int i = 0; i < kRT; ++i) {
          const int rr = ty * kRT + i;
          float av[4], dv[4];
          silu_grad_f(acc[i][0] + bb.x, av[0], dv[0]); silu_grad_f(acc[i][1] + bb.y, av[1], dv[1]);
          silu_grad_f(acc[i][2] + bb.z, av[2], dv[2]); silu_grad_f(acc[i][3] + bb.w, av[3], dv[3]);
          float sc = rowsum16(av[0] * w.x + av[1] * w.y + av[2] * w.z + av[3] * w.w);
          float gs = gsv_[rr];
          if (use_tanh) {
            sc = tanhf(sc);
            gs *= (1.f - sc * sc);
          }
          if (tx == 0) sout[rr] = sc;
          float4 g = make_float4(gs * w.x * dv[0], gs * w.y * dv[1], gs * w.z * dv[2], gs * w.w * dv[3]);
          *reinterpret_cast<float4*>(T3 + rr * kH + tx * 4) = g;
          cw[0] = fmaf(gs, av[0], cw[0]); cw[1] = fmaf(gs, av[1], cw[1]);
          cw[2] = fmaf(gs, av[2], cw[2]); cw[3] = fmaf(gs, av[3], cw[3]);
          cb[0] += g.x; cb[1] += g.y; cb[2] += g.z; cb[3] += g.w;
        }
      }
      if (head == 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { cwxv[j] += cw[j]; cbxv[j] += cb[j]; }
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) { cwX[j] += cw[j]; cbX[j] += cb[j]; }
      }
      __syncthreads();
      if (head == 0) wgrad_acc(wgWxv, T3, T2, kTM);
      else wgrad_acc(wgWX, T3, T2, kTM);
      // running du: starts from the upstream terms (phi_h path and pooled-sum path)
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int rr = ty * kRT + i;
        float4 g0 = make_float4(0, 0, 0, 0);
        if (head == 0) {
          const int key = s->skey[rr];
          if (key >= 0) {
            if (a.gu != nullptr)
              g0 = *reinterpret_cast<const float4*>(a.gu + ((size_t)tile * TN * C + rr) * kH + tx * 4);
            if (a.gUsum != nullptr) {
              float4 g1 = *reinterpret_cast<const float4*>(a.gUsum + (size_t)key * kH + tx * 4);
              g0.x += g1.x; g0.y += g1.y; g0.z += g1.z; g0.w += g1.w;
            }
          }
        } else {
          g0 = *reinterpret_cast<const float4*>(T4 + rr * kH + tx * 4);
        }
        acc[i][0] = g0.x; acc[i][1] = g0.y; acc[i][2] = g0.z; acc[i][3] = g0.w;
      }
      gemm_nn(acc, T3, Ws, ty, tx);
      if (head == 0) {
#pragma unroll
        for (int i = 0; i < kRT; ++i)
          *reinterpret_cast<float4*>(T4 + (ty * kRT + i) * kH + tx * 4) =
              make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
      }
      __syncthreads();   // T3 free for the next head / later reuse
    }
    // ---- through the gate and the second silu: gzv2 -> T4 (own elements)
    {
      const float4 wa = att ? *reinterpret_cast<const float4*>(s->wav + tx * 4) : make_float4(0, 0, 0, 0);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int rr = ty * kRT + i;
        const float4 z = *reinterpret_cast<const float4*>(T1 + rr * kH + tx * 4);
        float m0[4], d2[4];
        silu_grad_f(z.x, m0[0], d2[0]); silu_grad_f(z.y, m0[1], d2[1]);
        silu_grad_f(z.z, m0[2], d2[2]); silu_grad_f(z.w, m0[3], d2[3]);
        float g[4] = {acc[i][0], acc[i][1], acc[i][2], acc[i][3]};
        const bool valid = s->skey[rr] >= 0;
        if (att) {
          float ggate = rowsum16(g[0] * m0[0] + g[1] * m0[1] + g[2] * m0[2] + g[3] * m0[3]);
          float gate = s->sgate[rr];
          float gpre = valid ? ggate * gate * (1.f - gate) : 0.f;
          g[0] = g[0] * gate + gpre * wa.x; g[1] = g[1] * gate + gpre * wa.y;
          g[2] = g[2] * gate + gpre * wa.z; g[3] = g[3] * gate + gpre * wa.w;
          cwav[0] = fmaf(gpre, m0[0], cwav[0]); cwav[1] = fmaf(gpre, m0[1], cwav[1]);
          cwav[2] = fmaf(gpre, m0[2], cwav[2]); cwav[3] = fmaf(gpre, m0[3], cwav[3]);
          if (tx == 0) cbav += gpre;
        }
        float4 o = valid ? make_float4(g[0] * d2[0], g[1] * d2[1], g[2] * d2[2], g[3] * d2[3])
                         : make_float4(0, 0, 0, 0);
        *reinterpret_cast<float4*>(T4 + rr * kH + tx * 4) = o;
        cc2[0] += o.x; cc2[1] += o.y; cc2[2] += o.z; cc2[3] += o.w;
      }
    }
    __syncthreads();
    virt_assemble<2>(a, s, nullptr, T1);     // silu'(zv1) -> T1 (z2 is dead)
    wgrad_acc(wgV2, T4, T0, kTM);
    zero_acc(acc);
    gemm_nn(acc, T4, V2s, ty, tx);
    __syncthreads();                         // T1 fully written by the assemble above
    {
      const float4 vr = *reinterpret_cast<const float4*>(s->vr + tx * 4);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const int rr = ty * kRT + i;
        float4 d1 = *reinterpret_cast<const float4*>(T1 + rr * kH + tx * 4);
        float4 g = make_float4(acc[i][0] * d1.x, acc[i][1] * d1.y, acc[i][2] * d1.z, acc[i][3] * d1.w);
        *reinterpret_cast<float4*>(T1 + rr * kH + tx * 4) = g;
        const float rho = s->srho[rr];
        cvr[0] = fmaf(g.x, rho, cvr[0]); cvr[1] = fmaf(g.y, rho, cvr[1]);
        cvr[2] = fmaf(g.z, rho, cvr[2]); cvr[3] = fmaf(g.w, rho, cvr[3]);
        float grho = rowsum16(g.x * vr.x + g.y * vr.y + g.z * vr.z + g.w * vr.w);
        if (tx == 0) s->sgrho[rr] = grho;
      }
    }
    __syncthreads();
    // ---- outputs
    virt_rows_to_graph(T1, s, C, TN, single, a.gG1);
    {   // gAv[i] = sum_c gzv1[(i,c)]
      const int col = tid & 63, grp = tid >> 6;
      for (int jn = grp; jn < TN; jn += 4) {
        const int i = tile * TN + jn;
        if (i < a.N) {
          float sum = 0.f;
          for (int c = 0; c < C; ++c) sum += T1[(jn * C + c) * kH + col];
          a.gAv[(size_t)i * kH + col] = sum;
        }
      }
    }
    if (tid < kTM) {
      const int key = s->skey[tid];
      float gD[3] = {0, 0, 0};
      if (key >= 0) {
        const int b = key / C, c = key - b * C, jn = tid / C;
        const float rho = s->srho[tid];
        const float f = rho > 0.f ? s->sgrho[tid] / rho : 0.f;
        const float sxv = s->ssxv[tid], sX = s->ssX[tid], invC = 1.f / (float)C;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          gD[k] = -sxv * s->sgxn[jn * 3 + k] * invC + sX * a.gDsum[((size_t)b * 3 + k) * C + c] +
                  f * s->sD[tid * 3 + k];
          if (single) atomicAdd(&s->accSmall[k * C + c], gD[k]);
          else atomicAdd(a.gZ + ((size_t)b * 3 + k) * C + c, gD[k]);
        }
      }
      s->sgD[tid * 3 + 0] = gD[0]; s->sgD[tid * 3 + 1] = gD[1]; s->sgD[tid * 3 + 2] = gD[2];
    }
    __syncthreads();
    if (tid < TN) {
      const int i = tile * TN + tid;
      if (i < a.N) {
        const float di = a.dinv != nullptr ? a.dinv[i] : 1.f;
        float gsv = 0.f, gsg = 0.f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const float g = s->sgxn[tid * 3 + k];
          float sum = 0.f;
          for (int c = 0; c < C; ++c) sum += s->sgD[(tid * C + c) * 3 + k];
          a.gx[(size_t)i * 3 + k] = g - sum;
          a.gt[(size_t)i * 3 + k] = g * di;
          gsv = fmaf(g, a.v[(size_t)i * 3 + k], gsv);
          gsg = fmaf(g, a.grav[k], gsg);
        }
        a.gsv[i] = gsv;
        if (grav) a.gsg[i] = gsg;
      }
    }
  }
  virt_flush(s, cur_b, C, a.gG1, a.gZ, nullptr);
  wgrad_flush(wgV2, a.g_V2, kH, 0, 1);
  wgrad_flush(wgWxv, a.g_Wxv, kH, 0, 1);
  wgrad_flush(wgWX, a.g_WX, kH, 0, 1);
  {
    __syncthreads();                       // T0 is free: every tile is finished
    colsum_stash(T0, 0, cwxv); colsum_stash(T0, 1, cbxv); colsum_stash(T0, 2, cwX); colsum_stash(T0, 3, cbX);
    colsum_stash(T0, 4, cc2); colsum_stash(T0, 5, cvr); colsum_stash(T0, 6, cwav);
    const ColsumDst dsts[7] = {{a.g_wxv, 1}, {a.g_bxv, 1}, {a.g_wX, 1}, {a.g_bX, 1}, {a.g_c2, 1},
                               {a.g_wv1 != nullptr ? a.g_wv1 + 2 * kH : nullptr, a.ldv}, {att ? a.g_wav : nullptr, 1}};
    colsum_emit<7>(T0, dsts);
  }
  if (att) {
    if (tx == 0 && a.g_bav != nullptr) atomicAdd(a.g_bav, cbav);
  }
}

template <bool kDet = false, bool kSaved = false>
cudaError_t launch_virtual_fwd(const VirtArgs& a, int sms, cudaStream_t st) {
  static DevOnce attr;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(virtual_fwd_kernel<kDet, kSaved>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kVirtFwdSmem);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  const int TN = kTM / a.C;
  int ntiles = (a.N + TN - 1) / TN;
  if (ntiles == 0) return cudaSuccess;
  int grid = ntiles < sms ? ntiles : sms;
  virtual_fwd_kernel<kDet, kSaved><<<grid, kThreads, kVirtFwdSmem, st>>>(a); ++g_launches;
  return cudaGetLastError();
}
cudaError_t launch_virtual_bwd(const VirtArgs& a, int sms, cudaStream_t st) {
  static DevOnce attr;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(virtual_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kVirtBwdSmem);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  const int TN = kTM / a.C;
  int ntiles = (a.N + TN - 1) / TN;
  if (ntiles == 0) return cudaSuccess;
  int grid = ntiles < sms ? ntiles : sms;
  virtual_bwd_kernel<<<grid, kThreads, kVirtBwdSmem, st>>>(a); ++g_launches;
  return cudaGetLastError();
}

}  // namespace fegnn
