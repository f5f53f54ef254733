// virtual_tc.cu -- dense N x C real<->virtual phase on the tcgen05 tensor cores (single-pass TF32 tiles).
//
// Same contract as virtual_fwd_kernel / virtual_bwd_kernel (virtual_kernels.cu; reference models/FastEGNN.py:111-119,
// :133-150 and their autograd).  Rows of a tile are (node, channel) pairs, channel fastest, TN = 128 / C whole nodes per
// tile; thread (quarter, lane, cg) owns row 32*quarter + lane (= its tensor-memory lane) and CPT = 64 / CG columns.
//
//   forward   G1  z2 = a1 V2^T                 a1 built K-major in shared memory (half-warp per row, coalesced gather)
//             GH  [zxv | zX] = u [Wxv ; WX]^T  ONE N = 128 GEMM, u read from tensor memory (written by its row owner)
//   backward  two kernels with two dependent GEMM stages each (everything else hangs off the critical path):
//     heads   GH as above from the saved u; A = [gzxv | gzX] in tensor memory;
//             gu = gu_ext + gUsum + [gzxv | gzX] [Wxv ; WX]   (K = 128);   [dWxv ; dWX | db..] += [gzxv | gzX]^T [u | 1..]
//             gu is written over the gu buffer (which then feeds the trunk kernel); coordinate outputs except the rho term.
//     trunk   G1 recomputed for silu'(z2); gz2 = gu silu'(z2); ga1 = gz2 V2; gz1 = ga1 silu'(z1);
//             [dc2.. | dV2] += gz2^T [1.. | a1];  dvr += gz1^T rho;  gAv, gG1, and the rho term of gx / gZ.
// Weight-gradient operands are row-major tiles read MN-major (SWIZZLE_128B_BASE32B), see edge_tc_bwd2.cu.
// attention=True layers use the fp32 FMA kernels.
#include "common.cuh"
#include "umma.cuh"
#include <cuda_fp16.h>

namespace fegnn {
namespace vtc {

using bwd2::desc_advance;
using bwd2::gemm_ts_kmajor;
using bwd2::gemm_ts_mn;
using bwd2::gemm_wgrad;
using bwd2::idesc_tf32;
using bwd2::make_desc_mn;
using bwd2::mma_ts;
using bwd2::mn_chunk_off;
using bwd2::mn_load_row;
using bwd2::mn_store_row;
using bwd2::silu_grad_tc;
using bwd2::tmem_ld;
using bwd2::tmem_st;
using bwd2::tmem_st_wait;

// With t = z / 2: z (0.5 + 0.5 tanh t) = t + t tanh t (FMUL, MUFU, FFMA); silu_tc_hb takes HALF the bias, so that the bias
// add and the halving are one FFMA (3 instructions per activation instead of 5).
__device__ __forceinline__ float silu_tc(float z) {
  const float t = 0.5f * z;
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(t));
  return fmaf(t, th, t);
}
__device__ __forceinline__ float silu_tc_hb(float z, float half_bias) {
  const float t = fmaf(z, 0.5f, half_bias);
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(t));
  return fmaf(t, th, t);
}

// Weight staging in two phases: every global load of a thread (all weights of the kernel) is in flight before its first
// shared-memory store -- ONE L2 round trip per prologue.  (A load-store loop per weight serialised 4 round trips per weight:
// 16 % of the forward kernel's samples at 8 000 nodes, profiles/ncu_top_kernels_r1_final.txt.)
template <int NT>
struct WRegs {
  float4 v[kH * 16 / NT];
};
template <int NT>
__device__ __forceinline__ void wregs_load(WRegs<NT>& w, const float* __restrict__ g, int ld) {
#pragma unroll
  for (int j = 0; j < kH * 16 / NT; ++j) {
    const int i = threadIdx.x + j * NT, n = i >> 4, c = i & 15;
    w.v[j] = *reinterpret_cast<const float4*>(g + (size_t)n * ld + c * 4);
  }
}
// a reference [64][ld] weight K-major SWIZZLE_128B into rows [row0, row0+64) of a tile with R rows
template <int NT>
__device__ __forceinline__ void wregs_store_kmajor(const WRegs<NT>& w, uint8_t* dst, int row0, int R) {
#pragma unroll
  for (int j = 0; j < kH * 16 / NT; ++j) {
    const int i = threadIdx.x + j * NT, n = i >> 4, c = i & 15;
    *reinterpret_cast<float4*>(dst + umma::tile_chunk_off(row0 + n, c, R)) = w.v[j];
  }
}
// ... and row-major BASE32B (MN-major operand) into rows [row0, row0+64) of a tile with R rows
template <int NT>
__device__ __forceinline__ void wregs_store_mn(const WRegs<NT>& w, uint8_t* dst, int row0, int R) {
#pragma unroll
  for (int j = 0; j < kH * 16 / NT; ++j) {
    const int i = threadIdx.x + j * NT, n = i >> 4, c = i & 15;
    *reinterpret_cast<float4*>(dst + mn_chunk_off(row0 + n, c, R)) = w.v[j];
  }
}

// per-graph accumulators of a CTA that stays inside one graph (same policy as virtual_kernels.cu)
struct GraphAcc {
  float big[FEGNN_MAX_C * kH];     // Usum (fwd) / gG1 (bwd trunk)
  float small[3 * FEGNN_MAX_C];    // Dsum (fwd) / gZ (bwd)
  float x3[3];                     // xsum_new (fwd)
};
template <int NT>
__device__ __forceinline__ void acc_clear(GraphAcc* g) {
  for (int i = threadIdx.x; i < FEGNN_MAX_C * kH; i += NT) g->big[i] = 0.f;
  if (threadIdx.x < 3 * FEGNN_MAX_C) g->small[threadIdx.x] = 0.f;
  if (threadIdx.x < 3) g->x3[threadIdx.x] = 0.f;
}
// flush graph b (if any) and clear; all threads
template <int NT>
__device__ __forceinline__ void acc_flush(GraphAcc* g, int b, int C, float* dstBig, float* dstSmall, float* dstX) {
  __syncthreads();
  if (b >= 0) {
    if (dstBig != nullptr)
      for (int i = threadIdx.x; i < C * kH; i += NT) {
        atomicAdd(dstBig + (size_t)b * C * kH + i, g->big[i]);
        g->big[i] = 0.f;
      }
    if (dstSmall != nullptr && threadIdx.x < 3 * C) {
      atomicAdd(dstSmall + (size_t)b * 3 * C + threadIdx.x, g->small[threadIdx.x]);
      g->small[threadIdx.x] = 0.f;
    }
    if (dstX != nullptr && threadIdx.x < 3) {
      atomicAdd(dstX + (size_t)b * 3 + threadIdx.x, g->x3[threadIdx.x]);
      g->x3[threadIdx.x] = 0.f;
    }
  }
  __syncthreads();
}

// Tile inside one graph: small[k * C + c] += sum over the tile's nodes jn of rows[(jn * C + c) * 3 + k]  (rows = [kTM][3] with
// zeros in unused rows).  ONE warp, after the barrier that follows the row writes; it replaces three same-address shared-memory
// atomics per row (128 rows on 3 C addresses: 20-30 % of the backward kernels' stall samples at 8 000 nodes).
__device__ __forceinline__ void small_from_rows(const float* rows, GraphAcc* g, int C, int TN, int lane) {
  const int W = 3 * C;
  if (W <= 32) {
    int nseg = 32 / W;
    nseg = nseg > 4 ? 4 : nseg;
    const int seg = lane / W, p = lane - seg * W;
    float s = 0.f;
    if (seg < nseg) {
#pragma unroll 4
      for (int jn = seg; jn < TN; jn += nseg) s += rows[jn * W + p];
    }
    float tot = s;
    for (int i = 1; i < nseg; ++i) tot += __shfl_down_sync(0xffffffffu, s, i * W);
    if (lane < W) {
      const int c = p / 3, k = p - c * 3;
      g->small[k * C + c] += tot;
    }
  } else {
    for (int p = lane; p < W; p += 32) {
      float s = 0.f;
      for (int jn = 0; jn < TN; ++jn) s += rows[jn * W + p];
      const int c = p / 3, k = p - c * 3;
      g->small[k * C + c] += s;
    }
  }
}

// Add the rows of a BASE32B tile into the per-(graph, channel) [C][64] sums: thread (col, grp) walks the nodes of its
// group; single -> shared accumulator, otherwise one global atomic per key run.
template <int NT>
__device__ __forceinline__ void rows_to_graph(const uint8_t* T, const int* skey, GraphAcc* g, int C, int TN, bool single,
                                              float* __restrict__ dst) {
  constexpr int GR = NT / 64;
  const int col = threadIdx.x & 63, grp = threadIdx.x >> 6;
  const int per = (TN + GR - 1) / GR;
  const int j0 = grp * per, j1 = min(TN, j0 + per);
  const uint32_t cbase = (col >> 5) * (kTM * 128) + ((col & 7) << 2);
  const int c8 = (col & 31) >> 3;
  auto at = [&](int r) { return *reinterpret_cast<const float*>(T + cbase + r * 128 + ((c8 ^ (r & 3)) << 5)); };
  if (single) {
    // whole tile inside one graph (unused rows of the tile hold zeros): thread (channel, column) owns its sum -- no key reads,
    // independent loads, a plain add.  (The keyed walk below is one dependent shared-memory chain per row, and 8 groups adding
    // into the same shared word cost ~800 cycles per atomic: 3 400 cycles per tile at C = 3.)
    for (int c = grp; c < C; c += GR) {
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      int jn = 0;
      for (; jn + 3 < TN; jn += 4) {
        a0 += at(jn * C + c); a1 += at((jn + 1) * C + c); a2 += at((jn + 2) * C + c); a3 += at((jn + 3) * C + c);
      }
      for (; jn < TN; ++jn) a0 += at(jn * C + c);
      g->big[c * kH + col] += (a0 + a1) + (a2 + a3);
    }
    return;
  }
  for (int c = 0; c < C; ++c) {
    int cur = -1;
    float acc = 0.f;
    for (int jn = j0; jn < j1; ++jn) {
      const int r = jn * C + c;
      const int k = skey[r];
      if (k != cur) {
        if (cur >= 0) atomicAdd(dst + (size_t)cur * kH + col, acc);
        cur = k;
        acc = 0.f;
      }
      if (k >= 0) acc += at(r);
    }
    if (cur >= 0) atomicAdd(dst + (size_t)cur * kH + col, acc);
  }
}

// ------------------------------------------------------------------------------------------------- forward
struct FwdVec {
  float vr[kH], c2[kH], bh[2 * kH], wh[2 * kH];     // bh = (bxv | bX), wh = (wxv | wX)
  int skey[kTM], snode[kTM], sb[kTM];
  float sD[kTM * 3], srho[kTM], spx[4 * kTM], spX[4 * kTM], ssxv[kTM], ssX[kTM];
  float sval[kTM * 3];                               // D * sX per row (summed per graph and channel by one warp)
  int b_first, b_last;
  GraphAcc acc;
  uint64_t bar[2];
  uint32_t tmem_slot;
};
struct FwdSmem {
  static constexpr int off_V2 = 0;                       // [64][64]  K-major
  static constexpr int off_WH = 16384;                   // [128][64] K-major: rows 0-63 Wxv, 64-127 WX
  static constexpr int off_T = off_WH + 32768;           // a1 K-major for G1, then u BASE32B for the Usum walk
  static constexpr int off_vec = off_T + 32768;
  static constexpr size_t bytes = off_vec + sizeof(FwdVec) + 1024;
};
constexpr uint32_t kF_ACC0 = 0, kF_ACCH = 64, kF_OPA = 192;    // 256 columns

// kDet: no per-graph sums; the rows D sX go to the [N, C, 3] buffer in the Dsum slot (VirtArgs)
// kSaved: the saved-only form of a backward's recompute (FEGNN_F_RECOMPUTE): u, Dsum and Usum only -- x' and its per-graph
// sum are already in the next layer's state, and adding xsum_new again would double it
template <int CG, bool kDet, bool kSaved = false>
__global__ void __launch_bounds__(128 * CG, 2) virtual_fwd_tc_kernel(VirtArgs a) {
  VTR_DECL();
  constexpr int NT = 128 * CG, CPT = kH / CG, NW = NT / 32;
  using SM = FwdSmem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
  pdl_trigger();
  FwdVec* v = reinterpret_cast<FwdVec*>(smem + SM::off_vec);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int quarter = warp & 3, cg = warp >> 2, row = quarter * 32 + lane, c0 = cg * CPT;
  const int C = a.C, TN = kTM / C;
  const bool use_tanh = a.flags & FEGNN_F_TANH, grav = a.flags & FEGNN_F_GRAVITY;

  {
    WRegs<NT> w0, w1, w2;
    wregs_load<NT>(w0, a.V2, kH);
    wregs_load<NT>(w1, a.Wxv, kH);
    wregs_load<NT>(w2, a.WX, kH);
    wregs_store_kmajor<NT>(w0, smem + SM::off_V2, 0, kH);
    wregs_store_kmajor<NT>(w1, smem + SM::off_WH, 0, 2 * kH);
    wregs_store_kmajor<NT>(w2, smem + SM::off_WH, kH, 2 * kH);
  }
  for (int i = t; i < kH; i += NT) {
    v->vr[i] = a.wv1[(size_t)i * a.ldv + 2 * kH];
    v->c2[i] = 0.5f * a.c2[i];                                              // halved: silu_tc_hb
    v->bh[i] = 0.5f * a.bxv[i]; v->bh[kH + i] = 0.5f * a.bX[i];
    v->wh[i] = a.wxv[i]; v->wh[kH + i] = a.wX[i];
  }
  acc_clear<NT>(&v->acc);
  if (t == 0) {
    umma::mbar_init(&v->bar[0], 1);
    umma::mbar_init(&v->bar[1], 1);
    umma::mbar_fence_init();
  }
  if (warp == 0) umma::tmem_alloc<256>(&v->tmem_slot);
  umma::fence_smem_to_async();
  umma::fence_before();
  __syncthreads();
    VTR();
  umma::fence_after();
  pdl_wait();
  const uint32_t tmem = v->tmem_slot;
  const uint32_t tlane = tmem + ((uint32_t)(quarter * 32) << 16) + c0;
  const uint32_t id_g1 = umma::make_idesc_tf32(128, 64), id_gh = umma::make_idesc_tf32(128, 128);
  const uint64_t dV2 = umma::make_desc(umma::smem_u32(smem + SM::off_V2));
  const uint64_t dWH = umma::make_desc(umma::smem_u32(smem + SM::off_WH));
  const uint64_t dT = umma::make_desc(umma::smem_u32(smem + SM::off_T));
  uint8_t* T = smem + SM::off_T;
  uint32_t phase = 0;
  int cur_b = -1;

  const int ntiles = (a.N + TN - 1) / TN;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    umma::fence_before();
    __syncthreads();
    VTR();
    // ---- geometry: one thread per (node, channel) row
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
        if (c == 0) v->sb[jn] = b;
        if (t == 0) v->b_first = b;
        if (c == 0 && (jn == TN - 1 || i == a.N - 1)) v->b_last = b;
      }
      v->skey[t] = key;
      v->snode[t] = node;
      v->sD[t * 3 + 0] = D0; v->sD[t * 3 + 1] = D1; v->sD[t * 3 + 2] = D2;
      v->srho[t] = rho;
    }
    __syncthreads();
    VTR();
    const bool single = v->b_first == v->b_last;
    if (!kDet && (!single || v->b_first != cur_b)) {
      const int nb = single ? v->b_first : -1;
      if constexpr (kSaved) acc_flush<NT>(&v->acc, cur_b, C, a.Usum, a.Dsum, nullptr);
      else acc_flush<NT>(&v->acc, cur_b, C, a.Usum, a.Dsum, a.xsum_new);
      cur_b = nb;
    }
    // ---- assembly: a1 = silu(Av[node] + G1[key] + rho vr) -> T (K-major).  Half-warp per row, float4 per lane.
    {
      const int l16 = lane & 15, hsel = lane >> 4;
      const float4 vr = *reinterpret_cast<const float4*>(v->vr + 4 * l16);
      constexpr int RPW = kTM / NW;
#pragma unroll 1
      for (int i0 = 0; i0 < RPW; i0 += 8) {
        float4 p[4], g[4];
        int ki[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int rr = warp * RPW + i0 + 2 * j + hsel;
          ki[j] = v->skey[rr];
          p[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          g[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ki[j] >= 0) {
            p[j] = *reinterpret_cast<const float4*>(a.Av + (size_t)v->snode[rr] * kH + 4 * l16);
            g[j] = *reinterpret_cast<const float4*>(a.G1 + (size_t)ki[j] * kH + 4 * l16);
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int rr = warp * RPW + i0 + 2 * j + hsel;
          const float rho = v->srho[rr];
          float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ki[j] >= 0)
            o = make_float4(silu_tc(p[j].x + g[j].x + rho * vr.x), silu_tc(p[j].y + g[j].y + rho * vr.y),
                            silu_tc(p[j].z + g[j].z + rho * vr.z), silu_tc(p[j].w + g[j].w + rho * vr.w));
          *reinterpret_cast<float4*>(T + umma::tile_chunk_off(rr, l16, kTM)) = o;
        }
      }
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    __syncthreads();
    VTR();
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
        umma::gemm_k64_desc(tmem + kF_ACC0, dT, kTM, dV2, kH, id_g1, false);       // G1: z2 = a1 V2^T
        umma::commit(&v->bar[0]);
      }
      __syncwarp();
    }
    umma::mbar_wait(&v->bar[0], phase);
    VTR();
    umma::fence_after();
    // ---- epilogue 1: u = silu(z2 + c2) -> HBM (saved for backward / phi_h), tensor memory (A of GH), T (Usum walk)
    {
      float u[CPT];
      tmem_ld<CPT>(tlane + kF_ACC0, u);
      const bool valid = v->skey[row] >= 0;
#pragma unroll
      for (int j = 0; j < CPT; ++j) u[j] = valid ? silu_tc_hb(u[j], v->c2[c0 + j]) : 0.f;
      tmem_st<CPT>(tlane + kF_OPA, u);
      mn_store_row<CPT>(T, row, cg, u);          // G1 has finished reading T (bar[0])
      tmem_st_wait();
    }
    umma::fence_before();
    __syncthreads();
    VTR();
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)                                             // GH: [zxv | zX] = u [Wxv ; WX]^T
          mma_ts(tmem + kF_ACCH, tmem + kF_OPA + ks * 8, desc_advance(dWH, (ks >> 2) * (2 * kH * 128) + (ks & 3) * 32), id_gh, ks > 0);
        umma::commit(&v->bar[1]);
      }
      __syncwarp();
    }
    // u -> HBM (saved for backward / phi_h) from the T tile in (row, chunk) order: a warp-wide store covers 2 rows x 256
    // contiguous bytes (the row owners' stores touched 32 lines each)
    {
      float* ubase = a.u + (size_t)tile * TN * C * kH;
#pragma unroll
      for (int j = 0; j < kTM * 16 / NT; ++j) {
        const int i = t + j * NT, rr = i >> 4, c16 = i & 15;
        if (v->skey[rr] >= 0)
          *reinterpret_cast<float4*>(ubase + (size_t)rr * kH + 4 * c16) = *reinterpret_cast<const float4*>(T + mn_chunk_off(rr, c16, kTM));
      }
    }
    if (!kDet) rows_to_graph<NT>(T, v->skey, &v->acc, C, TN, single, a.Usum);       // overlaps GH
    umma::mbar_wait(&v->bar[1], phase);
    VTR();
    umma::fence_after();
    phase ^= 1;
    // ---- epilogue 2: the two coordinate heads  s = w . silu(z + b)
    {
      float z[CPT];
      tmem_ld<CPT>(tlane + kF_ACCH, z);
      float px = 0.f, pX = 0.f;
#pragma unroll
      for (int j = 0; j < CPT; ++j) px = fmaf(silu_tc_hb(z[j], v->bh[c0 + j]), v->wh[c0 + j], px);
      tmem_ld<CPT>(tlane + kF_ACCH + kH, z);
#pragma unroll
      for (int j = 0; j < CPT; ++j) pX = fmaf(silu_tc_hb(z[j], v->bh[kH + c0 + j]), v->wh[kH + c0 + j], pX);
      v->spx[cg * kTM + row] = px;
      v->spX[cg * kTM + row] = pX;
    }
    __syncthreads();
    VTR();
    if (t < kTM) {
      float sxv = 0.f, sX = 0.f;
#pragma unroll
      for (int g = 0; g < CG; ++g) { sxv += v->spx[g * kTM + t]; sX += v->spX[g * kTM + t]; }
      if (use_tanh) { sxv = tanhf(sxv); sX = tanhf(sX); }
      v->ssxv[t] = sxv;
      const int key = v->skey[t];
      float val[3] = {0.f, 0.f, 0.f};
      if (key >= 0) {                     // Dsum[b,:,c] += D * sX
        const int b = key / C, c = key - b * C;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          val[k] = v->sD[t * 3 + k] * sX;
          if (kDet) a.Dsum[((size_t)tile * TN * C + t) * 3 + k] = val[k];
          else if (!single) atomicAdd(a.Dsum + ((size_t)b * 3 + k) * C + c, val[k]);
        }
      }
      v->sval[t * 3 + 0] = val[0]; v->sval[t * 3 + 1] = val[1]; v->sval[t * 3 + 2] = val[2];
    }
    __syncthreads();
    VTR();
    if (!kDet && single && warp == NW - 1) small_from_rows(v->sval, &v->acc, C, TN, lane);
    if constexpr (kSaved) continue;
    if (warp * 32 < TN) {                 // x' (models/FastEGNN.py:133-142) and its per-graph sum
      const int i = tile * TN + t;
      float xs[3] = {0.f, 0.f, 0.f};
      if (t < TN && i < a.N) {
        const int b = v->sb[t];
        const float di = a.dinv != nullptr ? a.dinv[i] : 1.f, svi = a.sv[i];
        const float sgi = grav ? a.sg[i] : 0.f;
        const float invC = 1.f / (float)C;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          float vsum = 0.f;
          for (int c = 0; c < C; ++c) vsum += v->sD[(t * C + c) * 3 + k] * v->ssxv[t * C + c];
          float xn = a.x[(size_t)i * 3 + k] + a.tsum[(size_t)i * 3 + k] * di - vsum * invC + svi * a.v[(size_t)i * 3 + k];
          if (grav) xn += sgi * a.grav[k];
          a.x_new[(size_t)i * 3 + k] = xn;
          xs[k] = xn;
          if (!kDet && !single) atomicAdd(a.xsum_new + (size_t)b * 3 + k, xn);
        }
      }
      if (!kDet && single) {                       // one shared atomic per warp and coordinate instead of one per node
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          float sum = xs[k];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
          if (lane == 0) atomicAdd(&v->acc.x3[k], sum);
        }
      }
    }
  }
  if constexpr (kSaved) acc_flush<NT>(&v->acc, cur_b, C, a.Usum, a.Dsum, nullptr);
  else if (!kDet) acc_flush<NT>(&v->acc, cur_b, C, a.Usum, a.Dsum, a.xsum_new);
  umma::fence_before();
  __syncthreads();
    VTR();
  if (warp == 0) umma::tmem_dealloc<256>(tmem);
  VTR();
  VTR_PRINT("vfwd");
}


// ------------------------------------------------------------------------------------------------- backward
// chunk0 = first 16-byte chunk of this thread's CPT columns inside a BASE32B tile with 128-byte-row column blocks
template <int CPT>
__device__ __forceinline__ void mn_store_row_at(uint8_t* tile, int row, int chunk0, const float (&v)[CPT]) {
  const bool flip = row & 4;
#pragma unroll
  for (int p = 0; p < CPT / 8; ++p) {
    const float4 c0 = make_float4(v[8 * p], v[8 * p + 1], v[8 * p + 2], v[8 * p + 3]);
    const float4 c1 = make_float4(v[8 * p + 4], v[8 * p + 5], v[8 * p + 6], v[8 * p + 7]);
    const int k0 = chunk0 + 2 * p + (flip ? 1 : 0), k1 = k0 ^ 1;
    *reinterpret_cast<float4*>(tile + mn_chunk_off(row, k0, kTM)) = flip ? c1 : c0;
    *reinterpret_cast<float4*>(tile + mn_chunk_off(row, k1, kTM)) = flip ? c0 : c1;
  }
}

// geometry shared by the two backward kernels: keys, D = Z - x, rho, upstream coordinate gradients
struct BwdGeo {
  int skey[kTM], snode[kTM];
  float sD[kTM * 3], srho[kTM], sgxn[kTM * 3], sgsxv[kTM], sgsX[kTM], sgD[kTM * 3];
  int b_first, b_last;
};
__device__ __forceinline__ void bwd_geometry(const VirtArgs& a, BwdGeo* s, int tile, int TN, uint8_t* AUX) {
  const int t = threadIdx.x, C = a.C;
  if (t < kTM) {
    const int jn = t / C, c = t - jn * C;
    const int i = tile * TN + jn;
    const bool valid = jn < TN && i < a.N;
    int key = -1, node = -1;
    float D0 = 0, D1 = 0, D2 = 0, rho = 0, gsxv = 0, gsX = 0;
    if (valid) {
      const int b = a.batch[i];
      key = b * C + c;
      node = i;
      D0 = a.Z[((size_t)b * 3 + 0) * C + c] - a.x[(size_t)i * 3 + 0];
      D1 = a.Z[((size_t)b * 3 + 1) * C + c] - a.x[(size_t)i * 3 + 1];
      D2 = a.Z[((size_t)b * 3 + 2) * C + c] - a.x[(size_t)i * 3 + 2];
      rho = sqrtf(D0 * D0 + D1 * D1 + D2 * D2);
      if (t == 0) s->b_first = b;
      if (c == 0 && (jn == TN - 1 || i == a.N - 1)) s->b_last = b;
      float g0 = a.gx_new[(size_t)i * 3 + 0], g1 = a.gx_new[(size_t)i * 3 + 1], g2 = a.gx_new[(size_t)i * 3 + 2];
      if (a.gxsum_next != nullptr) {
        g0 += a.gxsum_next[(size_t)b * 3 + 0]; g1 += a.gxsum_next[(size_t)b * 3 + 1]; g2 += a.gxsum_next[(size_t)b * 3 + 2];
      }
      if (c == 0) { s->sgxn[jn * 3 + 0] = g0; s->sgxn[jn * 3 + 1] = g1; s->sgxn[jn * 3 + 2] = g2; }
      gsxv = -(D0 * g0 + D1 * g1 + D2 * g2) / (float)C;
      gsX = D0 * a.gDsum[((size_t)b * 3 + 0) * C + c] + D1 * a.gDsum[((size_t)b * 3 + 1) * C + c] +
            D2 * a.gDsum[((size_t)b * 3 + 2) * C + c];
    }
    s->skey[t] = key;
    s->snode[t] = node;
    s->sD[t * 3 + 0] = D0; s->sD[t * 3 + 1] = D1; s->sD[t * 3 + 2] = D2;
    s->srho[t] = rho;
    s->sgsxv[t] = gsxv;
    s->sgsX[t] = gsX;
    // aux columns (1, rho, 0 ...): logical 32-byte chunk 0 of the row (the rest of the tile stays zero)
    *reinterpret_cast<float4*>(AUX + t * 128 + ((t & 3) << 5)) = make_float4(valid ? 1.f : 0.f, rho, 0.f, 0.f);
  }
}


// ---- heads kernel
struct HeadsVec {
  float bh[2 * kH], wh[2 * kH], cwh[2 * kH];
  BwdGeo g;
  float spx[4 * kTM], spX[4 * kTM], ssxv[kTM], ssX[kTM];
  GraphAcc acc;
  uint64_t bar[3];
  uint32_t tmem_slot;
};
struct HeadsSmem {
  static constexpr int off_WHk = 0;                        // [128][64] K-major   (GH)
  static constexpr int off_WHm = 32768;                    // [128][64] BASE32B   (gu = [gzxv | gzX] [Wxv ; WX], K = 128)
  static constexpr int off_TU = 65536;                     // u [128][64] BASE32B
  static constexpr int off_AUX = off_TU + 32768;           // [128][32], adjacent: B = [TU | AUX], N = 96
  static constexpr int off_TGH = off_AUX + 16384;          // [gzxv | gzX] [128][128] BASE32B (A of the weight-gradient GEMM)
  static constexpr int off_SG = off_TGH + 65536;           // upstream dL/du rows of the tile [128][64] BASE32B (cp.async landing zone)
  static constexpr int off_vec = off_SG + 32768;
  static constexpr size_t bytes = off_vec + sizeof(HeadsVec) + 1024;
  static_assert(bytes <= 232448, "heads kernel: shared memory");
};
constexpr uint32_t kH_ACCH = 0, kH_ACCG = 128, kH_RW = 192, kH_OPA = 288;     // 416 columns

template <int CG>
__global__ void __launch_bounds__(128 * CG, 1) virtual_bwd_heads_tc_kernel(VirtArgs a) {
  VTR_DECL();
  constexpr int NT = 128 * CG, CPT = kH / CG, NW = NT / 32;
  using SM = HeadsSmem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
  pdl_trigger();
  HeadsVec* v = reinterpret_cast<HeadsVec*>(smem + SM::off_vec);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int quarter = warp & 3, cg = warp >> 2, row = quarter * 32 + lane, c0 = cg * CPT;
  const int C = a.C, TN = kTM / C;
  const bool use_tanh = a.flags & FEGNN_F_TANH, grav = a.flags & FEGNN_F_GRAVITY;

  {
    WRegs<NT> w1, w2;
    wregs_load<NT>(w1, a.Wxv, kH);
    wregs_load<NT>(w2, a.WX, kH);
    wregs_store_kmajor<NT>(w1, smem + SM::off_WHk, 0, 2 * kH);
    wregs_store_kmajor<NT>(w2, smem + SM::off_WHk, kH, 2 * kH);
    wregs_store_mn<NT>(w1, smem + SM::off_WHm, 0, 2 * kH);
    wregs_store_mn<NT>(w2, smem + SM::off_WHm, kH, 2 * kH);
  }
  for (int i = t; i < kH; i += NT) {
    v->bh[i] = a.bxv[i]; v->bh[kH + i] = a.bX[i];
    v->wh[i] = a.wxv[i]; v->wh[kH + i] = a.wX[i];
    v->cwh[i] = 0.f; v->cwh[kH + i] = 0.f;
  }
  for (int i = t; i < kTM * 128 / 16; i += NT) reinterpret_cast<float4*>(smem + SM::off_AUX)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  acc_clear<NT>(&v->acc);
  if (t == 0) {
#pragma unroll
    for (int i = 0; i < 3; ++i) umma::mbar_init(&v->bar[i], 1);
    umma::mbar_fence_init();
  }
  if (warp == 0) umma::tmem_alloc<512>(&v->tmem_slot);
  umma::fence_smem_to_async();
  umma::fence_before();
  __syncthreads();
    VTR();
  umma::fence_after();
  pdl_wait();
  const uint32_t tmem = v->tmem_slot;
  const uint32_t tlane = tmem + ((uint32_t)(quarter * 32) << 16) + c0;
  const uint32_t id_gh = umma::make_idesc_tf32(128, 128), id_gu = idesc_tf32(128, 64, 0, 1), id_w = idesc_tf32(128, 96, 1, 1);
  const uint64_t dWHk = umma::make_desc(umma::smem_u32(smem + SM::off_WHk));
  const uint64_t dWHm = make_desc_mn(umma::smem_u32(smem + SM::off_WHm), 2 * kH * 128);
  const uint64_t dTU = make_desc_mn(umma::smem_u32(smem + SM::off_TU), kTM * 128);       // [TU | AUX]
  const uint64_t dTGH = make_desc_mn(umma::smem_u32(smem + SM::off_TGH), kTM * 128);
  uint8_t* TU = smem + SM::off_TU;
  uint8_t* AUX = smem + SM::off_AUX;
  uint8_t* TGH = smem + SM::off_TGH;
  uint8_t* SG = smem + SM::off_SG;
  uint32_t phase = 0;
  bool first_tile = true;
  int cur_b = -1;
  float pwx[CPT], pwX[CPT];        // per-row partial sums of dwxv / dwX over this thread's tiles
  float st_gt = 0.f, st_x = 0.f;   // bound statistics of the edge backward over this thread's nodes: max|gt|, max|x - x_0|
#pragma unroll
  for (int j = 0; j < CPT; ++j) { pwx[j] = 0.f; pwX[j] = 0.f; }

  const int ntiles = (a.N + TN - 1) / TN;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    if (!first_tile) {                         // the previous tile's weight-gradient GEMM still reads TU, AUX and TGH
      umma::mbar_wait(&v->bar[2], phase ^ 1);
    VTR();
      umma::fence_after();
    }
    umma::fence_before();
    __syncthreads();
    VTR();
    // rows of this tile in the [N, C, 64] arrays; the upstream dL/du rows go in flight now, in (row, chunk) order, and are read
    // back by the row owners in epilogue 2 (a row-owner load touches 32 lines per access)
    const int nrows = min(TN, a.N - tile * TN) * C;
    const size_t tbase = (size_t)tile * TN * C * kH;
    // the saved u rows -> TU (first group: needed right after the geometry), the upstream rows -> SG (second group)
#pragma unroll
    for (int j = 0; j < kTM * 16 / NT; ++j) {
      const int i = t + j * NT, rr = i >> 4, c16 = i & 15;
      const bool ok = rr < nrows;
      cp_async16(TU + mn_chunk_off(rr, c16, kTM), a.u + tbase + (size_t)(ok ? rr : 0) * kH + 4 * c16, ok ? 16 : 0);
    }
    cp_async_commit();
    if (a.gu != nullptr) {
#pragma unroll
      for (int j = 0; j < kTM * 16 / NT; ++j) {
        const int i = t + j * NT, rr = i >> 4, c16 = i & 15;
        const bool ok = rr < nrows;
        cp_async16(SG + mn_chunk_off(rr, c16, kTM), a.gu + tbase + (size_t)(ok ? rr : 0) * kH + 4 * c16, ok ? 16 : 0);
      }
    }
    cp_async_commit();
    bwd_geometry(a, &v->g, tile, TN, AUX);
    cp_async_wait_group<1>();                  // u rows of this thread have landed (the barrier publishes everybody's)
    __syncthreads();
    VTR();
    const bool single = v->g.b_first == v->g.b_last;
    if (!single || v->g.b_first != cur_b) {
      const int nb = single ? v->g.b_first : -1;
      acc_flush<NT>(&v->acc, cur_b, C, nullptr, a.gZ, nullptr);
      cur_b = nb;
    }
    {
      float u[CPT];
      mn_load_row<CPT>(TU, row, cg, u);
      tmem_st<CPT>(tlane + kH_OPA, u);
      tmem_st_wait();
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    __syncthreads();
    VTR();
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)                                             // GH: [zxv | zX] = u [Wxv ; WX]^T
          mma_ts(tmem + kH_ACCH, tmem + kH_OPA + ks * 8, desc_advance(dWHk, (ks >> 2) * (2 * kH * 128) + (ks & 3) * 32), id_gh, ks > 0);
        umma::commit(&v->bar[0]);
      }
      __syncwarp();
    }
    umma::mbar_wait(&v->bar[0], phase);
    VTR();
    umma::fence_after();
    // ---- epilogue 1: head scalars, gz = gs w silu'(z) for both heads -> tensor memory (A of gu) and TGH (A of dW)
    {
      float gsx = v->g.sgsxv[row], gsX = v->g.sgsX[row];
      float z[CPT], av[CPT];
      if (use_tanh) {                          // the tanh derivative needs the complete head output first
        float px = 0.f, pX = 0.f;
        tmem_ld<CPT>(tlane + kH_ACCH, z);
#pragma unroll
        for (int j = 0; j < CPT; ++j) px = fmaf(silu_tc(z[j] + v->bh[c0 + j]), v->wh[c0 + j], px);
        tmem_ld<CPT>(tlane + kH_ACCH + kH, z);
#pragma unroll
        for (int j = 0; j < CPT; ++j) pX = fmaf(silu_tc(z[j] + v->bh[kH + c0 + j]), v->wh[kH + c0 + j], pX);
        v->spx[cg * kTM + row] = px;
        v->spX[cg * kTM + row] = pX;
        __syncthreads();
    VTR();
        float sx = 0.f, sX = 0.f;
#pragma unroll
        for (int g = 0; g < CG; ++g) { sx += v->spx[g * kTM + row]; sX += v->spX[g * kTM + row]; }
        sx = tanhf(sx); sX = tanhf(sX);
        gsx *= (1.f - sx * sx);
        gsX *= (1.f - sX * sX);
        __syncthreads();
    VTR();
      }
      float px = 0.f, pX = 0.f;
      tmem_ld<CPT>(tlane + kH_ACCH, z);
#pragma unroll
      for (int j = 0; j < CPT; ++j) {
        float d;
        silu_grad_tc(z[j] + v->bh[c0 + j], av[j], d);
        px = fmaf(av[j], v->wh[c0 + j], px);
        pwx[j] = fmaf(gsx, av[j], pwx[j]);
        z[j] = gsx * v->wh[c0 + j] * d;          // gzxv
      }
      tmem_st<CPT>(tlane + kH_OPA, z);
      mn_store_row_at<CPT>(TGH, row, cg * (CPT / 4), z);
      tmem_ld<CPT>(tlane + kH_ACCH + kH, z);
#pragma unroll
      for (int j = 0; j < CPT; ++j) {
        float d;
        silu_grad_tc(z[j] + v->bh[kH + c0 + j], av[j], d);
        pX = fmaf(av[j], v->wh[kH + c0 + j], pX);
        pwX[j] = fmaf(gsX, av[j], pwX[j]);
        z[j] = gsX * v->wh[kH + c0 + j] * d;     // gzX
      }
      tmem_st<CPT>(tlane + kH_OPA + kH, z);
      mn_store_row_at<CPT>(TGH, row, 16 + cg * (CPT / 4), z);
      v->spx[cg * kTM + row] = px;
      v->spX[cg * kTM + row] = pX;
      tmem_st_wait();
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    __syncthreads();
    VTR();
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
#pragma unroll
        for (int ks = 0; ks < 16; ++ks)                                            // gu(heads) = [gzxv | gzX] [Wxv ; WX]
          mma_ts(tmem + kH_ACCG, tmem + kH_OPA + ks * 8, desc_advance(dWHm, ks * 1024), id_gu, ks > 0);
        umma::commit(&v->bar[1]);
        gemm_wgrad(tmem + kH_RW, dTGH, dTU, id_w, !first_tile);                    // [dWxv ; dWX | db..] += [gzxv | gzX]^T [u | 1..]
        umma::commit(&v->bar[2]);
      }
      __syncwarp();
    }
    // ---- coordinate outputs that do not depend on the trunk (overlap the GEMMs)
    if (t < kTM) {
      float sx = 0.f, sX = 0.f;
#pragma unroll
      for (int g = 0; g < CG; ++g) { sx += v->spx[g * kTM + t]; sX += v->spX[g * kTM + t]; }
      if (use_tanh) { sx = tanhf(sx); sX = tanhf(sX); }
      const int key = v->g.skey[t];
      float gD[3] = {0, 0, 0};
      if (key >= 0) {
        const int b = key / C, c = key - b * C, jn = t / C;
        const float invC = 1.f / (float)C;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          gD[k] = -sx * v->g.sgxn[jn * 3 + k] * invC + sX * a.gDsum[((size_t)b * 3 + k) * C + c];
          if (!single) atomicAdd(a.gZ + ((size_t)b * 3 + k) * C + c, gD[k]);
        }
      }
      v->g.sgD[t * 3 + 0] = gD[0]; v->g.sgD[t * 3 + 1] = gD[1]; v->g.sgD[t * 3 + 2] = gD[2];
    }
    cp_async_wait();                           // this thread's share of the upstream dL/du rows has landed in SG
    __syncthreads();
    VTR();
    if (single && warp == NW - 1) small_from_rows(v->g.sgD, &v->acc, C, TN, lane);
    if (t < TN) {
      const int i = tile * TN + t;
      if (i < a.N) {
        const float di = a.dinv != nullptr ? a.dinv[i] : 1.f;
        float gsv = 0.f, gsg = 0.f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const float g = v->g.sgxn[t * 3 + k];
          float sum = 0.f;
          for (int c = 0; c < C; ++c) sum += v->g.sgD[(t * C + c) * 3 + k];
          // gt == NULL: virtual_bwd_gt_kernel wrote gt, and the edge backward may be adding its row and col terms to the
          // zeroed gx right now (fegnn_model_backward_inputs, "layer_overlap"), so this kernel and the trunk add too
          if (a.gt != nullptr) {
            a.gx[(size_t)i * 3 + k] = g - sum;        // the trunk kernel subtracts the rho term
            a.gt[(size_t)i * 3 + k] = g * di;
          } else {
            atomicAdd(a.gx + (size_t)i * 3 + k, g - sum);
          }
          if (a.stats != nullptr) {
            st_gt = fmaxf(st_gt, fabsf(g * di));
            st_x = fmaxf(st_x, fabsf(a.x[(size_t)i * 3 + k] - a.x[k]));
          }
          gsv = fmaf(g, a.v[(size_t)i * 3 + k], gsv);
          gsg = fmaf(g, a.grav[k], gsg);
        }
        a.gsv[i] = gsv;
        if (grav) a.gsg[i] = gsg;
      }
    }
    umma::mbar_wait(&v->bar[1], phase);
    VTR();
    umma::fence_after();
    // ---- epilogue 2: total dL/du of the row -> gu_work
    {
      float g[CPT];
      tmem_ld<CPT>(tlane + kH_ACCG, g);
      const int key = v->g.skey[row];
      if (key >= 0) {
        if (a.gu != nullptr) {
          float q[CPT];
          mn_load_row<CPT>(SG, row, cg, q);
#pragma unroll
          for (int j = 0; j < CPT; ++j) g[j] += q[j];
        }
        if (a.gUsum != nullptr) {
          const float4* src = reinterpret_cast<const float4*>(a.gUsum + (size_t)key * kH + c0);
#pragma unroll
          for (int ch = 0; ch < CPT / 4; ++ch) {
            const float4 q = src[ch];
            g[ch * 4] += q.x; g[ch * 4 + 1] += q.y; g[ch * 4 + 2] += q.z; g[ch * 4 + 3] += q.w;
          }
        }
        // gu_work: the tile's rows TRANSPOSED by 16-byte chunk -- chunk c16 of row r at tile base + (c16 * nrows + r) * 16 bytes --
        // so that the row owners' stores here and loads in the trunk kernel are contiguous across a warp.  In place over gu:
        // every upstream row of this tile was copied to SG before the barrier above.
        float4* dst = reinterpret_cast<float4*>(a.gu_work + tbase);
#pragma unroll
        for (int ch = 0; ch < CPT / 4; ++ch)
          dst[(size_t)(cg * (CPT / 4) + ch) * nrows + row] = make_float4(g[ch * 4], g[ch * 4 + 1], g[ch * 4 + 2], g[ch * 4 + 3]);
      }
    }
    phase ^= 1;
    first_tile = false;
  }
  acc_flush<NT>(&v->acc, cur_b, C, nullptr, a.gZ, nullptr);
  // ---- bound statistics of the edge backward (what its pre-pass kernel would compute from gt and x): one atomic pair per CTA
  if (a.stats != nullptr && warp < 4) {            // the threads t < TN <= 128 that wrote gt
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      st_gt = fmaxf(st_gt, __shfl_xor_sync(0xffffffffu, st_gt, o));
      st_x = fmaxf(st_x, __shfl_xor_sync(0xffffffffu, st_x, o));
    }
    if (lane == 0) {                               // non-negative floats order like their bit patterns
      atomicMax(a.stats + 0, __float_as_uint(st_gt));
      atomicMax(a.stats + 2, __float_as_uint(st_x));
    }
  }
  // ---- flush the weight gradients
  if (!first_tile) umma::mbar_wait(&v->bar[2], phase ^ 1);
    VTR();
  umma::fence_after();
  if constexpr (CPT == 16) {
    // the 2 x 16 per-row partial sums of a warp as ONE 32-column transposed reduction: 31 shuffles instead of 160
    float cs[32];
#pragma unroll
    for (int j = 0; j < 16; ++j) { cs[j] = pwx[j]; cs[16 + j] = pwX[j]; }
    const float tot = warp_colsum32(cs, lane);
    atomicAdd(&v->cwh[(lane < 16 ? c0 : kH + c0 - 16) + lane], tot);
  } else {
#pragma unroll
    for (int j = 0; j < CPT; ++j) {
      float sx = pwx[j], sX = pwX[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sx += __shfl_xor_sync(0xffffffffu, sx, o);
        sX += __shfl_xor_sync(0xffffffffu, sX, o);
      }
      if (lane == 0) {
        atomicAdd(&v->cwh[c0 + j], sx);
        atomicAdd(&v->cwh[kH + c0 + j], sX);
      }
    }
  }
  __syncthreads();
    VTR();
  if (!first_tile) {
    // RW: lane n = row of [dWxv ; dWX] (M = 128 layout: row m in lane m), columns 0-63 = k, column 64 = bias sum
    float w[CPT];
    tmem_ld<CPT>(tlane + kH_RW, w);
    float* gW = row < kH ? a.g_Wxv : a.g_WX;
    const int n = row & (kH - 1);
    if (gW != nullptr) {
      float* dst = gW + (size_t)n * kH + c0;
      if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
        for (int j = 0; j < CPT; j += 4) atomicAdd(reinterpret_cast<float4*>(dst + j), make_float4(w[j], w[j + 1], w[j + 2], w[j + 3]));
      } else {
#pragma unroll
        for (int j = 0; j < CPT; ++j) atomicAdd(dst + j, w[j]);
      }
    }
    if (cg == 0) {
      float x[16];
      tmem_ld<16>(tmem + ((uint32_t)(quarter * 32) << 16) + kH_RW + kH, x);
      float* gb = row < kH ? a.g_bxv : a.g_bX;
      if (gb != nullptr) atomicAdd(gb + n, x[0]);
    }
    if (t < 2 * kH) {
      float* gw = t < kH ? a.g_wxv : a.g_wX;
      if (gw != nullptr) atomicAdd(gw + (t & (kH - 1)), v->cwh[t]);
    }
  }
  umma::fence_before();
  __syncthreads();
    VTR();
  if (warp == 0) umma::tmem_dealloc<512>(tmem);
  VTR();
  VTR_PRINT("heads");
}

// ---- trunk kernel
struct TrunkVec {
  float vr[kH], c2[kH];
  BwdGeo g;
  float sgrp[4 * kTM];
  GraphAcc acc;
  uint64_t bar[3];
  uint32_t tmem_slot;
};
struct TrunkSmem {
  static constexpr int off_V2k = 0, off_V2m = 16384;
  static constexpr int off_AUX = 32768;                    // [128][32]; adjacent: B = [AUX | TA], N = 96
  static constexpr int off_TA = off_AUX + 16384;           // a1
  static constexpr int off_TG = off_TA + 32768;            // gz2 (A of the dV2 GEMM)
  static constexpr int off_TM = off_TG + 32768;            // gz1 (walks; A of the dvr GEMM)
  static constexpr int off_D1 = off_TM + 32768;            // silu'(z1) fp16
  static constexpr int off_vec = off_D1 + kTM * kH * 2;
  static constexpr size_t bytes = off_vec + sizeof(TrunkVec) + 1024;
};
constexpr uint32_t kT_ACC0 = 0, kT_ACC1 = 64, kT_R2 = 128, kT_DXZ = 224, kT_OPA = 256;     // 320 columns

template <int CG>
__global__ void __launch_bounds__(128 * CG, 1) virtual_bwd_trunk_tc_kernel(VirtArgs a) {
  VTR_DECL();
  constexpr int NT = 128 * CG, CPT = kH / CG, NW = NT / 32;
  using SM = TrunkSmem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
  pdl_trigger();
  TrunkVec* v = reinterpret_cast<TrunkVec*>(smem + SM::off_vec);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int quarter = warp & 3, cg = warp >> 2, row = quarter * 32 + lane, c0 = cg * CPT;
  const int C = a.C, TN = kTM / C;

  {
    WRegs<NT> w0;
    wregs_load<NT>(w0, a.V2, kH);
    wregs_store_kmajor<NT>(w0, smem + SM::off_V2k, 0, kH);
    wregs_store_mn<NT>(w0, smem + SM::off_V2m, 0, kH);
  }
  for (int i = t; i < kH; i += NT) {
    v->vr[i] = a.wv1[(size_t)i * a.ldv + 2 * kH];
    v->c2[i] = a.c2[i];
  }
  for (int i = t; i < kTM * 128 / 16; i += NT) reinterpret_cast<float4*>(smem + SM::off_AUX)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  acc_clear<NT>(&v->acc);
  if (t == 0) {
#pragma unroll
    for (int i = 0; i < 3; ++i) umma::mbar_init(&v->bar[i], 1);
    umma::mbar_fence_init();
  }
  if (warp == 0) umma::tmem_alloc<512>(&v->tmem_slot);
  umma::fence_smem_to_async();
  umma::fence_before();
  __syncthreads();
    VTR();
  umma::fence_after();
  pdl_wait();
  const uint32_t tmem = v->tmem_slot;
  const uint32_t tlane = tmem + ((uint32_t)(quarter * 32) << 16) + c0;
  const uint32_t id_k = idesc_tf32(128, 64, 0, 0), id_mn = idesc_tf32(128, 64, 0, 1);
  const uint32_t id_w96 = idesc_tf32(64, 96, 1, 1), id_aux = idesc_tf32(64, 32, 1, 1);
  const uint64_t dV2k = umma::make_desc(umma::smem_u32(smem + SM::off_V2k));
  const uint64_t dV2m = make_desc_mn(umma::smem_u32(smem + SM::off_V2m), kH * 128);
  const uint64_t dAUX = make_desc_mn(umma::smem_u32(smem + SM::off_AUX), kTM * 128);     // [AUX | TA]
  const uint64_t dTG = make_desc_mn(umma::smem_u32(smem + SM::off_TG), kTM * 128);
  const uint64_t dTM = make_desc_mn(umma::smem_u32(smem + SM::off_TM), kTM * 128);
  uint8_t* AUX = smem + SM::off_AUX;
  uint8_t* TA = smem + SM::off_TA;
  uint8_t* TG = smem + SM::off_TG;
  uint8_t* TM = smem + SM::off_TM;
  uint8_t* D1 = smem + SM::off_D1;
  uint32_t phase = 0;
  bool first_tile = true;
  int cur_b = -1;

  const int ntiles = (a.N + TN - 1) / TN;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    if (!first_tile) {                         // previous tile's last GEMMs still read AUX, TA, TG and TM
      umma::mbar_wait(&v->bar[2], phase ^ 1);
    VTR();
      umma::fence_after();
    }
    umma::fence_before();
    __syncthreads();
    VTR();
    bwd_geometry(a, &v->g, tile, TN, AUX);
    __syncthreads();
    VTR();
    const bool single = v->g.b_first == v->g.b_last;
    if (!single || v->g.b_first != cur_b) {
      const int nb = single ? v->g.b_first : -1;
      acc_flush<NT>(&v->acc, cur_b, C, a.gG1, a.gZ, nullptr);
      cur_b = nb;
    }
    // ---- assembly: a1 = silu(z1) -> TA, silu'(z1) -> D1 (fp16)
    {
      const int l16 = lane & 15, hsel = lane >> 4;
      const float4 vr = *reinterpret_cast<const float4*>(v->vr + 4 * l16);
      constexpr int RPW = kTM / NW;
#pragma unroll 1
      for (int i0 = 0; i0 < RPW; i0 += 8) {
        float4 p[4], g[4];
        int ki[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int rr = warp * RPW + i0 + 2 * j + hsel;
          ki[j] = v->g.skey[rr];
          p[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          g[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ki[j] >= 0) {
            p[j] = *reinterpret_cast<const float4*>(a.Av + (size_t)v->g.snode[rr] * kH + 4 * l16);
            g[j] = *reinterpret_cast<const float4*>(a.G1 + (size_t)ki[j] * kH + 4 * l16);
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int rr = warp * RPW + i0 + 2 * j + hsel;
          const float rho = v->g.srho[rr];
          float4 o = make_float4(0.f, 0.f, 0.f, 0.f), od = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ki[j] >= 0) {
            silu_grad_tc(p[j].x + g[j].x + rho * vr.x, o.x, od.x); silu_grad_tc(p[j].y + g[j].y + rho * vr.y, o.y, od.y);
            silu_grad_tc(p[j].z + g[j].z + rho * vr.z, o.z, od.z); silu_grad_tc(p[j].w + g[j].w + rho * vr.w, o.w, od.w);
          }
          *reinterpret_cast<float4*>(TA + mn_chunk_off(rr, l16, kTM)) = o;
          __half2 h01 = __floats2half2_rn(od.x, od.y), h23 = __floats2half2_rn(od.z, od.w);
          uint2 pk;
          pk.x = *reinterpret_cast<uint32_t*>(&h01);
          pk.y = *reinterpret_cast<uint32_t*>(&h23);
          *reinterpret_cast<uint2*>(D1 + rr * 128 + ((((l16 >> 1) ^ (rr & 7)) << 4) | ((l16 & 1) << 3))) = pk;
        }
      }
    }
    __syncthreads();
    VTR();
    {
      float a1[CPT];
      mn_load_row<CPT>(TA, row, cg, a1);
      tmem_st<CPT>(tlane + kT_OPA, a1);
      tmem_st_wait();
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    __syncthreads();
    VTR();
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
        gemm_ts_kmajor(tmem + kT_ACC0, tmem + kT_OPA, dV2k, id_k);                 // G1: z2 = a1 V2^T
        umma::commit(&v->bar[0]);
      }
      __syncwarp();
    }
    umma::mbar_wait(&v->bar[0], phase);
    VTR();
    umma::fence_after();
    // ---- epilogue 1: gz2 = dL/du * silu'(z2 + c2) -> tensor memory (A of ga1) and TG (A of dV2)
    {
      float z[CPT];
      tmem_ld<CPT>(tlane + kT_ACC0, z);
      const bool valid = v->g.skey[row] >= 0;
      if (valid) {
        // total dL/du of the row, written by the heads kernel transposed by 16-byte chunk (see there)
        const int nrows = min(TN, a.N - tile * TN) * C;
        const float4* src = reinterpret_cast<const float4*>(a.gu_work + (size_t)tile * TN * C * kH);
#pragma unroll
        for (int ch = 0; ch < CPT / 4; ++ch) {
          const float4 q = src[(size_t)(cg * (CPT / 4) + ch) * nrows + row];
          float u_, d;
          silu_grad_tc(z[ch * 4] + v->c2[c0 + ch * 4], u_, d); z[ch * 4] = q.x * d;
          silu_grad_tc(z[ch * 4 + 1] + v->c2[c0 + ch * 4 + 1], u_, d); z[ch * 4 + 1] = q.y * d;
          silu_grad_tc(z[ch * 4 + 2] + v->c2[c0 + ch * 4 + 2], u_, d); z[ch * 4 + 2] = q.z * d;
          silu_grad_tc(z[ch * 4 + 3] + v->c2[c0 + ch * 4 + 3], u_, d); z[ch * 4 + 3] = q.w * d;
        }
      } else {
#pragma unroll
        for (int j = 0; j < CPT; ++j) z[j] = 0.f;
      }
      tmem_st<CPT>(tlane + kT_OPA, z);
      mn_store_row<CPT>(TG, row, cg, z);
      tmem_st_wait();
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    __syncthreads();
    VTR();
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
        gemm_ts_mn(tmem + kT_ACC1, tmem + kT_OPA, dV2m, id_mn);                    // ga1 = gz2 V2
        umma::commit(&v->bar[1]);
        gemm_wgrad(tmem + kT_R2, dTG, dAUX, id_w96, !first_tile);                  // [dc2.. | dV2] += gz2^T [1, rho.. | a1]
      }
      __syncwarp();
    }
    umma::mbar_wait(&v->bar[1], phase);
    VTR();
    umma::fence_after();
    // ---- epilogue 2: gz1 = ga1 * silu'(z1) -> TM ; grho = gz1 . vr
    {
      float g1v[CPT];
      tmem_ld<CPT>(tlane + kT_ACC1, g1v);
      float gr = 0.f;
      if (v->g.skey[row] >= 0) {
#pragma unroll
        for (int c16 = 0; c16 < CPT / 8; ++c16) {
          const uint4 pk = *reinterpret_cast<const uint4*>(D1 + row * 128 + (((cg * (CPT / 8) + c16) ^ (row & 7)) << 4));
          const uint32_t w[4] = {pk.x, pk.y, pk.z, pk.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float2 dd = __half22float2(*reinterpret_cast<const __half2*>(&w[k]));
            const int j = c16 * 8 + k * 2;
            g1v[j] *= dd.x;
            g1v[j + 1] *= dd.y;
            gr = fmaf(g1v[j], v->vr[c0 + j], gr);
            gr = fmaf(g1v[j + 1], v->vr[c0 + j + 1], gr);
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < CPT; ++j) g1v[j] = 0.f;
      }
      mn_store_row<CPT>(TM, row, cg, g1v);
      v->sgrp[cg * kTM + row] = gr;
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    __syncthreads();
    VTR();
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
        gemm_wgrad(tmem + kT_DXZ, dTM, dAUX, id_aux, !first_tile);                 // dvr += gz1^T rho   (column 1)
        umma::commit(&v->bar[2]);
      }
      __syncwarp();
    }
    phase ^= 1;
    first_tile = false;
    // ---- outputs: gG1 by key, gAv by node, and the rho term of the coordinate gradients
    VTR();
    rows_to_graph<NT>(TM, v->g.skey, &v->acc, C, TN, single, a.gG1);
    VTR();
    {
      constexpr int GR = NT / 64;
      const int col = t & 63, grp = t >> 6;
      const uint32_t cbase = (col >> 5) * (kTM * 128) + ((col & 7) << 2);
      const int c8 = (col & 31) >> 3;
      // two nodes per trip with independent sums (the single-sum walk was a dependent shared-memory chain: 2 300 cycles per tile)
      auto at = [&](int r) { return *reinterpret_cast<const float*>(TM + cbase + r * 128 + ((c8 ^ (r & 3)) << 5)); };
      for (int jn = grp; jn < TN; jn += 2 * GR) {
        const int jb = jn + GR;
        const int ia = tile * TN + jn, ib = tile * TN + jb;
        const bool hb = jb < TN;                       // rows of nodes past N hold zeros
        float sa = 0.f, sb = 0.f;
        for (int c = 0; c < C; ++c) {
          sa += at(jn * C + c);
          if (hb) sb += at(jb * C + c);
        }
        if (ia < a.N) a.gAv[(size_t)ia * kH + col] = sa;
        if (hb && ib < a.N) a.gAv[(size_t)ib * kH + col] = sb;
      }
    }
    VTR();
    if (t < kTM) {
      const int key = v->g.skey[t];
      float gD[3] = {0, 0, 0};
      if (key >= 0) {
        const int b = key / C, c = key - b * C;
        float gr = 0.f;
#pragma unroll
        for (int g = 0; g < CG; ++g) gr += v->sgrp[g * kTM + t];
        const float rho = v->g.srho[t];
        const float f = rho > 0.f ? gr / rho : 0.f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          gD[k] = f * v->g.sD[t * 3 + k];
          if (!single) atomicAdd(a.gZ + ((size_t)b * 3 + k) * C + c, gD[k]);
        }
      }
      v->g.sgD[t * 3 + 0] = gD[0]; v->g.sgD[t * 3 + 1] = gD[1]; v->g.sgD[t * 3 + 2] = gD[2];
    }
    __syncthreads();
    VTR();
    if (single && warp == NW - 1) small_from_rows(v->g.sgD, &v->acc, C, TN, lane);
    if (t < TN) {
      const int i = tile * TN + t;
      if (i < a.N) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          float sum = 0.f;
          for (int c = 0; c < C; ++c) sum += v->g.sgD[(t * C + c) * 3 + k];
          if (a.gt != nullptr) a.gx[(size_t)i * 3 + k] -= sum;     // the heads kernel wrote g - (head terms)
          else atomicAdd(a.gx + (size_t)i * 3 + k, -sum);            // layer_overlap (see the heads kernel)
        }
      }
    }
  }
  acc_flush<NT>(&v->acc, cur_b, C, a.gG1, a.gZ, nullptr);
  if (!first_tile) umma::mbar_wait(&v->bar[2], phase ^ 1);
    VTR();
  umma::fence_after();
  if (!first_tile) {
    // R2 (M = 64 layout: row n in lane (n/16)*32 + n%16): columns 0-31 aux sums (0: dc2), 32-95: dV2[n][k]
    const int n = quarter * 16 + lane;
    float w[CPT];
    tmem_ld<CPT>(tlane + kT_R2 + 32, w);
    if (lane < 16 && a.g_V2 != nullptr) {
      float* dst = a.g_V2 + (size_t)n * kH + c0;
      if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
        for (int j = 0; j < CPT; j += 4) atomicAdd(reinterpret_cast<float4*>(dst + j), make_float4(w[j], w[j + 1], w[j + 2], w[j + 3]));
      } else {
#pragma unroll
        for (int j = 0; j < CPT; ++j) atomicAdd(dst + j, w[j]);
      }
    }
    if (cg == 0) {
      float x2[16], xz[16];
      const uint32_t tl = tmem + ((uint32_t)(quarter * 32) << 16);
      tmem_ld<16>(tl + kT_R2, x2);
      tmem_ld<16>(tl + kT_DXZ, xz);
      if (lane < 16) {
        if (a.g_c2 != nullptr) atomicAdd(a.g_c2 + n, x2[0]);
        if (a.g_wv1 != nullptr) atomicAdd(a.g_wv1 + (size_t)n * a.ldv + 2 * kH, xz[1]);
      }
    }
  }
  umma::fence_before();
  __syncthreads();
    VTR();
  if (warp == 0) umma::tmem_dealloc<512>(tmem);
  VTR();
  VTR_PRINT("trunk");
}

}  // namespace vtc

template <int CG, bool kDet = false, bool kSaved = false>
cudaError_t launch_virtual_fwd_tc(const VirtArgs& a, int sms, cudaStream_t st) {
  static DevOnce attr;
  const size_t bytes = vtc::FwdSmem::bytes;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(vtc::virtual_fwd_tc_kernel<CG, kDet, kSaved>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  const int TN = kTM / a.C;
  const int ntiles = (a.N + TN - 1) / TN;
  if (ntiles == 0) return cudaSuccess;
  const int grid = ntiles < 2 * sms ? ntiles : 2 * sms;
  if (cudaError_t e_ = launch_pdl(vtc::virtual_fwd_tc_kernel<CG, kDet, kSaved>, grid, 128 * CG, bytes, st, a)) return e_;
  return cudaGetLastError();
}

}  // namespace fegnn

namespace fegnn {
// grid = min(tiles, cap): cap = sms keeps one persistent CTA per SM; a larger cap leaves the extra tiles to the block
// scheduler, which places them wherever an SM frees up (next to the edge backward on another stream)
template <int CG>
cudaError_t launch_virtual_bwd_tc(const VirtArgs& a, int cap, cudaStream_t st) {
  static DevOnce attr;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(vtc::virtual_bwd_heads_tc_kernel<CG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)vtc::HeadsSmem::bytes);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(vtc::virtual_bwd_trunk_tc_kernel<CG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)vtc::TrunkSmem::bytes);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  const int TN = kTM / a.C;
  const int ntiles = (a.N + TN - 1) / TN;
  if (ntiles == 0) return cudaSuccess;
  const int grid = ntiles < cap ? ntiles : cap;
  if (cudaError_t e_ = launch_pdl(vtc::virtual_bwd_heads_tc_kernel<CG>, grid, 128 * CG, vtc::HeadsSmem::bytes, st, a)) return e_;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (cudaError_t e_ = launch_pdl(vtc::virtual_bwd_trunk_tc_kernel<CG>, grid, 128 * CG, vtc::TrunkSmem::bytes, st, a)) return e_;
  return cudaGetLastError();
}

// gt = (dL/dx'_i + gxsum_next[batch_i]) dinv_i, the coordinate gradient the edge backward gathers by row: the heads kernel's
// expression, formed ahead of the virtual backward so that the edge backward need not wait for it.  With `stats` it also
// folds max|gt| and max|x - x_0| into stats[0] / stats[2] (the FEGNN_F_STATS_READY bounds): one atomicMax pair per CTA.
// One thread per (node, component).  gx_new / gxsum_next come from the kernels ahead: plain loads after the wait.
constexpr int kGtThreads = 256;
__global__ void __launch_bounds__(kGtThreads) virtual_bwd_gt_kernel(int N, const float* __restrict__ x, const float* gx_new,
                                                                   const float* gxsum_next, const int* __restrict__ batch,
                                                                   const float* __restrict__ dinv, float* gt, unsigned* stats) {
  __shared__ float red[2][kGtThreads / 32];
  pdl_trigger();
  pdl_wait();
  const int idx = blockIdx.x * kGtThreads + threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float mg = 0.f, mx = 0.f;
  if (idx < N * 3) {
    const int i = idx / 3, k = idx - i * 3;
    float g = gx_new[idx];
    if (gxsum_next != nullptr) g += gxsum_next[batch[i] * 3 + k];
    g *= dinv != nullptr ? dinv[i] : 1.f;
    gt[idx] = g;
    mg = fabsf(g);
    mx = fabsf(x[idx] - x[k]);
  }
  if (stats == nullptr) return;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mg = fmaxf(mg, __shfl_xor_sync(0xffffffffu, mg, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if (lane == 0) { red[0][warp] = mg; red[1][warp] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kGtThreads / 32; ++w) { mg = fmaxf(mg, red[0][w]); mx = fmaxf(mx, red[1][w]); }
    atomicMax(stats + 0, __float_as_uint(mg));     // non-negative floats order like their bit patterns
    atomicMax(stats + 2, __float_as_uint(mx));
  }
}
inline cudaError_t launch_virtual_bwd_gt(const VirtArgs& a, unsigned* stats, cudaStream_t st) {
  if (a.N == 0) return cudaSuccess;
  if (cudaError_t e = launch_pdl(virtual_bwd_gt_kernel, (a.N * 3 + kGtThreads - 1) / kGtThreads, kGtThreads, 0, st, a.N, a.x,
                                 a.gx_new, a.gxsum_next, a.batch, a.dinv, a.gt, stats))
    return e;
  return cudaGetLastError();
}
}  // namespace fegnn
