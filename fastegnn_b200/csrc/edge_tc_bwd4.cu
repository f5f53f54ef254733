// edge_tc_bwd4.cu -- fourth tcgen05 formulation of the fused real-edge backward (edge_backward modes 7 / 8).
//
// Same contract as bwd2 / bwd3 (autograd of models/FastEGNN.py:102-108,125-129,156) and the same skeleton as bwd3
// (fp16 operand tiles, kind::f16 with fp32 accumulation, two independent thread groups per CTA = two 128-edge tiles in
// flight, one power-of-two scale per launch and gradient tensor).  bwd3 ran at 29 % issue utilisation with 23 k warp
// instructions per tile (ncu, profiles/ncu_bwd3_r2.txt): every warp is a serial chain of ~2 900 instructions per tile
// between four MMA round trips, so the chain length IS the tile latency.  This version cuts the chain:
//   * epilogue arithmetic on packed fp16 pairs (HFMA2 / tanh.approx.f16x2: SiLU and its derivative in 5 instructions per
//     PAIR instead of 6 per element), every scale folded into an existing multiply, the accumulator converted once;
//   * silu'(z1) lives in tensor memory (packed, 32 columns) instead of a shared-memory tile; the freed tile holds
//     a3 = silu(z3), so that dw4 = a3^T (gs) is one more N = 8 product against the aux tile: the 32 per-thread fp32
//     accumulators of dw4 and their shuffle reduction are gone (32 registers per thread);
//   * gQ (by col) and gP (by row) are scattered from the fp16 gz1 tile by half-warps that own whole rows: one
//     red.global.add.v4.f32 covers 2 rows x 256 contiguous bytes (the row-owner layout touched 32 different lines per
//     instruction: the scatter was 15 % of the kernel at 3.6 M edges);
//   * row dot products (s = w4 . a3, gq = gz1 . wq) as chunked packed sums exchanged through ONE barrier; 9 group
//     barriers per tile instead of 14;
//   * templated on the column groups per tile: CG = 2 (256 threads per tile, 32 columns per thread) or CG = 4 (512
//     threads per tile, 16 columns per thread, 1 024 threads per CTA).
// Precision: operands are fp16 as in bwd3 (10-bit mantissa = TF32); additionally the pre-activation is rounded to fp16
// before SiLU (tanh.approx.f16x2 has the same 2^-11 bound as tanh.approx.f32).  Stated tolerance: tests/gpu_util.py.
#include "common.cuh"
#include "umma.cuh"
#include <cuda_fp16.h>

namespace fegnn {
namespace bwd4 {

using bwd2::elect_one;
using bwd2::tmem_ld;
using bwd2::tmem_st_wait;
using bwd3::desc_add;
using bwd3::gemm_ts_k;
using bwd3::gemm_ts_mn;
using bwd3::gemm_wgrad;
using bwd3::h_chunk_off;
using bwd3::idesc_f16;
using bwd3::kTileBytes;
using bwd3::kWBytes;
using bwd3::make_desc_h;
using bwd3::pack2;
using bwd3::unpack2;

__device__ __forceinline__ uint32_t h2u(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }
__device__ __forceinline__ __half2 u2h(uint32_t u) { return *reinterpret_cast<__half2*>(&u); }
__device__ __forceinline__ __half2 tanh_h2(__half2 x) {
  uint32_t r;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(r) : "r"(h2u(x)));
  return u2h(r);
}
// t = z / 2 (packed pair)  ->  a = silu(z) = t (1 + tanh t),  d = silu'(z) = s + a (1 - s) with s = (1 + tanh t) / 2
__device__ __forceinline__ void silu_grad_h2(__half2 t, __half2& a, __half2& d) {
  const __half2 hf = __float2half2_rn(0.5f), nhf = __float2half2_rn(-0.5f);
  const __half2 th = tanh_h2(t);
  a = __hfma2(t, th, t);
  const __half2 s = __hfma2(th, hf, hf), oms = __hfma2(th, nhf, hf);
  d = __hfma2(a, oms, s);
}

template <int N>
__device__ __forceinline__ void tmem_stu(uint32_t taddr, const uint32_t (&p)[N]);
template <>
__device__ __forceinline__ void tmem_stu<16>(uint32_t taddr, const uint32_t (&p)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      :: "r"(taddr), "r"(p[0]), "r"(p[1]), "r"(p[2]), "r"(p[3]), "r"(p[4]), "r"(p[5]), "r"(p[6]), "r"(p[7]), "r"(p[8]),
         "r"(p[9]), "r"(p[10]), "r"(p[11]), "r"(p[12]), "r"(p[13]), "r"(p[14]), "r"(p[15]) : "memory");
}
template <>
__device__ __forceinline__ void tmem_stu<8>(uint32_t taddr, const uint32_t (&p)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "r"(taddr), "r"(p[0]), "r"(p[1]), "r"(p[2]), "r"(p[3]), "r"(p[4]), "r"(p[5]), "r"(p[6]), "r"(p[7])
               : "memory");
}
// packed loads WITHOUT the wait (pair them with an accumulator load, then tmem_ld_wait once)
template <int N>
__device__ __forceinline__ void tmem_ldu_nw(uint32_t taddr, uint32_t (&r)[N]);
template <>
__device__ __forceinline__ void tmem_ldu_nw<16>(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
template <>
__device__ __forceinline__ void tmem_ldu_nw<8>(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// this thread's CPT columns (column group cg) of row `row` <-> fp16 tile (CPT / 8 chunks of 16 bytes)
template <int NP>
__device__ __forceinline__ void store_row(uint8_t* tile, int row, int cg, const uint32_t (&p)[NP]) {
#pragma unroll
  for (int c = 0; c < NP / 4; ++c)
    *reinterpret_cast<uint4*>(tile + h_chunk_off(row, cg * (NP / 4) + c)) = make_uint4(p[4 * c], p[4 * c + 1], p[4 * c + 2], p[4 * c + 3]);
}
template <int NP>
__device__ __forceinline__ void load_row(const uint8_t* tile, int row, int cg, uint32_t (&p)[NP]) {
#pragma unroll
  for (int c = 0; c < NP / 4; ++c) {
    const uint4 u = *reinterpret_cast<const uint4*>(tile + h_chunk_off(row, cg * (NP / 4) + c));
    p[4 * c] = u.x; p[4 * c + 1] = u.y; p[4 * c + 2] = u.z; p[4 * c + 3] = u.w;
  }
}

struct SharedVec {                 // read-only after the prologue, all groups
  uint32_t hwqh[kH / 2], hWah[kTcMaxFe * kH / 2];   // packed fp16 0.5 wq, 0.5 Wa (the assembly forms t = z1 / 2 directly)
  float hb2[kH], hb3[kH];                   // 0.5 b2, 0.5 b3
  uint32_t w4b[kH / 2];                     // packed fp16 w4 * sb   (g3 = d3 * w4b * (gs sa))
  uint32_t w4d[kH / 2];                     // packed fp16 w4 * sdot (row dot s = w4 . a3)
  uint32_t wqs[kH / 2];                     // packed fp16 wq * swq  (row dot gq = gz1 . wq)
  float w4f[kH], wqf[kH];
  unsigned mw[2];                           // max |W2|, max |W3| (ordered uint bits)
  uint32_t tmem_slot;
};
struct Geo {                       // per-edge geometry of one tile
  int srow[kTM], scol[kTM];
  float sq[kTM], snrm[kTM], sd[kTM * 3], sgte[kTM * 3], sgs[kTM], sea[kTM * kTcMaxFe];
};
template <int CG>
struct GroupVec {
  Geo geo[2];                      // this tile's / the next tile's (written under the first MMA of this tile)
  int irow[kTM], icol[kTM];        // cp.async landing zone of the next tile's indices and edge attributes: slot tg is
  float iea[kTM * kTcMaxFe];       // written and read by thread tg only
  float spart[CG * kTM], sgqp[CG * kTM], ss[kTM];
  uint64_t bar[6];
  int qt[4];                       // this group's tiles: slot n & 3 holds its n-th (current, next, the one after)
  int had;                         // the group processed a tile (its weight-gradient lanes are defined)
};
__device__ __forceinline__ void cp_async4(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(umma::smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
template <int CG>
struct Smem4 {
  static constexpr int off_W2 = 0, off_W3 = kWBytes;
  static constexpr int off_groups = 2 * kWBytes;
  // per group: TA | TM | AUX | TG | T3   ([TM | AUX] and [TA | .. | AUX] are the two-block B operands of the weight-gradient
  // GEMMs; T3 holds silu'(z1) between the assembly and its move to tensor memory, then a3 = silu(z3) for the dw4 product)
  static constexpr int g_TA = 0, g_TM = kTileBytes, g_AUX = 2 * kTileBytes, g_TG = 3 * kTileBytes, g_T3 = 4 * kTileBytes;
  static constexpr int g_vec = 5 * kTileBytes;
  static constexpr int g_bytes = ((g_vec + (int)sizeof(GroupVec<CG>) + 1023) / 1024) * 1024;
  static constexpr int off_svec = off_groups + 2 * g_bytes;
  static constexpr size_t bytes = off_svec + sizeof(SharedVec) + 1024;
};
// tensor-memory columns: group g uses [160 g, 160 g + 160); the weight-gradient accumulators (M = 64) are shared, group 0
// at lane 0 and group 1 at lane 16 of the same columns
constexpr uint32_t kACC = 0, kOPA = 64, kD2T = 96, kD1T = 128, kGroupCols = 160;
constexpr uint32_t kR3 = 320, kR2 = 392, kDXZ = 464, kDW4 = 472;      // [dW3 64 | aux 8] [dW2 64 | aux 8] [aux 8] [aux 8]

__device__ __forceinline__ float pow2_to(float bound, int e_target) {   // largest power of two s with bound * s <= 2^e_target
  if (!(bound > 0.f) || !(bound < 3.0e38f)) return 1.f;
  int e;
  frexpf(bound, &e);                         // bound = f * 2^e, f in [0.5, 1)
  e = e_target - e;
  e = e < -60 ? -60 : (e > 60 ? 60 : e);
  return ldexpf(1.f, e);
}

// kEa: also g_ea[perm[e]][f] += gz1[e] . Wa_f (edge_attr enters phi_e's first Linear only), from the fp16 gz1 values of
// epilogue 4 and the packed 0.5 Wa of the assembly, widened to fp32 and accumulated in fp32.  The per-column-group partials
// go to T3, which holds nothing between the dw4 GEMM (waited in epilogue 3) and the next tile's assembly; the edge's owning
// thread sums them in the tail.
//
// claim: NULL = static split (group G of CTA b takes tiles 2 b + G + n 2 gridDim.x); else a zeroed counter from which
// each group takes its tiles one at a time, two ahead of the one it works on, so that a CTA that starts late (its SM held
// by a kernel of another stream) takes what is left instead of a fixed share.
//
// kLive: the live edge count (live_edges, read after the wait) bounds the tiles, the static split and the dynamic claim,
// instead of the capacity a.E that sized the grid
template <int CG, bool kEa, bool kLive = false>
__global__ void __launch_bounds__(256 * CG, 1) edge_bwd_tc4_kernel(EdgeArgs a, const unsigned* stats, unsigned* claim) {
  VTR_DECL();
  constexpr int NTG = 128 * CG, NT = 2 * NTG, CPT = kH / CG, NP = CPT / 2, NWG = NTG / 32, RPW = kTM / NWG;
  using SM = Smem4<CG>;
  using GV = GroupVec<CG>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
  SharedVec* sv = reinterpret_cast<SharedVec*>(smem + SM::off_svec);
  const int t = threadIdx.x, G = t / NTG, tg = t - G * NTG, wg = tg >> 5, lane = t & 31;
  const int quarter = wg & 3, cg = wg >> 2, row = quarter * 32 + lane, c0 = cg * CPT;
  uint8_t* gs = smem + SM::off_groups + G * SM::g_bytes;
  GV* v = reinterpret_cast<GV*>(gs + SM::g_vec);
  uint8_t *TA = gs + SM::g_TA, *TM = gs + SM::g_TM, *AUX = gs + SM::g_AUX, *TG = gs + SM::g_TG, *T3 = gs + SM::g_T3;
  const bool use_tanh = a.flags & FEGNN_F_TANH, norm = a.flags & FEGNN_F_NORMALIZE;
  auto group_sync = [&]() { asm volatile("bar.sync %0, %1;" :: "r"(1 + G), "n"(NTG) : "memory"); };
  pdl_trigger();

  // ---- prologue (whole CTA): fp16 weight tiles (+ their max magnitudes), fp32 vectors, zero AUX, barriers, tensor memory
  float mw2 = 0.f, mw3 = 0.f;
  for (int i = t; i < kH * 8; i += NT) {                   // 64 rows x 8 chunks of 8 columns
    const int n = i >> 3, c8 = i & 7;
    const float4 w20 = *reinterpret_cast<const float4*>(a.W2 + (size_t)n * kH + c8 * 8);
    const float4 w21 = *reinterpret_cast<const float4*>(a.W2 + (size_t)n * kH + c8 * 8 + 4);
    const float4 w30 = *reinterpret_cast<const float4*>(a.W3 + (size_t)n * kH + c8 * 8);
    const float4 w31 = *reinterpret_cast<const float4*>(a.W3 + (size_t)n * kH + c8 * 8 + 4);
    *reinterpret_cast<uint4*>(smem + SM::off_W2 + h_chunk_off(n, c8)) =
        make_uint4(pack2(w20.x, w20.y), pack2(w20.z, w20.w), pack2(w21.x, w21.y), pack2(w21.z, w21.w));
    *reinterpret_cast<uint4*>(smem + SM::off_W3 + h_chunk_off(n, c8)) =
        make_uint4(pack2(w30.x, w30.y), pack2(w30.z, w30.w), pack2(w31.x, w31.y), pack2(w31.z, w31.w));
    mw2 = fmaxf(mw2, fmaxf(fmaxf(fmaxf(fabsf(w20.x), fabsf(w20.y)), fmaxf(fabsf(w20.z), fabsf(w20.w))),
                           fmaxf(fmaxf(fabsf(w21.x), fabsf(w21.y)), fmaxf(fabsf(w21.z), fabsf(w21.w)))));
    mw3 = fmaxf(mw3, fmaxf(fmaxf(fmaxf(fabsf(w30.x), fabsf(w30.y)), fmaxf(fabsf(w30.z), fabsf(w30.w))),
                           fmaxf(fmaxf(fabsf(w31.x), fabsf(w31.y)), fmaxf(fabsf(w31.z), fabsf(w31.w)))));
  }
  for (int o = 16; o > 0; o >>= 1) {
    mw2 = fmaxf(mw2, __shfl_xor_sync(0xffffffffu, mw2, o));
    mw3 = fmaxf(mw3, __shfl_xor_sync(0xffffffffu, mw3, o));
  }
  if (t == 0) { sv->mw[0] = 0u; sv->mw[1] = 0u; }
  for (int i = t; i < kH; i += NT) {
    const float wq = a.w1[(size_t)i * a.ld1 + 2 * kH];
    sv->wqf[i] = wq;
    {
      __half* hq = reinterpret_cast<__half*>(sv->hwqh);
      __half* ha = reinterpret_cast<__half*>(sv->hWah);
      hq[i] = __float2half_rn(0.5f * wq);
#pragma unroll
      for (int f = 0; f < kTcMaxFe; ++f)
        ha[f * kH + i] = __float2half_rn(f < a.Fe ? 0.5f * a.w1[(size_t)i * a.ld1 + 2 * kH + 1 + f] : 0.f);
    }
    sv->hb2[i] = 0.5f * a.b2[i];
    sv->hb3[i] = 0.5f * a.b3[i];
    sv->w4f[i] = a.w4[i];
  }
  for (int i = tg; i < kTileBytes / 16; i += NTG) reinterpret_cast<uint4*>(AUX)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (tg == 0) {
#pragma unroll
    for (int i = 0; i < 6; ++i) umma::mbar_init(&v->bar[i], 1);
    umma::mbar_fence_init();
  }
  if (t < 32) umma::tmem_alloc<512>(&sv->tmem_slot);
  __syncthreads();                               // mw[] zeroed, fp32 vectors staged
    VTR();
  if (lane == 0) {
    atomicMax(&sv->mw[0], __float_as_uint(mw2));
    atomicMax(&sv->mw[1], __float_as_uint(mw3));
  }
  __syncthreads();
    VTR();
  pdl_wait();                                    // everything above read weights only; `stats` comes from the pre-pass
  if constexpr (kLive) a.E = live_edges(a);
  // ---- per-launch power-of-two scales (every thread, identical arithmetic).  Bounds from the pre-pass `stats`:
  //      |gs| <= dmax * sqrt3 * max|gt|  ->  sa ;  |w4| -> sb ;  g3 is stored times s3 = sa sb (<= 2^14)
  //      |g2| <= (max|gm| + 64 |g3| max|W3|) -> s2 ;  |gz1| <= 64 |g2| max|W2| -> s1   (stored values <= 2^15)
  float sa, sb, s2, s1, sdot, swq;
  {
    float mw4 = 0.f, mwq = 0.f;
    for (int i = 0; i < kH; ++i) {
      mw4 = fmaxf(mw4, fabsf(sv->w4f[i]));
      mwq = fmaxf(mwq, fabsf(sv->wqf[i]));
    }
    // (no const __restrict__ / ld.global.nc on `stats`: the compiler would hoist those loads above griddepcontrol.wait)
    const float mgt = __uint_as_float(__ldcg(stats)), mgm = __uint_as_float(__ldcg(stats + 1)), ext = 2.f * __uint_as_float(__ldcg(stats + 2));
    const float dmax = norm ? 1.f : ext * 1.7320508f;
    const float bgs = dmax * mgt * 1.7320508f * 1.05f;
    sa = pow2_to(bgs, 7);
    sb = pow2_to(mw4 * 1.1f, 7);
    const float b3 = bgs * mw4 * 1.1f;
    const float b2 = (mgm + 64.f * b3 * __uint_as_float(sv->mw[1])) * 1.1f;
    const float b1 = 64.f * b2 * __uint_as_float(sv->mw[0]) * 1.1f;
    s2 = pow2_to(b2, 15);
    s1 = pow2_to(b1, 15);
    sdot = pow2_to(mw4, 3);
    swq = pow2_to(mwq, -5);
  }
  for (int i = t; i < kH / 2; i += NT) {
    sv->w4b[i] = pack2(sv->w4f[2 * i] * sb, sv->w4f[2 * i + 1] * sb);
    sv->w4d[i] = pack2(sv->w4f[2 * i] * sdot, sv->w4f[2 * i + 1] * sdot);
    sv->wqs[i] = pack2(sv->wqf[2 * i] * swq, sv->wqf[2 * i + 1] * swq);
  }
  umma::fence_smem_to_async();
  umma::fence_before();
  __syncthreads();
    VTR();
  umma::fence_after();
  const uint32_t tmem = sv->tmem_slot;
  const float s3 = sa * sb;
  const float k32 = s2 / s3, k21 = s1 / s2;                                         // exact: powers of two
  const float r3 = 1.f / s3, r2 = 1.f / s2, r1 = 1.f / s1, ra = 1.f / sa, rdot = 1.f / sdot, rq = 1.f / (s1 * swq);
  const uint32_t tbase = tmem + G * kGroupCols;                                     // this group's columns
  const uint32_t tlane = tbase + ((uint32_t)(quarter * 32) << 16);                  // + this thread's lane
  const uint32_t twg = tmem + ((uint32_t)(16 * G) << 16);                           // weight-gradient accumulators: lane 0 / 16
  const uint32_t id_k = idesc_f16(128, 64, 0, 0), id_mn = idesc_f16(128, 64, 0, 1);
  const uint32_t id_wg72 = idesc_f16(64, 72, 1, 1), id_aux = idesc_f16(64, 8, 1, 1);
  const uint64_t dW2k = make_desc_h(umma::smem_u32(smem + SM::off_W2), 16), dW3k = make_desc_h(umma::smem_u32(smem + SM::off_W3), 16);
  const uint64_t dW2m = make_desc_h(umma::smem_u32(smem + SM::off_W2), kWBytes), dW3m = make_desc_h(umma::smem_u32(smem + SM::off_W3), kWBytes);
  const uint64_t dTG = make_desc_h(umma::smem_u32(TG), kTileBytes);               // A of the weight-gradient GEMMs (M = 64: one block)
  const uint64_t dTM_AUX = make_desc_h(umma::smem_u32(TM), kTileBytes);           // B = [TM | AUX], N = 72
  const uint64_t dTA_AUX = make_desc_h(umma::smem_u32(TA), 2 * kTileBytes);       // B = [TA | AUX], N = 72
  const uint64_t dTMa = make_desc_h(umma::smem_u32(TM), kTileBytes);              // A = gz1 (after m is dead)
  const uint64_t dT3a = make_desc_h(umma::smem_u32(T3), kTileBytes);              // A = a3
  const uint64_t dAUX = make_desc_h(umma::smem_u32(AUX), kTileBytes);             // B = AUX, N = 8
  bool first_tile = true;
  const int l16 = lane & 15, hsel = lane >> 4;

  const int ntiles = (a.E + kTM - 1) / kTM;
  // the tile after `prev` of this group (one thread per group asks; the answer goes through v->qt)
  auto claim_tile = [&](int prev) { return claim != nullptr ? (int)atomicAdd(claim, 1u) : prev + (int)gridDim.x * 2; };
  // indices / edge attributes of tile `tl` -> this thread's landing slots (asynchronous; rows past E get row = -1)
  auto load_idx_async = [&](int tl) {
    const int e = tl * kTM + tg;
    if (e < a.E) {
      cp_async4(&v->irow[tg], a.row + e);
      cp_async4(&v->icol[tg], a.col + e);
      for (int f = 0; f < a.Fe; ++f) cp_async4(&v->iea[tg * kTcMaxFe + f], a.ea + (size_t)e * a.Fe + f);
    } else {
      v->irow[tg] = -1;
    }
  };
  // one thread per edge: landed indices -> x / gt gathers -> geometry of the tile into `gg`
  auto geometry = [&](Geo* gg) {
    cp_async_wait_all();
    const int r = v->irow[tg];
    int c = 0;
    float d0 = 0, d1 = 0, d2 = 0, q = 0, nrm = 1.f, g0 = 0, g1 = 0, g2 = 0;
    float ea[kTcMaxFe];
#pragma unroll
    for (int f = 0; f < kTcMaxFe; ++f) ea[f] = 0.f;
    if (r >= 0) {
      c = v->icol[tg];
      d0 = a.x[(size_t)r * 3 + 0] - a.x[(size_t)c * 3 + 0];
      d1 = a.x[(size_t)r * 3 + 1] - a.x[(size_t)c * 3 + 1];
      d2 = a.x[(size_t)r * 3 + 2] - a.x[(size_t)c * 3 + 2];
      q = d0 * d0 + d1 * d1 + d2 * d2;
      g0 = a.gt[(size_t)r * 3 + 0]; g1 = a.gt[(size_t)r * 3 + 1]; g2 = a.gt[(size_t)r * 3 + 2];
#pragma unroll
      for (int f = 0; f < kTcMaxFe; ++f)
        if (f < a.Fe) ea[f] = v->iea[tg * kTcMaxFe + f];
    }
#pragma unroll
    for (int f = 0; f < kTcMaxFe; ++f) gg->sea[tg * kTcMaxFe + f] = ea[f];
    gg->sd[tg * 3 + 0] = d0; gg->sd[tg * 3 + 1] = d1; gg->sd[tg * 3 + 2] = d2;
    if (norm) {
      nrm = sqrtf(q) + a.eps;
      const float inv = 1.f / nrm;
      d0 *= inv; d1 *= inv; d2 *= inv;
    }
    gg->srow[tg] = r;
    gg->scol[tg] = c;
    gg->sq[tg] = q;
    gg->snrm[tg] = nrm;
    gg->sgte[tg * 3 + 0] = g0; gg->sgte[tg * 3 + 1] = g1; gg->sgte[tg * 3 + 2] = g2;
    gg->sgs[tg] = d0 * g0 + d1 * g1 + d2 * g2;
  };
  if (tg == 0) {
    v->qt[0] = claim != nullptr ? (int)atomicAdd(claim, 1u) : (int)blockIdx.x * 2 + G;
    v->qt[1] = claim_tile(v->qt[0]);
  }
  group_sync();
  if (tg < kTM && v->qt[0] < ntiles) {                   // first tile: nothing to hide the gathers under
    load_idx_async(v->qt[0]);
    geometry(&v->geo[0]);
    if (v->qt[1] < ntiles) load_idx_async(v->qt[1]);
  }
  // k: this group's tile count; its tile is v->qt[k & 3] (the ids stay in shared memory: the kernel is at its register cap)
  // the mbarrier phase of tile k is k & 1
  int k = 0;
  for (; v->qt[k & 3] < ntiles; ++k) {
    const uint32_t phase = k & 1;
    const Geo* geo = &v->geo[k & 1];
    if (tg == 0) v->qt[(k + 2) & 3] = claim_tile(v->qt[(k + 1) & 3]);   // read after the group barriers below; its slot was last read in tile k - 1
    if (!first_tile) {                           // the previous tile's last GEMMs still read AUX, TM, TA, TG
      umma::mbar_wait(&v->bar[4], phase ^ 1);
    VTR();
      umma::fence_after();
    }
    umma::fence_before();
    group_sync();
    VTR();
    // ---- aux columns (1, q, ea0..ea3, gs sa [written in epilogue 2], 0) = chunk 0 of the row, from the geometry that was
    //      computed one tile ahead
    if (tg < kTM)
      *reinterpret_cast<uint4*>(AUX + h_chunk_off(tg, 0)) =
          make_uint4(pack2(geo->srow[tg] >= 0 ? 1.f : 0.f, geo->sq[tg]), pack2(geo->sea[tg * kTcMaxFe], geo->sea[tg * kTcMaxFe + 1]),
                     pack2(geo->sea[tg * kTcMaxFe + 2], geo->sea[tg * kTcMaxFe + 3]), 0u);
    group_sync();
    VTR();
    // ---- assembly: t = z1 / 2 (P + Q in fp32, then packed), a1 = silu(z1) -> TA, silu'(z1) -> T3 (both fp16).  Half-warp per row, 4 columns
    //      per lane.  Rows past E carry t = 0 (a1 = 0, silu' = 1/2): their upstream gradients are zero.
    {
      // rank-(1 + Fe) update q wq + sum_f ea_f Wa_f on packed pairs (constants hoisted: 2 + 2 Fe registers)
      const uint2 wqh = *reinterpret_cast<const uint2*>(sv->hwqh + 2 * l16);
      uint2 wah[kTcMaxFe];
#pragma unroll
      for (int f = 0; f < kTcMaxFe; ++f) wah[f] = *reinterpret_cast<const uint2*>(sv->hWah + f * (kH / 2) + 2 * l16);
      const __half2 hf = __float2half2_rn(0.5f);
      constexpr int JB = CG == 2 ? 4 : 2;        // rows per half-warp and iteration
#pragma unroll 1
      for (int i0 = 0; i0 < RPW; i0 += 2 * JB) {
        float4 p[JB], qv[JB];
#pragma unroll
        for (int j = 0; j < JB; ++j) {
          const int rr = wg * RPW + i0 + 2 * j + hsel;
          const int ri = geo->srow[rr];
          p[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          qv[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ri >= 0 && !(a.exp & 4u)) {
            p[j] = *reinterpret_cast<const float4*>(a.P + (size_t)ri * kH + 4 * l16);
            qv[j] = *reinterpret_cast<const float4*>(a.Q + (size_t)geo->scol[rr] * kH + 4 * l16);
          }
        }
#pragma unroll
        for (int j = 0; j < JB; ++j) {
          const int rr = wg * RPW + i0 + 2 * j + hsel;
          const __half2 q2 = __float2half2_rn(geo->sq[rr]);
          __half2 u01 = __hmul2(q2, u2h(wqh.x)), u23 = __hmul2(q2, u2h(wqh.y));
#pragma unroll
          for (int f = 0; f < kTcMaxFe; ++f) {
            if (f < a.Fe) {
              const __half2 e2 = __float2half2_rn(geo->sea[rr * kTcMaxFe + f]);
              u01 = __hfma2(e2, u2h(wah[f].x), u01);
              u23 = __hfma2(e2, u2h(wah[f].y), u23);
            }
          }
          const __half2 t01 = __hfma2(__floats2half2_rn(p[j].x + qv[j].x, p[j].y + qv[j].y), hf, u01);
          const __half2 t23 = __hfma2(__floats2half2_rn(p[j].z + qv[j].z, p[j].w + qv[j].w), hf, u23);
          __half2 a01, d01, a23, d23;
          silu_grad_h2(t01, a01, d01);
          silu_grad_h2(t23, a23, d23);
          const uint32_t off = h_chunk_off(rr, l16 >> 1) + ((l16 & 1) << 3);       // 4 fp16 = half a chunk
          *reinterpret_cast<uint2*>(TA + off) = make_uint2(h2u(a01), h2u(a23));
          *reinterpret_cast<uint2*>(T3 + off) = make_uint2(h2u(d01), h2u(d23));
        }
      }
    }
    group_sync();
    VTR();
    // ---- row owners move a1 (A operand of G1) and silu'(z1) into tensor memory
    {
      uint32_t p[NP], pd[NP];
      load_row<NP>(TA, row, cg, p);
      load_row<NP>(T3, row, cg, pd);
      tmem_stu<NP>(tlane + kOPA + cg * NP, p);
      tmem_stu<NP>(tlane + kD1T + cg * NP, pd);
      tmem_st_wait();
    }
    umma::fence_smem_to_async();       // TA / AUX: generic-proxy writes -> visible to the tensor core
    umma::fence_before();
    group_sync();
    VTR();
    if (wg == 0) {
      umma::fence_after();
      if (elect_one()) {
        gemm_ts_k(tbase + kACC, tbase + kOPA, dW2k, id_k);                      // G1: z2 = a1 W2^T
        umma::commit(&v->bar[0]);
      }
      __syncwarp();
    }
    // ---- under G1: geometry of the NEXT tile (its indices landed long ago), then the indices of the one after
    if (tg < kTM && v->qt[(k + 1) & 3] < ntiles) {
      geometry(&v->geo[(k & 1) ^ 1]);
      if (v->qt[(k + 2) & 3] < ntiles) load_idx_async(v->qt[(k + 2) & 3]);
    }
    umma::mbar_wait(&v->bar[0], phase);
    VTR();
    umma::fence_after();
    // ---- epilogue 1: m = silu(z2 + b2) -> A operand and TM ; silu'(z2) -> D2T
    {
      float z[CPT];
      uint32_t pm[NP], pd[NP];
      tmem_ld<CPT>(tlane + kACC + c0, z);
#pragma unroll
      for (int j = 0; j < CPT; j += 4) {
        const float4 hb = *reinterpret_cast<const float4*>(sv->hb2 + c0 + j);
        __half2 a0, e0, a1v, e1;
        silu_grad_h2(__floats2half2_rn(fmaf(z[j], 0.5f, hb.x), fmaf(z[j + 1], 0.5f, hb.y)), a0, e0);
        silu_grad_h2(__floats2half2_rn(fmaf(z[j + 2], 0.5f, hb.z), fmaf(z[j + 3], 0.5f, hb.w)), a1v, e1);
        pm[j >> 1] = h2u(a0); pm[(j >> 1) + 1] = h2u(a1v);
        pd[j >> 1] = h2u(e0); pd[(j >> 1) + 1] = h2u(e1);
      }
      tmem_stu<NP>(tlane + kOPA + cg * NP, pm);
      tmem_stu<NP>(tlane + kD2T + cg * NP, pd);
      store_row<NP>(TM, row, cg, pm);
      tmem_st_wait();
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    group_sync();
    VTR();
    if (wg == 0) {
      umma::fence_after();
      if (elect_one()) {
        gemm_ts_k(tbase + kACC, tbase + kOPA, dW3k, id_k);                      // G2: z3 = m W3^T
        umma::commit(&v->bar[1]);
      }
      __syncwarp();
    }
    umma::mbar_wait(&v->bar[1], phase);
    VTR();
    umma::fence_after();
    // ---- epilogue 2: a3 = silu(z3 + b3) -> T3, s = w4 . a3 ; g3 = (gs sa) (w4 sb) silu'(z3) -> A operand and TG
    {
      float z[CPT];
      uint32_t pa[NP], pd[NP];
      tmem_ld<CPT>(tlane + kACC + c0, z);
      float part = 0.f;
#pragma unroll
      for (int j = 0; j < CPT; j += 8) {          // chunks of 4 pairs: packed partial dot, widened once per chunk
        __half2 cs = __float2half2_rn(0.f);
#pragma unroll
        for (int k = 0; k < 8; k += 4) {
          const float4 hb = *reinterpret_cast<const float4*>(sv->hb3 + c0 + j + k);
          const uint2 wd = *reinterpret_cast<const uint2*>(sv->w4d + ((c0 + j + k) >> 1));
          __half2 a0, e0, a1v, e1;
          silu_grad_h2(__floats2half2_rn(fmaf(z[j + k], 0.5f, hb.x), fmaf(z[j + k + 1], 0.5f, hb.y)), a0, e0);
          silu_grad_h2(__floats2half2_rn(fmaf(z[j + k + 2], 0.5f, hb.z), fmaf(z[j + k + 3], 0.5f, hb.w)), a1v, e1);
          cs = __hfma2(a0, u2h(wd.x), cs);
          cs = __hfma2(a1v, u2h(wd.y), cs);
          pa[(j + k) >> 1] = h2u(a0); pa[((j + k) >> 1) + 1] = h2u(a1v);
          pd[(j + k) >> 1] = h2u(e0); pd[((j + k) >> 1) + 1] = h2u(e1);
        }
        const float2 f = __half22float2(cs);
        part += f.x + f.y;
      }
      v->spart[cg * kTM + row] = part;
      store_row<NP>(T3, row, cg, pa);
      group_sync();
    VTR();
      float s = 0.f;
#pragma unroll
      for (int g = 0; g < CG; ++g) s += v->spart[g * kTM + row];
      s *= rdot;
      float gsv = geo->sgs[row];
      if (use_tanh) {
        s = tanhf(s);
        gsv *= (1.f - s * s);
      }
      const __half gh = __float2half_rn(gsv * sa);
      if (cg == 0) {
        v->ss[row] = s;
        *reinterpret_cast<__half*>(AUX + h_chunk_off(row, 0) + 12) = gh;          // aux column 6
      }
      const __half2 gh2 = __half2half2(gh);
#pragma unroll
      for (int j = 0; j < NP; j += 2) {
        const uint2 wb = *reinterpret_cast<const uint2*>(sv->w4b + (c0 >> 1) + j);
        pd[j] = h2u(__hmul2(__hmul2(u2h(pd[j]), u2h(wb.x)), gh2));
        pd[j + 1] = h2u(__hmul2(__hmul2(u2h(pd[j + 1]), u2h(wb.y)), gh2));
      }
      tmem_stu<NP>(tlane + kOPA + cg * NP, pd);
      store_row<NP>(TG, row, cg, pd);
      tmem_st_wait();
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    group_sync();
    VTR();
    if (wg == 0) {
      umma::fence_after();
      if (elect_one()) {
        gemm_ts_mn(tbase + kACC, tbase + kOPA, dW3m, id_mn);                    // D3 : g3 W3
        umma::commit(&v->bar[2]);
        gemm_wgrad(twg + kR3, dTG, dTM_AUX, id_wg72, !first_tile);              // [dW3 | db3 ..] += g3^T [m | 1, q, ea, gs]
        gemm_wgrad(twg + kDW4, dT3a, dAUX, id_aux, !first_tile);                // [.. dw4 ..]   += a3^T [.. gs ..]  (column 6)
        umma::commit(&v->bar[5]);                                               // TG / TM / T3 may be overwritten after this
      }
      __syncwarp();
    }
    // ---- epilogue 3: g2 = (gm[row] + g3 W3) * silu'(z2) (times s2) -> A operand and TG.  gm is fetched under the MMA.
    {
      float u[CPT];
      const int r = geo->srow[row];
      if (r >= 0 && a.gm != nullptr) {
        const float4* gmr = reinterpret_cast<const float4*>(a.gm + (size_t)r * kH + c0);
#pragma unroll
        for (int ch = 0; ch < CPT / 4; ++ch) {
          const float4 g = gmr[ch];
          u[ch * 4] = g.x * s2; u[ch * 4 + 1] = g.y * s2; u[ch * 4 + 2] = g.z * s2; u[ch * 4 + 3] = g.w * s2;
        }
      } else {
#pragma unroll
        for (int j = 0; j < CPT; ++j) u[j] = 0.f;
      }
      umma::mbar_wait(&v->bar[2], phase);
    VTR();
      umma::fence_after();
      float acc[CPT];
      uint32_t pd[NP];
      tmem_ldu_nw<NP>(tlane + kD2T + cg * NP, pd);
      tmem_ld<CPT>(tlane + kACC + c0, acc);      // (waits for both loads)
#pragma unroll
      for (int j = 0; j < CPT; j += 2)
        pd[j >> 1] = h2u(__hmul2(__floats2half2_rn(fmaf(acc[j], k32, u[j]), fmaf(acc[j + 1], k32, u[j + 1])), u2h(pd[j >> 1])));
      tmem_stu<NP>(tlane + kOPA + cg * NP, pd);
      umma::mbar_wait(&v->bar[5], phase);        // the dW3 / dw4 GEMMs have finished reading TG (g3), TM (m), T3 (a3)
    VTR();
      store_row<NP>(TG, row, cg, pd);
      tmem_st_wait();
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    group_sync();
    VTR();
    if (wg == 0) {
      umma::fence_after();
      if (elect_one()) {
        gemm_ts_mn(tbase + kACC, tbase + kOPA, dW2m, id_mn);                    // D2 : g2 W2
        umma::commit(&v->bar[3]);
        gemm_wgrad(twg + kR2, dTG, dTA_AUX, id_wg72, !first_tile);              // [dW2 | db2 ..] += g2^T [a1 | 1, q, ea, gs]
      }                                                                         // (completion: bar[4] below)
      __syncwarp();
    }
    umma::mbar_wait(&v->bar[3], phase);
    VTR();
    umma::fence_after();
    // ---- epilogue 4: gz1 = (g2 W2) * silu'(z1) (times s1) -> TM ; gq = gz1 . wq
    {
      float acc[CPT];
      uint32_t pd[NP];
      tmem_ldu_nw<NP>(tlane + kD1T + cg * NP, pd);
      tmem_ld<CPT>(tlane + kACC + c0, acc);
      float gq = 0.f;
#pragma unroll
      for (int j = 0; j < NP; j += 4) {
        const uint4 wq = *reinterpret_cast<const uint4*>(sv->wqs + (c0 >> 1) + j);
        const uint32_t wqa[4] = {wq.x, wq.y, wq.z, wq.w};
        __half2 cs = __float2half2_rn(0.f);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const __half2 g = __hmul2(__floats2half2_rn(acc[2 * (j + k)] * k21, acc[2 * (j + k) + 1] * k21), u2h(pd[j + k]));
          cs = __hfma2(g, u2h(wqa[k]), cs);
          pd[j + k] = h2u(g);
        }
        const float2 f = __half22float2(cs);
        gq += f.x + f.y;
      }
      store_row<NP>(TM, row, cg, pd);
      v->sgqp[cg * kTM + row] = gq;
      if constexpr (kEa) {
        float* sge = reinterpret_cast<float*>(T3);
        for (int f = 0; f < a.Fe; ++f) {
          float ge = 0.f;
#pragma unroll
          for (int j = 0; j < NP; j += 4) {
            const uint4 w = *reinterpret_cast<const uint4*>(sv->hWah + f * (kH / 2) + (c0 >> 1) + j);
            const uint32_t wa4[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float2 g2 = __half22float2(u2h(pd[j + k])), w2 = __half22float2(u2h(wa4[k]));
              ge = fmaf(g2.x, w2.x, fmaf(g2.y, w2.y, ge));
            }
          }
          sge[(f * CG + cg) * kTM + row] = ge;
        }
      }
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    group_sync();
    VTR();
    if (wg == 0) {
      umma::fence_after();
      if (elect_one()) {
        gemm_wgrad(twg + kDXZ, dTMa, dAUX, id_aux, !first_tile);                // (dwq, dWa) += gz1^T (q, ea)  (columns 1..5)
        umma::commit(&v->bar[4]);        // waited at the top of the next tile / before the final flush
      }
      __syncwarp();
    }
    first_tile = false;
    // ---- gQ (by col) and gP (by row) from the fp16 gz1 tile: a half-warp owns RPW / 2 consecutive rows, 4 columns per
    //      lane; one vector red per row for gQ, one per row run for gP
    if (!(a.exp & 3u)) {
      constexpr int RH = RPW / 2;
      int rk[RH + 1], ck[RH];
      uint2 uu[RH];
#pragma unroll
      for (int i = 0; i < RH; ++i) {             // every load of the pass first: no row waits for its predecessor
        const int rr = wg * RPW + hsel * RH + i;
        rk[i] = geo->srow[rr];
        ck[i] = geo->scol[rr];
        uu[i] = *reinterpret_cast<const uint2*>(TM + h_chunk_off(rr, l16 >> 1) + ((l16 & 1) << 3));
      }
      rk[RH] = -2;                               // closes the last run
      float4 run = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int i = 0; i < RH; ++i) {
        const float2 f0 = unpack2(uu[i].x), f1 = unpack2(uu[i].y);
        const float4 g = make_float4(f0.x * r1, f0.y * r1, f1.x * r1, f1.y * r1);
        if (rk[i] >= 0) atomicAdd(reinterpret_cast<float4*>(a.gQ + (size_t)ck[i] * kH + 4 * l16), g);
        run.x += g.x; run.y += g.y; run.z += g.z; run.w += g.w;      // rows past E carry exact zeros
        if (rk[i] != rk[i + 1]) {
          if (rk[i] >= 0) atomicAdd(reinterpret_cast<float4*>(a.gP + (size_t)rk[i] * kH + 4 * l16), run);
          run = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    }
    VTR();
    if (tg < kTM && !(a.exp & 2u)) {
      const int r = geo->srow[tg], c = geo->scol[tg];
      float gqs = 0.f;
#pragma unroll
      for (int g = 0; g < CG; ++g) gqs += v->sgqp[g * kTM + tg];
      const float s = v->ss[tg], gq2 = 2.f * gqs * rq;
      const float inv = norm ? 1.f / geo->snrm[tg] : 1.f;
      float gd[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        gd[k] = (r == c || r < 0) ? 0.f : s * geo->sgte[tg * 3 + k] * inv + gq2 * geo->sd[tg * 3 + k];
        if (r >= 0 && r != c) atomicAdd(a.gx + (size_t)c * 3 + k, -gd[k]);
      }
      // segmented inclusive sums over lanes with equal, contiguous row keys (one key shuffle per step for the 3 components)
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int ku = __shfl_up_sync(0xffffffffu, r, o);
        const float u0 = __shfl_up_sync(0xffffffffu, gd[0], o), u1 = __shfl_up_sync(0xffffffffu, gd[1], o),
                    u2 = __shfl_up_sync(0xffffffffu, gd[2], o);
        if (lane >= o && ku == r) { gd[0] += u0; gd[1] += u1; gd[2] += u2; }
      }
      const int kd = __shfl_down_sync(0xffffffffu, r, 1);
      if ((lane == 31 || kd != r) && r >= 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) atomicAdd(a.gx + (size_t)r * 3 + k, gd[k]);
      }
    }
    if constexpr (kEa) {
      if (tg < kTM && geo->srow[tg] >= 0) {
        const int e = v->qt[k & 3] * kTM + tg;
        float* dst = a.g_ea + (size_t)(a.perm != nullptr ? a.perm[e] : e) * a.Fe;
        for (int f = 0; f < a.Fe; ++f) {
          float ge = 0.f;
#pragma unroll
          for (int g = 0; g < CG; ++g) ge += reinterpret_cast<const float*>(T3)[(f * CG + g) * kTM + tg];
          dst[f] += ge * (2.f * r1);               // gz1 is stored times s1, hWah holds Wa / 2
        }
      }
    }
    VTR();
  }
  // ---- flush: each group waits for its last aux GEMM; then the whole CTA meets and group 0's warps read BOTH groups'
  //      weight-gradient tiles (M = 64 layout: row n of group g in lane (n / 16) * 32 + n % 16 + 16 g)
  if (!first_tile) umma::mbar_wait(&v->bar[4], (k & 1) ^ 1);
    VTR();
  if (tg == 0) v->had = first_tile ? 0 : 1;
  umma::fence_after();
  umma::fence_before();
  __syncthreads();
    VTR();
  umma::fence_after();
  // a group that saw no tile left its accumulator lanes undefined: only groups with a tile contribute
  const bool has0 = reinterpret_cast<const GV*>(smem + SM::off_groups + SM::g_vec)->had != 0;
  const bool has1 = reinterpret_cast<const GV*>(smem + SM::off_groups + SM::g_bytes + SM::g_vec)->had != 0;
  if (G == 0) {
    const int n = quarter * 16 + (lane & 15);
    const bool mine = (lane < 16) ? has0 : has1;
    const uint32_t tl = tmem + ((uint32_t)(quarter * 32) << 16);
    float w[CPT];
    auto flush_rows = [&](float* base, const float (&w)[CPT], float r) {
      if (!mine || base == nullptr) return;
      float* dst = base + (size_t)n * kH + c0;
      if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
        for (int j = 0; j < CPT; j += 4)      // red.global.add.v4.f32
          atomicAdd(reinterpret_cast<float4*>(dst + j), make_float4(w[j] * r, w[j + 1] * r, w[j + 2] * r, w[j + 3] * r));
      } else {
#pragma unroll
        for (int j = 0; j < CPT; ++j) atomicAdd(dst + j, w[j] * r);
      }
    };
    tmem_ld<CPT>(tl + kR3 + c0, w);
    flush_rows(a.g_W3, w, r3);
    tmem_ld<CPT>(tl + kR2 + c0, w);
    flush_rows(a.g_W2, w, r2);
    if (cg == 0) {
      float x3[16], x2[16], xz[16];
      tmem_ld<16>(tl + kR3 + 64, x3);          // only columns 64..71 were written; the rest of the x16 read is ignored
      tmem_ld<16>(tl + kR2 + 64, x2);
      tmem_ld<16>(tl + kDXZ, xz);              // [dxz 8 | dw4 8]
      if (mine) {
        if (a.g_b3 != nullptr) atomicAdd(a.g_b3 + n, x3[0] * r3);
        if (a.g_b2 != nullptr) atomicAdd(a.g_b2 + n, x2[0] * r2);
        if (a.g_w4 != nullptr) atomicAdd(a.g_w4 + n, xz[8 + 6] * ra);
        if (a.g_w1 != nullptr) {
          atomicAdd(a.g_w1 + (size_t)n * a.ld1 + 2 * kH, xz[1] * r1);
#pragma unroll
          for (int f = 0; f < kTcMaxFe; ++f)
            if (f < a.Fe) atomicAdd(a.g_w1 + (size_t)n * a.ld1 + 2 * kH + 1 + f, xz[2 + f] * r1);
        }
      }
    }
  }
  umma::fence_before();
  __syncthreads();
    VTR();
  if (t < 32) umma::tmem_dealloc<512>(tmem);
  VTR();
  VTR_PRINT("edge_bwd");
}

}  // namespace bwd4

// stats: 4 unsigned of caller scratch (device); claim: NULL (static tile split) or a zeroed word (tiles claimed dynamically);
// sms: the grid's cap
template <int CG, bool kEa = false, bool kLive = false>
inline cudaError_t launch_edge_bwd_tc4(const EdgeArgs& a, unsigned* stats, int sms, cudaStream_t st, bool zero_stats = true,
                                       bool run_stats = true, unsigned* claim = nullptr) {
  static DevOnce attr;
  const size_t bytes = bwd4::Smem4<CG>::bytes;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(bwd4::edge_bwd_tc4_kernel<CG, kEa, kLive>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  const int ntiles = (a.E + kTM - 1) / kTM;
  if (ntiles == 0) return cudaSuccess;
  const int pairs = (ntiles + 1) / 2;
  const int grid = pairs < sms ? pairs : sms;
  // the bound pre-pass takes maxima: stale (larger) entries only make the scales more conservative, so a caller that zeroed
  // the scratch words once per step (FEGNN_F_PREZEROED) may run the backward again on the same block
  cudaError_t e = zero_stats ? cudaMemsetAsync(stats, 0, 4 * sizeof(unsigned), st) : cudaSuccess;
  if (e != cudaSuccess) return e;
  // at most one block per SM: the final atomicMax is one same-address atomic per block and statistic (they serialise in L2)
  int sblocks = (int)(((size_t)a.N * kH + 256 * 4 - 1) / (256 * 4));
  sblocks = sblocks < 1 ? 1 : (sblocks > sms ? sms : sblocks);
  if (run_stats) {
    e = launch_pdl(bwd3::edge_bwd_stats_kernel, sblocks, 256, 0, st, a.N, a.Nl, a.x, a.gt, a.gm, stats);
    if (e != cudaSuccess) return e;
  }
  e = launch_pdl(bwd4::edge_bwd_tc4_kernel<CG, kEa, kLive>, grid, 256 * CG, bytes, st, a, (const unsigned*)stats, claim);
  if (e != cudaSuccess) return e;
  return cudaGetLastError();
}

}  // namespace fegnn
