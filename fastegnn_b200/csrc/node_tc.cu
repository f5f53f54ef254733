// node_tc.cu -- per-node dense phases on the tcgen05 tensor cores (single-pass TF32 tiles).
//
// node_pre forward (models/FastEGNN.py:104,115,139,142,162, the h-dependent half of every first Linear):
//   one 128-node tile of h (K-major SWIZZLE_128B in shared memory, coalesced loads) times up to three stacked
//   64x64 weight blocks = ONE GEMM with N = 64 * nb, accumulators in tensor memory.  Work item = (tile, group):
//   group 0 = {P, Q, Av}, group 1 = {Uh (unless last layer), phi_v head, phi_g head (gravity)}; 2 CTAs / SM.
// The fp32 FMA kernels (node_kernels.cu) remain mode 0.
#include "common.cuh"
#include "umma.cuh"

namespace fegnn {
namespace ntc {

using bwd2::desc_advance;
using bwd2::tmem_ld;

__device__ __forceinline__ float silu_tc(float z) {
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(0.5f * z));
  return z * fmaf(0.5f, th, 0.5f);
}

// stage a [64][64] block (element (n,k) = g[n*ld + off + k]) K-major SWIZZLE_128B into rows [row0, row0+64) of an R-row tile
template <int NT>
__device__ __forceinline__ void stage_block_kmajor(uint8_t* dst, const float* __restrict__ g, int ld, int off, int row0, int R) {
  if (((ld | off) & 3) == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0) {
    for (int i = threadIdx.x; i < kH * 16; i += NT) {
      const int n = i >> 4, c = i & 15;
      *reinterpret_cast<float4*>(dst + umma::tile_chunk_off(row0 + n, c, R)) =
          *reinterpret_cast<const float4*>(g + (size_t)n * ld + off + c * 4);
    }
  } else {
    float w[kH * kH / NT];
#pragma unroll
    for (int j = 0; j < kH * kH / NT; ++j) {
      const int i = threadIdx.x + j * NT;
      w[j] = g[(size_t)(i >> 6) * ld + off + (i & 63)];
    }
#pragma unroll
    for (int j = 0; j < kH * kH / NT; ++j) {
      const int i = threadIdx.x + j * NT;
      *reinterpret_cast<float*>(dst + umma::tile_off(row0 + (i >> 6), i & 63, R)) = w[j];
    }
  }
}

struct PreVec {
  float bias[3 * kH];      // first-layer bias of each block (0 where the reference has none)
  float w2[3 * kH];        // output weights of head blocks
  float sp[2 * kTM];       // cross-column-group partial sums of a head
  uint64_t bar;
  uint32_t tmem_slot;
};
struct PreSmem {
  static constexpr int off_W = 0;                    // up to [192][64] K-major
  static constexpr int off_A = 3 * 16384;            // h tile [128][64] K-major
  static constexpr int off_vec = off_A + 32768;
  static constexpr size_t bytes = off_vec + sizeof(PreVec) + 1024;
  static constexpr int off_attr = (off_vec + sizeof(PreVec) + 15) / 16 * 16;
  static constexpr size_t attr_bytes = bytes + 16 + kAttrWBytes;
};

template <bool kAttr>
__global__ void __launch_bounds__(256, 2) node_pre_fwd_tc_kernel(NodePreArgs a, NodeAttrArgs at) {
  constexpr int NT = 256, CPT = 32;
  using SM = PreSmem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
  PreVec* v = reinterpret_cast<PreVec*>(smem + SM::off_vec);
  [[maybe_unused]] float* sWa = reinterpret_cast<float*>(smem + SM::off_attr);     // attribute instantiation: U1att [f][n]
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int quarter = warp & 3, cg = warp >> 2, row = quarter * 32 + lane, c0 = cg * CPT;
  const bool grav = a.flags & FEGNN_F_GRAVITY, last = a.flags & FEGNN_F_LAST;
  const int group = blockIdx.x & 1, cta = blockIdx.x >> 1, nctas = gridDim.x >> 1;
  // block ids: 0 P, 1 Q, 2 Av, 3 Uh, 4 phi_v head, 5 phi_g head
  int blk[3], nb;
  if (group == 0) { blk[0] = 0; blk[1] = 1; blk[2] = 2; nb = 3; }
  else {
    nb = 0;
    if (!last) blk[nb++] = 3;
    blk[nb++] = 4;
    if (grav) blk[nb++] = 5;
    for (int j = nb; j < 3; ++j) blk[j] = -1;
  }
  const int R = nb * kH;
  for (int j = 0; j < nb; ++j) {
    const int b = blk[j];
    const float* wsrc = b <= 1 ? a.edge_w0 : b == 2 ? a.edgev_w0 : b == 3 ? a.node_w0 : b == 4 ? a.vel_w0 : a.grav_w0;
    const int ld = b <= 1 ? a.ld1 : b == 2 ? a.ldv : b == 3 ? a.ldn : kH;
    stage_block_kmajor<NT>(smem + SM::off_W, wsrc, ld, b == 1 ? kH : 0, j * kH, R);
    const float* bias = b == 0 ? a.edge_b0 : b == 2 ? a.edgev_b0 : b == 3 ? a.node_b0 : b == 4 ? a.vel_b0 : b == 5 ? a.grav_b0 : nullptr;
    const float* w2 = b == 4 ? a.vel_w2 : b == 5 ? a.grav_w2 : nullptr;
    for (int i = t; i < kH; i += NT) {
      v->bias[j * kH + i] = bias != nullptr ? bias[i] : 0.f;
      v->w2[j * kH + i] = w2 != nullptr ? w2[i] : 0.f;
    }
    if constexpr (kAttr) {
      if (b == 3) attr_stage_w(sWa, at, NT);
    }
  }
  if (t == 0) {
    umma::mbar_init(&v->bar, 1);
    umma::mbar_fence_init();
  }
  if (warp == 0) umma::tmem_alloc<256>(&v->tmem_slot);
  umma::fence_smem_to_async();
  umma::fence_before();
  __syncthreads();
  umma::fence_after();
  const uint32_t tmem = v->tmem_slot;
  const uint32_t tlane = tmem + ((uint32_t)(quarter * 32) << 16) + c0;
  const uint32_t idesc = umma::make_idesc_tf32(128, R);
  const uint64_t dW = umma::make_desc(umma::smem_u32(smem + SM::off_W));
  const uint64_t dA = umma::make_desc(umma::smem_u32(smem + SM::off_A));
  uint8_t* A = smem + SM::off_A;
  uint32_t phase = 0;

  const int ntiles = (a.N + kTM - 1) / kTM;
  for (int tile = cta; tile < ntiles; tile += nctas) {
    const int i0 = tile * kTM, nvalid = min(kTM, a.N - i0);
    umma::fence_before();
    __syncthreads();
    // ---- h tile -> shared memory (half-warp per row, one 16-byte chunk per lane)
    {
      const int l16 = lane & 15, hsel = lane >> 4;
#pragma unroll 4
      for (int i = 0; i < kTM / 8 / 2; ++i) {
        const int rr = warp * (kTM / 8) + 2 * i + hsel;
        float4 hv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rr < nvalid) hv = *reinterpret_cast<const float4*>(a.h + (size_t)(i0 + rr) * kH + 4 * l16);
        *reinterpret_cast<float4*>(A + umma::tile_chunk_off(rr, l16, kTM)) = hv;
      }
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    __syncthreads();
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)
          umma::mma_tf32(tmem, desc_advance(dA, (ks >> 2) * (kTM * 128) + (ks & 3) * 32),
                         desc_advance(dW, (ks >> 2) * (R * 128) + (ks & 3) * 32), idesc, ks > 0);
        umma::commit(&v->bar);
      }
      __syncwarp();
    }
    umma::mbar_wait(&v->bar, phase);
    umma::fence_after();
    phase ^= 1;
    // ---- epilogue: bias + store (P, Q, Av, Uh) or head output w2 . silu(z + b0) + b2 (sv, sg)
    for (int j = 0; j < nb; ++j) {
      const int b = blk[j];
      float z[CPT];
      tmem_ld<CPT>(tlane + j * kH, z);
      if (b < 4) {
        float* out = b == 0 ? a.P : b == 1 ? a.Q : b == 2 ? a.Av : a.Uh;
        if constexpr (kAttr) {
          if (b == 3 && row < nvalid) {                  // + U1att a_i in fp32
            const float* ar = at.a + (size_t)(i0 + row) * at.Fa;
            for (int f = 0; f < at.Fa; ++f) {
              const float af = ar[f];
#pragma unroll
              for (int jj = 0; jj < CPT; ++jj) z[jj] = fmaf(af, sWa[f * kH + c0 + jj], z[jj]);
            }
          }
        }
        if (row < nvalid) {
          float4* dst = reinterpret_cast<float4*>(out + (size_t)(i0 + row) * kH + c0);
#pragma unroll
          for (int ch = 0; ch < CPT / 4; ++ch)
            dst[ch] = make_float4(z[ch * 4] + v->bias[j * kH + c0 + ch * 4], z[ch * 4 + 1] + v->bias[j * kH + c0 + ch * 4 + 1],
                                  z[ch * 4 + 2] + v->bias[j * kH + c0 + ch * 4 + 2], z[ch * 4 + 3] + v->bias[j * kH + c0 + ch * 4 + 3]);
        }
      } else {
        float s = 0.f;
#pragma unroll
        for (int jj = 0; jj < CPT; ++jj) s = fmaf(silu_tc(z[jj] + v->bias[j * kH + c0 + jj]), v->w2[j * kH + c0 + jj], s);
        v->sp[cg * kTM + row] = s;
        __syncthreads();
        if (cg == 0 && row < nvalid) {
          const float b2 = b == 4 ? a.vel_b2[0] : a.grav_b2[0];
          (b == 4 ? a.sv : a.sg)[i0 + row] = s + v->sp[kTM + row] + b2;
        }
        __syncthreads();
      }
    }
  }
  umma::fence_before();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc<256>(tmem);
}


// ------------------------------------------------------------------------------------------------- node_h forward
// phi_h (models/FastEGNN.py:153-166) on the tensor cores with fp32-grade results (error-compensated 3xTF32, the same split as
// edge_forward mode 3), so that it may be the DEFAULT of the forward pass -- single-pass TF32 on h breaks the script's
// equivariance tolerance (DESIGN.md 3.2):
//     zh1 = Uh + (msum / deg) W0a^T + sum_c u[:, c, :] W0u_c^T          h' = h + silu(zh1) W2^T + b2
// The fp32 FMA form (node_kernels.cu) accumulated zh1 with one red.global.add pass per K-block (1 + C passes over [N, 64])
// and ran at 14 TFLOP/s at 1 M nodes; a step spent 13 % of its time there.  Here a CTA owns a 128-node tile and WALKS the
// K-blocks through a two-stage ring: the rows of block b + 1 (and its 64x64 weight block) are in flight in registers while
// the three tcgen05.mma passes of block b run (a_hi w_hi + a_lo w_hi + a_hi w_lo; fp32 accumulator in tensor memory for the
// whole sum -- no atomics, zh1 is written once).  silu(zh1) is split on chip into the next ring slot, so the output Linear is
// just one more block.  Rows travel global -> registers -> swizzled K-major tiles in (row, 16-byte chunk) order (a warp-wide
// access covers 2 rows x 256 contiguous bytes) and the accumulators leave through a staging tile the same way: Uh and h are
// added in that phase in exact fp32.  Algorithmic bytes per node: 256 (3 + C) read + 512 written; HBM-bound from ~10^5 nodes.
struct HVec {
  float b2[kH];
  uint64_t bar[2];                 // MMAs that read operand slot 0 / 1
  uint32_t tmem_slot;
};
struct HSmem {
  static constexpr int kT = kTM * kH * 4, kW = kH * kH * 4;
  static constexpr int off_A = 0;                  // [2 slots][hi | lo] operand tiles
  static constexpr int off_W = 4 * kT;             // [3 slots][hi | lo] weight tiles (cp.async ring)
  static constexpr int off_vec = off_W + 6 * kW;
  static constexpr size_t bytes = off_vec + sizeof(HVec) + 1024;
  static_assert(bytes <= 232448, "node_h forward: shared memory");
};
constexpr uint32_t kNH_ACC1 = 0, kNH_ACC2 = 64;    // 128 tensor-memory columns
constexpr int kWimgFloats = 2 * kH * kH;           // one weight block: hi | lo operand-tile images

// Weight pre-pass: block b of layer l -> its operand-tile image (what the main kernel's ring slot holds, byte for byte), so the
// main loop moves weights with cp.async only.  In the reference layout the u blocks are interleaved (flatten order k * C + c,
// models/FastEGNN.py:157): read in place, one 64x64 block drags the whole [64, 64 C] slab through L1 -- measured at C = 8:
// 128 KB of L2 traffic per block against 32 KB of node rows, 7 000 cycles per block.
struct WPrepArgs {
  int C, ldn;
  const float* w0[32];
  const float* w2[32];
  float* wimg[32];
};
__global__ void __launch_bounds__(256) node_h_wprep_kernel(const __grid_constant__ WPrepArgs a) {
  constexpr int NT = 256, NWR = kH * kH / NT;
  pdl_trigger();
  const int b = blockIdx.x, l = blockIdx.y, t = threadIdx.x, nb1 = a.C + 1;
  const float* base = b < nb1 ? a.w0[l] : a.w2[l];
  const int ld = b < nb1 ? a.ldn : kH, off = b == 0 ? kH : b < nb1 ? 2 * kH + (b - 1) : 0, wks = (b == 0 || b >= nb1) ? 1 : a.C;
  float w[NWR];
#pragma unroll
  for (int j = 0; j < NWR / 4; ++j) {
    const int i = t + j * NT, n = i >> 4, c = i & 15;
#pragma unroll
    for (int q = 0; q < 4; ++q) w[4 * j + q] = base[(size_t)n * ld + off + (size_t)(4 * c + q) * wks];
  }
  pdl_wait();      // the images are written only after the predecessor has completed (a shared block may still be read)
  float* img = a.wimg[l] + (size_t)b * kWimgFloats;
#pragma unroll
  for (int j = 0; j < NWR / 4; ++j) {
    const int i = t + j * NT, n = i >> 4, c = i & 15;
    const float4 x = make_float4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
    const float4 hi = make_float4(umma::to_tf32(x.x), umma::to_tf32(x.y), umma::to_tf32(x.z), umma::to_tf32(x.w));
    const uint32_t o = umma::tile_chunk_off(n, c, kH) >> 2;
    *reinterpret_cast<float4*>(img + o) = hi;
    *reinterpret_cast<float4*>(img + kH * kH + o) = make_float4(x.x - hi.x, x.y - hi.y, x.z - hi.z, x.w - hi.w);
  }
}

// kSaved: the saved-only form of a backward's recompute (FEGNN_F_RECOMPUTE): zh1 only -- h' is already in the next layer's
// state, so the output Linear, its residual add and the h' write-out do not run
template <bool kSaved = false>
__global__ void __launch_bounds__(256, 1) node_h_fwd_tc_kernel(NodeHArgs a) {
  VTR_DECL();
  constexpr int NT = 256, CPT = 32, NA = kTM * 16 / NT;
  using SM = HSmem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
  pdl_trigger();
  HVec* v = reinterpret_cast<HVec*>(smem + SM::off_vec);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int quarter = warp & 3, cg = warp >> 2, row = quarter * 32 + lane, c0 = cg * CPT;
  const int rr0 = t >> 4, c16 = t & 15;            // cooperative phases: rows rr0 + 16 j, chunk c16
  const int nb1 = a.C + 1;                         // K-blocks of zh1: 0 = message mean, 1 + c = u[:, c, :]
  auto At = [&](int s_) { return smem + SM::off_A + s_ * 2 * SM::kT; };
  auto Wt = [&](int w_) { return smem + SM::off_W + w_ * 2 * SM::kW; };

  // TWO register sets of operand rows: the blocks of a tile alternate between them (block b of every tile in set b & 1), so
  // the rows of blocks b + 1 and b + 2 are both in flight while block b is split and multiplied -- one 32 KB block in
  // flight per SM was what bounded the kernel at 1 M nodes (2.2 TB/s of row traffic)
  float4 areg0[NA], areg1[NA];
  float sc0[NA], sc1[NA];
  // weight block b -> ring slot w_ (32 KB image, 8 x 16 bytes per thread), one cp.async group; b < 0: an empty group
  auto fetch_w = [&](int b, int w_) {
    if (b >= 0) {
      const uint8_t* src = reinterpret_cast<const uint8_t*>(a.wimg + (size_t)b * kWimgFloats);
#pragma unroll
      for (int j = 0; j < 2 * SM::kW / 16 / NT; ++j) {
        const int i = t + j * NT;
        cp_async16(Wt(w_) + 16 * i, src + 16 * i, 16);
      }
    }
    cp_async_commit();
  };
  auto load_rows = [&](float4 (&dst)[NA], const float* src, size_t ld, int i0) {
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      const int r = i0 + rr0 + 16 * j;
      dst[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < a.N) dst[j] = *reinterpret_cast<const float4*>(src + (size_t)r * ld + 4 * c16);
    }
  };
  auto load_a = [&](int b, int i0, float4 (&areg)[NA], float (&sc)[NA]) {
    if (b == 0) {
      load_rows(areg, a.msum, kH, i0);
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        const int r = i0 + rr0 + 16 * j;
        sc[j] = (a.dinv != nullptr && r < a.N) ? a.dinv[r] : 1.f;      // nullptr: plain sums (FEGNN_F_NODE_SUM)
      }
    } else {
      load_rows(areg, a.u + (size_t)(b - 1) * kH, (size_t)a.C * kH, i0);
#pragma unroll
      for (int j = 0; j < NA; ++j) sc[j] = 1.f;
    }
  };
  auto store_split = [&](uint8_t* tile, int j, float4 x) {
    const float4 hi = make_float4(umma::to_tf32(x.x), umma::to_tf32(x.y), umma::to_tf32(x.z), umma::to_tf32(x.w));
    const uint32_t o = umma::tile_chunk_off(rr0 + 16 * j, c16, kTM);
    *reinterpret_cast<float4*>(tile + o) = hi;
    *reinterpret_cast<float4*>(tile + SM::kT + o) = make_float4(x.x - hi.x, x.y - hi.y, x.z - hi.z, x.w - hi.w);
  };
  auto store_a = [&](int s_, const float4 (&areg)[NA], const float (&sc)[NA]) {
#pragma unroll
    for (int j = 0; j < NA; ++j)
      store_split(At(s_), j, make_float4(areg[j].x * sc[j], areg[j].y * sc[j], areg[j].z * sc[j], areg[j].w * sc[j]));
  };

  // ---- prologue (weights only): vectors, barriers, tensor memory
  for (int i = t; i < kH; i += NT) v->b2[i] = a.node_b2[i];
  if (t == 0) {
    umma::mbar_init(&v->bar[0], 1);
    umma::mbar_init(&v->bar[1], 1);
    umma::mbar_fence_init();
  }
  if (warp == 0) umma::tmem_alloc<128>(&v->tmem_slot);
  umma::fence_before();
  __syncthreads();
  umma::fence_after();
  VTR();
  pdl_wait();                                      // the weight images come from the pre-pass, the rows from the layer's phases
  VTR();
  const uint32_t tmem = v->tmem_slot;
  const uint32_t tlane = tmem + ((uint32_t)(quarter * 32) << 16) + c0;
  const uint32_t idesc = umma::make_idesc_tf32(128, kH);
  // descriptors of slot 0; operand slot 1 lies 2 kT, weight slot w 2 w kW bytes further (only the 14-bit address field moves)
  const uint64_t dA0 = umma::make_desc(umma::smem_u32(At(0))), dW0 = umma::make_desc(umma::smem_u32(Wt(0)));
  // D (+)= A W^T in three passes: operand slot s_, weight slot w_
  auto issue = [&](uint32_t acc, int s_, int w_, bool accumulate) {
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
        const uint64_t dA = dA0 + (uint64_t)(s_ * ((2 * SM::kT) >> 4)), dW = dW0 + (uint64_t)(w_ * ((2 * SM::kW) >> 4));
        umma::gemm_k64_desc(acc, dA, kTM, dW, kH, idesc, accumulate);
        umma::gemm_k64_desc(acc, dA + (uint64_t)(SM::kT >> 4), kTM, dW, kH, idesc, true);
        umma::gemm_k64_desc(acc, dA, kTM, dW + (uint64_t)(SM::kW >> 4), kH, idesc, true);
        umma::commit(&v->bar[s_]);
      }
      __syncwarp();
    }
  };
  uint32_t ph_bits = 0, pend_bits = 0;             // per operand slot: mbarrier phase, commit outstanding
  auto wait_slot = [&](int s_) {                   // the MMAs that read operand slot s_ have completed
    if ((pend_bits >> s_) & 1u) {
      umma::mbar_wait(&v->bar[s_], (ph_bits >> s_) & 1u);
      umma::fence_after();
      ph_bits ^= 1u << s_;
      pend_bits &= ~(1u << s_);
    }
  };

  const int ntiles = (a.N + kTM - 1) / kTM;
  int g = 0, wq = 0;                               // running block count: operand slot g & 1, weight slot wq = g % 3
  if ((int)blockIdx.x < ntiles) {
    fetch_w(0, 0);
    load_a(0, blockIdx.x * kTM, areg0, sc0);
    load_a(1, blockIdx.x * kTM, areg1, sc1);       // nb1 = C + 1 >= 2
  }
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int i0 = tile * kTM;
    const bool more = tile + (int)gridDim.x < ntiles;
    float4 uh[NA], hr[NA];
    // block b of the tile out of register set `par` = b & 1 (a compile-time constant at both call sites below)
    auto block_iter = [&](int b, int par, float4 (&areg)[NA], float (&sc)[NA]) {
      const int s_ = g & 1, wn = wq == 2 ? 0 : wq + 1;
      wait_slot(s_);                               // block g - 2 is done: operand slot s_ and weight slot (g + 1) % 3 are free
      VTR();
      fetch_w(b + 1, wn);                          // next block's weights (b + 1 == nb1: the output Linear) travel a full block ahead
      store_a(s_, areg, sc);
      cp_async_wait_group<1>();                    // this block's weights have landed
      umma::fence_smem_to_async();
      umma::fence_before();
      __syncthreads();
      VTR();
      // the freed register set takes the block two ahead: of this tile, else the block of the NEXT tile with this parity
      if (b + 2 < nb1) load_a(b + 2, i0, areg, sc);
      else if (more) load_a(par, (tile + gridDim.x) * kTM, areg, sc);
      if (b == nb1 - 1) {                          // the rows the write-out phases add: Uh (zh1) and h (h')
        load_rows(uh, a.Uh, kH, i0);
        if constexpr (!kSaved) load_rows(hr, a.h, kH, i0);
      }
      issue(tmem + kNH_ACC1, s_, wq, b > 0);
      pend_bits |= 1u << s_;
      wq = wn;
      ++g;
    };
    for (int b = 0; b < nb1; b += 2) {
      block_iter(b, 0, areg0, sc0);
      if (b + 1 < nb1) block_iter(b + 1, 1, areg1, sc1);
    }
    // ---- output Linear = one more block whose operand is made on chip
    const int s2 = g & 1, so = s2 ^ 1, wn = wq == 2 ? 0 : wq + 1;
    wait_slot(s2);
    fetch_w(more ? 0 : -1, wn);                    // first block of the next tile
    VTR();
    wait_slot(so);                                 // zh1 - Uh is complete in tensor memory; both operand slots are free
    VTR();
    uint8_t* ST = At(so);                          // staging tile (row owners -> (row, chunk) order)
    {
      float z[CPT];
      tmem_ld<CPT>(tlane + kNH_ACC1, z);
#pragma unroll
      for (int ch = 0; ch < CPT / 4; ++ch)
        *reinterpret_cast<float4*>(ST + umma::tile_chunk_off(row, cg * (CPT / 4) + ch, kTM)) =
            make_float4(z[4 * ch], z[4 * ch + 1], z[4 * ch + 2], z[4 * ch + 3]);
    }
    umma::fence_before();
    __syncthreads();
    VTR();
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      const int rr = rr0 + 16 * j;
      float4 z = *reinterpret_cast<const float4*>(ST + umma::tile_chunk_off(rr, c16, kTM));
      z.x += uh[j].x; z.y += uh[j].y; z.z += uh[j].z; z.w += uh[j].w;
      if (i0 + rr < a.N) *reinterpret_cast<float4*>(a.zh1 + (size_t)(i0 + rr) * kH + 4 * c16) = z;
      if constexpr (!kSaved) store_split(At(s2), j, make_float4(silu_f(z.x), silu_f(z.y), silu_f(z.z), silu_f(z.w)));
    }
    cp_async_wait_group<1>();                      // the output Linear's weights have landed
    if constexpr (kSaved) {                        // same slot and weight-ring sequence, no output Linear
      ++g;
      wq = wn;
      __syncthreads();                             // ST has been read
      continue;
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    __syncthreads();
    VTR();
    issue(tmem + kNH_ACC2, s2, wq, false);
    pend_bits |= 1u << s2;
    wait_slot(s2);
    VTR();
    {
      float o[CPT];
      tmem_ld<CPT>(tlane + kNH_ACC2, o);
#pragma unroll
      for (int ch = 0; ch < CPT / 4; ++ch) {
        const float4 bb = *reinterpret_cast<const float4*>(v->b2 + c0 + 4 * ch);
        *reinterpret_cast<float4*>(ST + umma::tile_chunk_off(row, cg * (CPT / 4) + ch, kTM)) =
            make_float4(o[4 * ch] + bb.x, o[4 * ch + 1] + bb.y, o[4 * ch + 2] + bb.z, o[4 * ch + 3] + bb.w);
      }
    }
    umma::fence_before();
    __syncthreads();
    VTR();
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      const int rr = rr0 + 16 * j;
      if (i0 + rr < a.N) {
        const float4 o = *reinterpret_cast<const float4*>(ST + umma::tile_chunk_off(rr, c16, kTM));
        *reinterpret_cast<float4*>(a.h_new + (size_t)(i0 + rr) * kH + 4 * c16) =
            make_float4(hr[j].x + o.x, hr[j].y + o.y, hr[j].z + o.z, hr[j].w + o.w);
      }
    }
    ++g;
    wq = wn;
    __syncthreads();                               // ST (= the slot the next block is stored to) has been read
    VTR();
  }
  cp_async_wait();
  umma::fence_before();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc<128>(tmem);
  VTR_PRINT("node_h_fwd");
}


// ------------------------------------------------------------------------------------------------- node_pre forward, 3xTF32
// The h-side halves of every first Linear (models/FastEGNN.py:104,115,139,142,162) with fp32-grade results: one CTA per
// 128-node tile loads h ONCE (split hi | lo into the operand tile) and walks the 3-6 active weight blocks (P, Q, Av, Uh,
// phi_v head, phi_g head); block k's three tcgen05.mma passes run into accumulator k & 1 while block k - 1 leaves through a
// staging tile in (row, chunk) order and block k + 1's weights are split into the next slot of a three-slot ring.  The fp32
// FMA kernel is a (tile, block) decomposition that reads h once per block and runs at a quarter of the FFMA peak.
struct P3Vec {
  float bias[2][kH], w2[2][kH];    // of block k in buffer k & 1: first-layer bias ; head output weights
  float sp[kTM];                   // head: partial dot of the second column group
  uint64_t bar[2];                 // MMAs into accumulator 0 / 1
  uint32_t tmem_slot;
};
struct P3Smem {
  static constexpr int kT = kTM * kH * 4, kW = kH * kH * 4;
  static constexpr int off_A = 0;                  // h tile, hi | lo
  static constexpr int off_W = 2 * kT;             // [3 slots][hi | lo]
  static constexpr int off_ST = off_W + 6 * kW;    // staging tile
  static constexpr int off_vec = off_ST + kT;
  static constexpr size_t bytes = off_vec + sizeof(P3Vec) + 1024;
  static_assert(bytes <= 232448, "node_pre forward (3xTF32): shared memory");
  static constexpr int off_attr = (off_vec + sizeof(P3Vec) + 15) / 16 * 16;
  static constexpr size_t attr_bytes = bytes + 16 + kAttrWBytes;
  static_assert(attr_bytes <= 232448, "node_pre forward (3xTF32, node attributes): shared memory");
};

template <bool kAttr>
__global__ void __launch_bounds__(256, 1) node_pre_fwd_tc3_kernel(NodePreArgs a, int nactive, NodeAttrArgs at) {
  constexpr int NT = 256, CPT = 32, NA = kTM * 16 / NT, NWR = kH * kH / NT;
  using SM = P3Smem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
  pdl_trigger();
  P3Vec* v = reinterpret_cast<P3Vec*>(smem + SM::off_vec);
  [[maybe_unused]] float* sWa = reinterpret_cast<float*>(smem + SM::off_attr);     // attribute instantiation: U1att [f][n]
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int quarter = warp & 3, cg = warp >> 2, row = quarter * 32 + lane, c0 = cg * CPT;
  const int rr0 = t >> 4, c16 = t & 15;
  const bool grav = a.flags & FEGNN_F_GRAVITY, last = a.flags & FEGNN_F_LAST, rf = a.flags & FEGNN_F_RF;
  uint8_t* At = smem + SM::off_A;
  uint8_t* ST = smem + SM::off_ST;
  auto Wt = [&](int w_) { return smem + SM::off_W + w_ * 2 * SM::kW; };
  auto blk_of = [&](int k) { return node_pre_block_id(k, last, grav, rf); };     // 0 P, 1 Q, 2 Av, 3 Uh, 4 phi_v, 5 phi_g
  // block range of this CTA: with few tiles (gridDim.y = 2) two CTAs share a tile, each takes half of the blocks
  const int kb = (int)blockIdx.y * nactive / (int)gridDim.y, ke = ((int)blockIdx.y + 1) * nactive / (int)gridDim.y;

  float wreg[NWR];
  float4 hreg[NA];
  auto load_w = [&](int k) {                       // weights of the k-th active block: 4 x 16 contiguous bytes per thread
    const int b = blk_of(k);
    const float* src = b <= 1 ? a.edge_w0 : b == 2 ? a.edgev_w0 : b == 3 ? a.node_w0 : b == 4 ? a.vel_w0 : a.grav_w0;
    const int ld = b <= 1 ? a.ld1 : b == 2 ? a.ldv : b == 3 ? a.ldn : kH, off = b == 1 ? kH : 0;
    if (((ld | off) & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
#pragma unroll
      for (int j = 0; j < NWR / 4; ++j) {
        const int i = t + j * NT, n = i >> 4, c = i & 15;
        const float4 w = *reinterpret_cast<const float4*>(src + (size_t)n * ld + off + 4 * c);
        wreg[4 * j] = w.x; wreg[4 * j + 1] = w.y; wreg[4 * j + 2] = w.z; wreg[4 * j + 3] = w.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < NWR / 4; ++j) {
        const int i = t + j * NT, n = i >> 4, c = i & 15;
#pragma unroll
        for (int q = 0; q < 4; ++q) wreg[4 * j + q] = src[(size_t)n * ld + off + 4 * c + q];
      }
    }
  };
  auto store_w = [&](int w_) {
#pragma unroll
    for (int j = 0; j < NWR / 4; ++j) {
      const int i = t + j * NT, n = i >> 4, c = i & 15;
      const float4 w = make_float4(wreg[4 * j], wreg[4 * j + 1], wreg[4 * j + 2], wreg[4 * j + 3]);
      const float4 hi = make_float4(umma::to_tf32(w.x), umma::to_tf32(w.y), umma::to_tf32(w.z), umma::to_tf32(w.w));
      const uint32_t o = umma::tile_chunk_off(n, c, kH);
      *reinterpret_cast<float4*>(Wt(w_) + o) = hi;
      *reinterpret_cast<float4*>(Wt(w_) + SM::kW + o) = make_float4(w.x - hi.x, w.y - hi.y, w.z - hi.z, w.w - hi.w);
    }
  };
  auto load_h = [&](int i0) {
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      const int r = i0 + rr0 + 16 * j;
      hreg[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < a.N) hreg[j] = *reinterpret_cast<const float4*>(a.h + (size_t)r * kH + 4 * c16);
    }
  };
  auto store_h = [&]() {
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      const float4 x = hreg[j];
      const float4 hi = make_float4(umma::to_tf32(x.x), umma::to_tf32(x.y), umma::to_tf32(x.z), umma::to_tf32(x.w));
      const uint32_t o = umma::tile_chunk_off(rr0 + 16 * j, c16, kTM);
      *reinterpret_cast<float4*>(At + o) = hi;
      *reinterpret_cast<float4*>(At + SM::kT + o) = make_float4(x.x - hi.x, x.y - hi.y, x.z - hi.z, x.w - hi.w);
    }
  };

  // ---- prologue (weights only)
  load_w(kb);
  if constexpr (kAttr) {
    if (!last) attr_stage_w(sWa, at, NT);
  }
  if (t == 0) {
    umma::mbar_init(&v->bar[0], 1);
    umma::mbar_init(&v->bar[1], 1);
    umma::mbar_fence_init();
  }
  if (warp == 0) umma::tmem_alloc<128>(&v->tmem_slot);
  store_w(0);
  load_w(kb + 1 < ke ? kb + 1 : kb);
  umma::fence_before();
  __syncthreads();
  umma::fence_after();
  pdl_wait();
  const uint32_t tmem = v->tmem_slot;
  const uint32_t tlane = tmem + ((uint32_t)(quarter * 32) << 16) + c0;
  const uint32_t idesc = umma::make_idesc_tf32(128, kH);
  const uint64_t dA = umma::make_desc(umma::smem_u32(At)), dW0 = umma::make_desc(umma::smem_u32(Wt(0)));
  auto issue = [&](int acc_, int w_) {
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
        const uint32_t acc = tmem + 64 * acc_;
        const uint64_t dW = dW0 + (uint64_t)(w_ * ((2 * SM::kW) >> 4));
        umma::gemm_k64_desc(acc, dA, kTM, dW, kH, idesc, false);
        umma::gemm_k64_desc(acc, dA + (uint64_t)(SM::kT >> 4), kTM, dW, kH, idesc, true);
        umma::gemm_k64_desc(acc, dA, kTM, dW + (uint64_t)(SM::kW >> 4), kH, idesc, true);
        umma::commit(&v->bar[acc_]);
      }
      __syncwarp();
    }
  };
  uint32_t ph_bits = 0;
  // block k (accumulator k & 1) -> global memory: + bias, through the staging tile, rows in (row, chunk) order ; heads: the
  // output dot product of the row
  auto epilogue = [&](int k, int i0) {
    const int b = blk_of(k), acc_ = (k - kb) & 1;
    umma::mbar_wait(&v->bar[acc_], (ph_bits >> acc_) & 1u);
    umma::fence_after();
    ph_bits ^= 1u << acc_;
    float z[CPT];
    tmem_ld<CPT>(tlane + 64 * acc_, z);
    if (b < 4) {
#pragma unroll
      for (int ch = 0; ch < CPT / 4; ++ch) {
        const float4 bb = *reinterpret_cast<const float4*>(v->bias[acc_] + c0 + 4 * ch);
        *reinterpret_cast<float4*>(ST + umma::tile_chunk_off(row, cg * (CPT / 4) + ch, kTM)) =
            make_float4(z[4 * ch] + bb.x, z[4 * ch + 1] + bb.y, z[4 * ch + 2] + bb.z, z[4 * ch + 3] + bb.w);
      }
      umma::fence_before();
      __syncthreads();
      float* out = b == 0 ? a.P : b == 1 ? a.Q : b == 2 ? a.Av : a.Uh;
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        const int rr = rr0 + 16 * j;
        if (i0 + rr < a.N) {
          float4 o = *reinterpret_cast<const float4*>(ST + umma::tile_chunk_off(rr, c16, kTM));
          if constexpr (kAttr) {
            if (b == 3) {                          // + U1att a_i in fp32
              const float* ar = at.a + (size_t)(i0 + rr) * at.Fa;
              for (int f = 0; f < at.Fa; ++f) {
                const float af = ar[f];
                const float4 w = *reinterpret_cast<const float4*>(sWa + f * kH + 4 * c16);
                o.x = fmaf(af, w.x, o.x); o.y = fmaf(af, w.y, o.y); o.z = fmaf(af, w.z, o.z); o.w = fmaf(af, w.w, o.w);
              }
            }
          }
          *reinterpret_cast<float4*>(out + (size_t)(i0 + rr) * kH + 4 * c16) = o;
        }
      }
    } else {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < CPT; ++j) s = fmaf(silu_f(z[j] + v->bias[acc_][c0 + j]), v->w2[acc_][c0 + j], s);
      if (cg == 1) v->sp[row] = s;
      umma::fence_before();
      __syncthreads();
      if (cg == 0 && i0 + row < a.N) (b == 4 ? a.sv : a.sg)[i0 + row] = s + v->sp[row] + (b == 4 ? a.vel_b2[0] : a.grav_b2[0]);
    }
  };
  // bias / head vectors of block k -> buffer k & 1 (written at the top of iteration k, read by epilogue(k) an iteration later)
  auto stage_vecs = [&](int k) {
    const int b = blk_of(k);
    if (t < kH) {
      const float* bias = b == 0 ? a.edge_b0 : b == 2 ? a.edgev_b0 : b == 3 ? a.node_b0 : b == 4 ? a.vel_b0 : b == 5 ? a.grav_b0 : nullptr;
      const float* w2 = b == 4 ? a.vel_w2 : b == 5 ? a.grav_w2 : nullptr;
      v->bias[(k - kb) & 1][t] = bias != nullptr ? bias[t] : 0.f;
      v->w2[(k - kb) & 1][t] = w2 != nullptr ? w2[t] : 0.f;
    }
  };

  const int ntiles = (a.N + kTM - 1) / kTM;
  if ((int)blockIdx.x < ntiles) load_h(blockIdx.x * kTM);
  int wq = 0;                                      // weight ring slot of the block at hand (runs on across tiles)
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int i0 = tile * kTM;
    store_h();                                     // the previous tile's last block has completed (its epilogue waited)
    if (tile + (int)gridDim.x < ntiles) load_h((tile + gridDim.x) * kTM);      // next tile's rows travel under this tile's blocks
    for (int k = kb; k < ke; ++k) {
      // at this point: W(k) sits in slot wq (stored an iteration ago), the registers hold the weights of the block after it
      stage_vecs(k);
      umma::fence_smem_to_async();
      umma::fence_before();
      __syncthreads();                             // W(k) [and h] visible ; staging tile and accumulator of block k - 2 consumed
      issue((k - kb) & 1, wq);
      const int wn = wq == 2 ? 0 : wq + 1;
      const int k1 = k + 1 < ke ? k + 1 : kb, k2 = k1 + 1 < ke ? k1 + 1 : kb;      // past the last block: the next tile's
      store_w(wn);                                 // slot of block k - 2, which has completed (epilogue(k - 2) waited for it)
      load_w(k2);
      wq = wn;
      if (k > kb) epilogue(k - 1, i0);
    }
    __syncthreads();                               // the staging tile of the block before the last has been written out
    epilogue(ke - 1, i0);
  }
  umma::fence_before();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc<128>(tmem);
}

}  // namespace ntc

// at != nullptr: the attribute instantiation (Fa > 0 and a Uh block: not the last layer)
cudaError_t launch_node_pre_fwd_tc(const NodePreArgs& a, int sms, cudaStream_t st, const NodeAttrArgs* at = nullptr) {
  static DevOnce attr;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(ntc::node_pre_fwd_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)ntc::PreSmem::bytes);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ntc::node_pre_fwd_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)ntc::PreSmem::attr_bytes);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  const int ntiles = (a.N + kTM - 1) / kTM;
  if (ntiles == 0) return cudaSuccess;
  int per = ntiles < sms ? ntiles : sms;          // CTAs per group; 2 groups -> up to 2 CTAs / SM
  if (at != nullptr) ntc::node_pre_fwd_tc_kernel<true><<<2 * per, 256, ntc::PreSmem::attr_bytes, st>>>(a, *at);
  else ntc::node_pre_fwd_tc_kernel<false><<<2 * per, 256, ntc::PreSmem::bytes, st>>>(a, NodeAttrArgs{});
  ++g_launches;
  return cudaGetLastError();
}

cudaError_t launch_node_pre_fwd_tc3(const NodePreArgs& a, int sms, cudaStream_t st, const NodeAttrArgs* at = nullptr) {
  static DevOnce attr;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(ntc::node_pre_fwd_tc3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)ntc::P3Smem::bytes);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(ntc::node_pre_fwd_tc3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)ntc::P3Smem::attr_bytes);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  const int ntiles = (a.N + kTM - 1) / kTM;
  if (ntiles == 0) return cudaSuccess;
  const bool grav = a.flags & FEGNN_F_GRAVITY, last = a.flags & FEGNN_F_LAST;
  const int nactive = 4 + (grav ? 2 : 1) - (last ? 1 : 0) - ((a.flags & FEGNN_F_RF) ? 1 : 0);
  const int nsplit = 2 * ntiles <= sms ? 2 : 1;   // few tiles: two CTAs per tile, half of the blocks each
  const dim3 grid(ntiles < sms ? ntiles : sms, nsplit);
  if (at != nullptr) {
    if (cudaError_t e_ = launch_pdl(ntc::node_pre_fwd_tc3_kernel<true>, grid, 256, ntc::P3Smem::attr_bytes, st, a, nactive, *at))
      return e_;
    return cudaGetLastError();
  }
  if (cudaError_t e_ = launch_pdl(ntc::node_pre_fwd_tc3_kernel<false>, grid, 256, ntc::P3Smem::bytes, st, a, nactive, NodeAttrArgs{}))
    return e_;
  return cudaGetLastError();
}

cudaError_t launch_node_h_wprep(int C, int ldn, int nl, const float* const* w0, const float* const* w2, float* const* wimg,
                                cudaStream_t st) {
  if (nl <= 0) return cudaSuccess;
  ntc::WPrepArgs a;
  memset(&a, 0, sizeof(a));
  a.C = C; a.ldn = ldn;
  for (int l = 0; l < nl; ++l) { a.w0[l] = w0[l]; a.w2[l] = w2[l]; a.wimg[l] = wimg[l]; }
  if (cudaError_t e_ = launch_pdl(ntc::node_h_wprep_kernel, dim3(C + 2, nl), 256, 0, st, a)) return e_;
  return cudaGetLastError();
}

template <bool kSaved = false>
cudaError_t launch_node_h_fwd_tc(const NodeHArgs& a, int sms, cudaStream_t st) {
  static DevOnce attr;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(ntc::node_h_fwd_tc_kernel<kSaved>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)ntc::HSmem::bytes);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  const int ntiles = (a.N + kTM - 1) / kTM;
  if (ntiles == 0) return cudaSuccess;
  if (cudaError_t e_ = launch_pdl(ntc::node_h_fwd_tc_kernel<kSaved>, ntiles < sms ? ntiles : sms, 256, ntc::HSmem::bytes, st, a)) return e_;
  return cudaGetLastError();
}

}  // namespace fegnn
