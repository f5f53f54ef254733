// edge_tc.cu -- fused real-edge FORWARD phase on the 5th-generation tensor cores (tcgen05 + TMEM).
//
// Same contract as edge_fwd_kernel (edge_kernels.cu; reference models/FastEGNN.py:102-108,125-129,156):
// tiles of 128 CSR-sorted edges, nothing per-edge written to HBM.  Here one thread owns one edge
// row (= one TMEM lane): it gathers P[row], Q[col], builds a1 = silu(z1) straight into the
// K-major/SWIZZLE_128B operand tile, one elected thread issues  z2 = a1 W2^T  and  z3 = m W3^T  as
// tcgen05.mma kind::tf32 (M=128, N=64, K=64, accumulators in TMEM columns 0-63 / 64-127), and the
// epilogues (bias, SiLU, attention gate, phi_x output dot, segment sums) run out of tcgen05.ld.
//
// SPLIT = 1 : single-pass TF32 (10-bit mantissa operands, fp32 accumulate).
// SPLIT = 3 : error-compensated 3xTF32 (a_hi b_hi + a_lo b_hi + a_hi b_lo), fp32-grade results.
#include "common.cuh"
#include "umma.cuh"

namespace fegnn {

constexpr int kTcThreads = 256;
constexpr int kTcMaxFe = 4;   // wider edge attributes use the fp32 FMA kernel (keeps 3 CTAs/SM worth of shared memory)

struct EdgeTcVec {
  float wq[kH], Wa[kTcMaxFe * kH], b2[kH], b3[kH], w4[kH], wa[kH];
  float ba;
  int srow[kTM], scol[kTM];
  float sq[kTM], sdn[kTM * 3], sea[kTM * kTcMaxFe];
  float spart[kTM];          // second-half partial sums (phi_x output dot, attention logit)
  uint64_t bar[2];
  uint32_t tmem_slot;
};

// One operand tile (hi [+ lo]) is enough: GEMM1 has finished reading a1 before epilogue 1 writes m in place.
template <int SPLIT>
struct EdgeTcSmem {
  static constexpr int kW = kH * kH * 4;            // one 64x64 fp32 weight tile, bytes
  static constexpr int kT = kTM * kH * 4;           // one 128x64 fp32 operand tile, bytes
  static constexpr int kParts = SPLIT == 3 ? 2 : 1; // hi (+ lo)
  static constexpr int off_W2 = 0;
  static constexpr int off_W3 = off_W2 + kParts * kW;
  static constexpr int off_A = off_W3 + kParts * kW;
  static constexpr int off_vec = off_A + kParts * kT;
  static constexpr size_t bytes = off_vec + sizeof(EdgeTcVec) + 1024;   // + alignment slack
  static constexpr int ctas_per_sm = SPLIT == 3 ? 1 : 3;
};

// 16-byte chunk c of row n of the reference [64][ld] matrices -> chunk slot of the swizzled tiles.  Both weights are loaded
// before the first store (one L2 round trip for the prologue).
template <int SPLIT>
__device__ __forceinline__ void tc_stage_weights2(uint8_t* dst0, const float* __restrict__ g0, uint8_t* dst1,
                                                  const float* __restrict__ g1, int ld) {
  constexpr int NJ = kH * 16 / kTcThreads;
  float4 w0[NJ], w1[NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const int i = threadIdx.x + j * kTcThreads, n = i >> 4, c = i & 15;
    w0[j] = *reinterpret_cast<const float4*>(g0 + (size_t)n * ld + c * 4);
    w1[j] = *reinterpret_cast<const float4*>(g1 + (size_t)n * ld + c * 4);
  }
#pragma unroll
  for (int j = 0; j < 2 * NJ; ++j) {
    const int jj = j % NJ;
    const int i = threadIdx.x + jj * kTcThreads, n = i >> 4, c = i & 15;
    const float4 w = j < NJ ? w0[jj] : w1[jj];
    uint8_t* dst = j < NJ ? dst0 : dst1;
    const uint32_t o = umma::tile_chunk_off(n, c, kH);
    if (SPLIT == 3) {
      const float4 hi = make_float4(umma::to_tf32(w.x), umma::to_tf32(w.y), umma::to_tf32(w.z), umma::to_tf32(w.w));
      *reinterpret_cast<float4*>(dst + o) = hi;
      *reinterpret_cast<float4*>(dst + EdgeTcSmem<SPLIT>::kW + o) = make_float4(w.x - hi.x, w.y - hi.y, w.z - hi.z, w.w - hi.w);
    } else {
      *reinterpret_cast<float4*>(dst + o) = w;
    }
  }
}

// store 2 consecutive columns (col, col+1; col even) of row `row` into an operand tile (hi [+ lo])
template <int SPLIT>
__device__ __forceinline__ void tc_store_pair(uint8_t* tile, int row, int col, float2 v) {
  const uint32_t o = umma::tile_off(row, col, kTM);
  if (SPLIT == 3) {
    float2 hi = make_float2(umma::to_tf32(v.x), umma::to_tf32(v.y));
    *reinterpret_cast<float2*>(tile + o) = hi;
    *reinterpret_cast<float2*>(tile + EdgeTcSmem<SPLIT>::kT + o) = make_float2(v.x - hi.x, v.y - hi.y);
  } else {
    *reinterpret_cast<float2*>(tile + o) = v;
  }
}

// store 4 consecutive columns (chunk c) of row `row` into an operand tile (hi [+ lo])
template <int SPLIT>
__device__ __forceinline__ void tc_store_chunk(uint8_t* tile, int row, int c, float4 v) {
  const uint32_t o = umma::tile_chunk_off(row, c, kTM);
  if (SPLIT == 3) {
    float4 hi = make_float4(umma::to_tf32(v.x), umma::to_tf32(v.y), umma::to_tf32(v.z), umma::to_tf32(v.w));
    *reinterpret_cast<float4*>(tile + o) = hi;
    *reinterpret_cast<float4*>(tile + EdgeTcSmem<SPLIT>::kT + o) = make_float4(v.x - hi.x, v.y - hi.y, v.z - hi.z, v.w - hi.w);
  } else {
    *reinterpret_cast<float4*>(tile + o) = v;
  }
}

// D = A W^T with A (hi[,lo]) at a_tile and W (hi[,lo]) at w_tile
template <int SPLIT>
__device__ __forceinline__ void tc_issue_gemm(uint32_t tmem_d, uint64_t a_desc, uint64_t w_desc, uint32_t idesc) {
  umma::gemm_k64_desc(tmem_d, a_desc, kTM, w_desc, kH, idesc, false);
  if (SPLIT == 3) {
    umma::gemm_k64_desc(tmem_d, a_desc + (uint64_t)(EdgeTcSmem<SPLIT>::kT >> 4), kTM, w_desc, kH, idesc, true);
    umma::gemm_k64_desc(tmem_d, a_desc, kTM, w_desc + (uint64_t)(EdgeTcSmem<SPLIT>::kW >> 4), kH, idesc, true);
  }
}


// SiLU of the tensor-core kernels.  SPLIT == 3 (fp32-grade): z / (1 + 2^(-z log2 e)), two MUFU ops.
// SPLIT == 1 (TF32-grade): z (0.5 + 0.5 tanh.approx(z/2)), one MUFU op; tanh.approx has ~2^-11 relative error,
// the same order as the TF32 operand rounding of that mode.
// With t = z / 2: z (0.5 + 0.5 tanh t) = t + t tanh t -- FMUL, MUFU, FFMA; with the bias pre-halved in shared memory
// (tc_silu_hb) the bias add and the halving are one FFMA: 3 instructions per activation instead of 5.
template <int SPLIT>
__device__ __forceinline__ float tc_silu(float z) {
  if (SPLIT == 3) return silu_f(z);
  const float t = 0.5f * z;
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(t));
  return fmaf(t, th, t);
}
// silu(z + b); `b` is the bias (SPLIT == 3) resp. HALF the bias (SPLIT == 1), as staged by the kernel prologue
template <int SPLIT>
__device__ __forceinline__ float tc_silu_hb(float z, float b) {
  if (SPLIT == 3) return silu_f(z + b);
  const float t = fmaf(z, 0.5f, b);
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(t));
  return fmaf(t, th, t);
}

// kDet: msum / tsum through edge_det_msum / edge_det_tsum and the boundary slab (edge_kernels.cu; same terms, summed in row
// order)
template <int SPLIT, bool kDet>
__global__ void __launch_bounds__(kTcThreads, EdgeTcSmem<SPLIT>::ctas_per_sm) edge_fwd_tc_kernel(EdgeArgs a) {
  using SM = EdgeTcSmem<SPLIT>;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment for SWIZZLE_128B, derived from the __shared__ symbol so that accesses stay LDS/STS
  uint8_t* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
  pdl_trigger();
  EdgeTcVec* v = reinterpret_cast<EdgeTcVec*>(smem + SM::off_vec);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  // thread (warp, lane) owns row (warp&3)*32 + lane (a TMEM lane) and the 32 columns of half `half`
  const int row = (warp & 3) * 32 + lane, half = warp >> 2;
  const bool att = a.flags & FEGNN_F_ATTENTION, use_tanh = a.flags & FEGNN_F_TANH, norm = a.flags & FEGNN_F_NORMALIZE;

  tc_stage_weights2<SPLIT>(smem + SM::off_W2, a.W2, smem + SM::off_W3, a.W3, kH);
  for (int i = t; i < kH; i += kTcThreads) {
    v->wq[i] = a.w1[(size_t)i * a.ld1 + 2 * kH];
    for (int f = 0; f < a.Fe; ++f) v->Wa[f * kH + i] = a.w1[(size_t)i * a.ld1 + 2 * kH + 1 + f];
    v->b2[i] = (SPLIT == 3 ? 1.f : 0.5f) * a.b2[i];      // tc_silu_hb
    v->b3[i] = (SPLIT == 3 ? 1.f : 0.5f) * a.b3[i];
    v->w4[i] = a.w4[i];
    if (att) v->wa[i] = a.wa[i];
  }
  if (t == 0) {
    if (att) v->ba = a.ba[0];
    umma::mbar_init(&v->bar[0], 1);
    umma::mbar_init(&v->bar[1], 1);
    umma::mbar_fence_init();
  }
  if (warp == 0) umma::tmem_alloc<128>(&v->tmem_slot);
  umma::fence_smem_to_async();
  umma::fence_before();
  __syncthreads();
  umma::fence_after();
  pdl_wait();
  const uint32_t tmem = v->tmem_slot;
  const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16) + half * 32;
  const uint32_t idesc = umma::make_idesc_tf32(128, 64);
  const uint64_t dW2 = umma::make_desc(umma::smem_u32(smem + SM::off_W2)), dW3 = umma::make_desc(umma::smem_u32(smem + SM::off_W3));
  const uint64_t dA = umma::make_desc(umma::smem_u32(smem + SM::off_A));
  uint8_t* At = smem + SM::off_A;
  uint32_t phase = 0;

  const int ntiles = (a.E + kTM - 1) / kTM;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    umma::fence_before();
    __syncthreads();                       // previous tile fully consumed (per-row scalars, TMEM columns, operand tile)
    // ---- geometry: one thread per edge
    if (t < kTM) {
      const int e = tile * kTM + t;
      int r = -1, c = 0;
      float d0 = 0, d1 = 0, d2 = 0, q = 0;
      if (e < a.E) {
        r = a.row[e];
        c = a.col[e];
        d0 = a.x[(size_t)r * 3 + 0] - a.x[(size_t)c * 3 + 0];
        d1 = a.x[(size_t)r * 3 + 1] - a.x[(size_t)c * 3 + 1];
        d2 = a.x[(size_t)r * 3 + 2] - a.x[(size_t)c * 3 + 2];
        q = d0 * d0 + d1 * d1 + d2 * d2;
        if (norm) {
          const float inv = 1.f / (sqrtf(q) + a.eps);
          d0 *= inv; d1 *= inv; d2 *= inv;
        }
        for (int f = 0; f < a.Fe; ++f) v->sea[t * kTcMaxFe + f] = a.ea[(size_t)e * a.Fe + f];
      } else {
        for (int f = 0; f < a.Fe; ++f) v->sea[t * kTcMaxFe + f] = 0.f;
      }
      v->srow[t] = r;
      v->scol[t] = c;
      v->sq[t] = q;
      v->sdn[t * 3 + 0] = d0; v->sdn[t * 3 + 1] = d1; v->sdn[t * 3 + 2] = d2;
    }
    __syncthreads();
    // ---- a1 = silu(P[row] + Q[col] + q wq + Wa a_e) -> operand tile.  Warp w builds rows 16w..16w+15, two rows per
    //      step: a half-warp gathers one 256-byte row of P and of Q as 16 float4 (lane&15 = 16-byte chunk), so a
    //      chunk goes from global memory to its swizzled slot with one LDG.128 x2 and one STS.128.
    {
      const int l16 = lane & 15, hsel = lane >> 4;
      const float4 wq = *reinterpret_cast<const float4*>(v->wq + 4 * l16);
#pragma unroll 1
      for (int i0 = 0; i0 < 16; i0 += 8) {
        float4 p[4], qv[4];
        int ri[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int rr = warp * 16 + i0 + 2 * j + hsel;
          ri[j] = v->srow[rr];
          p[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          qv[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ri[j] >= 0) {
            p[j] = *reinterpret_cast<const float4*>(a.P + (size_t)ri[j] * kH + 4 * l16);
            qv[j] = *reinterpret_cast<const float4*>(a.Q + (size_t)v->scol[rr] * kH + 4 * l16);
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int rr = warp * 16 + i0 + 2 * j + hsel;
          const float qi = v->sq[rr];
          float z0 = p[j].x + qv[j].x + qi * wq.x, z1 = p[j].y + qv[j].y + qi * wq.y,
                z2 = p[j].z + qv[j].z + qi * wq.z, z3 = p[j].w + qv[j].w + qi * wq.w;
#pragma unroll
          for (int f = 0; f < kTcMaxFe; ++f) {
            if (f < a.Fe) {
              const float ef = v->sea[rr * kTcMaxFe + f];
              const float4 wf = *reinterpret_cast<const float4*>(v->Wa + f * kH + 4 * l16);
              z0 = fmaf(ef, wf.x, z0); z1 = fmaf(ef, wf.y, z1); z2 = fmaf(ef, wf.z, z2); z3 = fmaf(ef, wf.w, z3);
            }
          }
          float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ri[j] >= 0) o = make_float4(tc_silu<SPLIT>(z0), tc_silu<SPLIT>(z1), tc_silu<SPLIT>(z2), tc_silu<SPLIT>(z3));
          tc_store_chunk<SPLIT>(At, rr, l16, o);
        }
      }
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    __syncthreads();
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
        tc_issue_gemm<SPLIT>(tmem, dA, dW2, idesc);
        umma::commit(&v->bar[0]);
      }
      __syncwarp();
    }
    umma::mbar_wait(&v->bar[0], phase);
    umma::fence_after();
    // ---- epilogue 1: m = silu(z2 + b2) [* gate] -> operand tile (in place of a1: GEMM1 is complete)
    {
      float m[32];
      umma::tmem_ld32(tlane, m);
#pragma unroll
      for (int j = 0; j < 32; ++j) m[j] = tc_silu_hb<SPLIT>(m[j], v->b2[half * 32 + j]);
      if (att) {
        float dot = 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j) dot = fmaf(m[j], v->wa[half * 32 + j], dot);
        if (half == 1) v->spart[row] = dot;
        __syncthreads();
        const float other = half == 1 ? 0.f : v->spart[row];
        __syncthreads();
        if (half == 0) v->spart[row] = dot;
        __syncthreads();
        const float tot = half == 0 ? dot + other : dot + v->spart[row];
        const float gate = sigmoid_f(tot + v->ba);
#pragma unroll
        for (int j = 0; j < 32; ++j) m[j] *= gate;
      }
#pragma unroll
      for (int ch = 0; ch < 8; ++ch)
        tc_store_chunk<SPLIT>(At, row, half * 8 + ch, make_float4(m[ch * 4], m[ch * 4 + 1], m[ch * 4 + 2], m[ch * 4 + 3]));
    }
    umma::fence_smem_to_async();
    umma::fence_before();
    __syncthreads();
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
        tc_issue_gemm<SPLIT>(tmem + 64, dA, dW3, idesc);
        umma::commit(&v->bar[1]);
      }
      __syncwarp();
    }
    // ---- msum: walk over the m tile while the tensor core runs (read-only on both sides).  Thread (c4, grp) owns the
    //      16-byte column quad c4 of the 8 rows of swizzle atom grp: one LDS.128 per row, one red.global.add.v4.f32 per
    //      run of equal row ids (the scalar 32-row column walk this replaces was 17 % of the kernel's instructions).
    if constexpr (kDet) {
      edge_det_msum(a, v->srow, tile, [&](int rr, int c4) {
        const uint32_t o = (c4 >> 3) * (kTM * 128) + (rr >> 3) * 1024 + (rr & 7) * 128 + (((c4 & 7) ^ (rr & 7)) << 4);
        float4 mv = *reinterpret_cast<const float4*>(At + o);
        if (SPLIT == 3) {
          const float4 lo = *reinterpret_cast<const float4*>(At + SM::kT + o);
          mv.x += lo.x; mv.y += lo.y; mv.z += lo.z; mv.w += lo.w;
        }
        return mv;
      });
    } else {
      const int c4 = t & 15, grp = t >> 4;
      const uint8_t* gbase = At + (c4 >> 3) * (kTM * 128) + grp * 1024;
      int cur = -1;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = v->srow[grp * 8 + j];
        const uint32_t o = j * 128 + (((c4 & 7) ^ j) << 4);
        float4 mv = *reinterpret_cast<const float4*>(gbase + o);
        if (SPLIT == 3) {
          const float4 lo = *reinterpret_cast<const float4*>(gbase + SM::kT + o);
          mv.x += lo.x; mv.y += lo.y; mv.z += lo.z; mv.w += lo.w;
        }
        if (k != cur) {
          if (cur >= 0) atomicAdd(reinterpret_cast<float4*>(a.msum + (size_t)cur * kH + c4 * 4), acc);
          cur = k;
          acc = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (k >= 0) { acc.x += mv.x; acc.y += mv.y; acc.z += mv.z; acc.w += mv.w; }
      }
      if (cur >= 0) atomicAdd(reinterpret_cast<float4*>(a.msum + (size_t)cur * kH + c4 * 4), acc);
    }
    umma::mbar_wait(&v->bar[1], phase);
    umma::fence_after();
    phase ^= 1;
    // ---- epilogue 2: s = w4 . silu(z3 + b3) ; tsum[row] += dn * s
    {
      float z[32];
      umma::tmem_ld32(tlane + 64, z);
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 32; ++j) s = fmaf(tc_silu_hb<SPLIT>(z[j], v->b3[half * 32 + j]), v->w4[half * 32 + j], s);
      if (half == 1) v->spart[row] = s;
      __syncthreads();
      if constexpr (kDet) {
        if (half == 0) {
          s += v->spart[row];
          if (use_tanh) s = tanhf(s);
          v->sq[row] = s;                  // sq (|x_i - x_j|^2) was last read by the assembly
        }
        __syncthreads();
        edge_det_tsum(a, v->srow, tile, [&](int rr, int k) { return v->sdn[rr * 3 + k] * v->sq[rr]; });
      } else if (half == 0) {
        s += v->spart[row];
        if (use_tanh) s = tanhf(s);
        const int r = v->srow[row];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          bool tail;
          float tot = warp_segsum(r >= 0 ? v->sdn[row * 3 + k] * s : 0.f, r, lane, tail);
          if (tail && r >= 0) atomicAdd(a.tsum + (size_t)r * 3 + k, tot);
        }
      }
    }
  }
  umma::fence_before();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc<128>(tmem);
}

template <int SPLIT, bool kDet = false>
cudaError_t launch_edge_fwd_tc(const EdgeArgs& a, int sms, cudaStream_t st) {
  static DevOnce attr;
  const size_t bytes = EdgeTcSmem<SPLIT>::bytes;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(edge_fwd_tc_kernel<SPLIT, kDet>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  const int ntiles = (a.E + kTM - 1) / kTM;
  if (ntiles == 0) return cudaSuccess;
  const int per_sm = EdgeTcSmem<SPLIT>::ctas_per_sm;
  const int grid = ntiles < per_sm * sms ? ntiles : per_sm * sms;
  if (cudaError_t e_ = launch_pdl(edge_fwd_tc_kernel<SPLIT, kDet>, grid, kTcThreads, bytes, st, a)) return e_;
  if (cudaError_t e_ = cudaGetLastError()) return e_;
  return kDet ? launch_edge_det_fixup(a, st) : cudaSuccess;
}

}  // namespace fegnn
