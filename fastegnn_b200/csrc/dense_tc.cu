// dense_tc.cu -- the per-node dense phases of the BACKWARD pass on the 5th-generation tensor cores (tcgen05 + TMEM).
//
// node_pre_backward (models/FastEGNN.py:104,115,139,142,162, h-side halves of every first Linear) and node_h_backward
// (phi_h, :153-166) are sums of [128 x 64] x [64 x 64] products per node tile and weight block:
//     D_b   = X_b W_b                      data gradient   (gh += gP Ws, gm = gzh1 U1a, gu_c = gzh1 U1u_c, gzh1 = gh' U2 ...)
//     dW_b += X_b^T Y_b ,  db_b += sum X_b  weight gradient (Y_b = h, msum / deg, u_c, silu(zh1))
// They were fp32-FMA kernels (19 TFLOP/s at Water-3D: 8.6 % + 7.5 % of the step's kernel time, 24 % at 1 M nodes).  Here ONE
// generic kernel runs any list of such blocks: work item = (node tile, block); the row owner thread (one TMEM lane) loads
// its X and Y rows from global memory straight into registers, writes X to tensor memory (the TS-form A operand of the data
// gradient, as in edge_tc_bwd2.cu) and both rows to row-major SWIZZLE_128B_BASE32B tiles, which the weight-gradient GEMM
// reads as MN-major operands (no transposed copies); dW accumulates in tensor memory across the CTA's tiles.  Backward-only:
// TF32 rounding of gradients does not touch the forward equivariance (DESIGN.md 3.2).
// Head blocks (phi_v / phi_g, :139,:142) first recompute z = h W^T on the tensor core and form X = gs w2 silu'(z + b).
#include "common.cuh"
#include "umma.cuh"

namespace fegnn {
namespace dtc {

using bwd2::desc_advance;
using bwd2::gemm_ts_kmajor;
using bwd2::gemm_ts_mn;
using bwd2::idesc_tf32;
using bwd2::make_desc_mn;
using bwd2::mn_chunk_off;
using bwd2::mn_load_row;
using bwd2::mn_off;
using bwd2::mn_store_row;
using bwd2::tmem_ld;
using bwd2::tmem_st;
using bwd2::tmem_st_wait;

constexpr int kMaxBlk = FEGNN_MAX_C + 2;
// Up to this many node tiles per SM the per-tile kernel (below) is used: every size.  It was written for small graphs, but
// measured on the B200 it also wins where the (tile, block) kernel was the default (no red.add pass over [N, 64] per block):
// 12.89 -> 11.95 ms per step at 160 000 nodes / 3.6 M edges, 122.8 -> 120.1 ms at 1 M nodes / C = 8.  The (tile, block) kernel
// stays selectable (FEGNN_DENSE_ROWS_MAX_TILES_PER_SM=2).
constexpr int kRowsMaxTilesPerSm = 1 << 20;

struct Blk {
  // X rows [N][64] (row stride ldx floats), optional per-row scale: the gradient-side operand
  const float* X;
  const float* xscale;
  // Y rows [N][64] (row stride ldy), optional per-row scale, ysilu: Y = silu(rows)
  const float* Y;
  const float* yscale;
  // weight block: element (n, k) = W[n * ldw + k * wks]   (n = output feature of the forward Linear, k = input feature)
  const float* W;
  // D = X W (rows [N][64], stride ldd): dmode 0 none, 1 store, 2 red.add ; optional D *= silu'(dz row) ; D *= dscale[row]
  float* D;
  const float* dz;
  const float* dscale;
  unsigned* dmax; // per-tile kernel: atomicMax of the bit patterns of |D| (bound statistic of a consumer), or nullptr
  float* gW;     // += X^T Y   (same ldw / wks addressing)
  float* gb;     // += column sums of X (or nullptr)
  // head block (phi_v / phi_g): X = gs[row] * hw2 * silu'(Y W^T + hb) ; g_hw2 += sum gs silu(z) ; g_hb2 += sum gs
  const float *gs, *hb, *hw2;
  float *g_hw2, *g_hb2;
  int ldx, ldy, ldd, ldw, wks, dmode, ysilu, head;
};

struct Args {
  int N, nblk;
  unsigned same_y_mask, chain_mask;   // bit b: block b reads block b - 1's Y tile / block b + 1 adds into block b's D (host-computed)
  int nsplit;                  // per-tile kernel: the block list is cut into nsplit ranges, one CTA per (tile, range)
  int split[kMaxBlk + 1];      // range s = blocks [split[s], split[s + 1])
  Blk blk[kMaxBlk];
};

struct Vec {
  float hb[kH], hw2[kH];
  float cb[kH], cw2[kH];          // per-CTA column sums (bias gradient, head output-weight gradient)
  float cb2;
  uint64_t bar[3];
  uint32_t tmem_slot;
};
struct Smem {
  static constexpr int kW = kH * kH * 4, kT = kTM * kH * 4;
  static constexpr int off_Wm = 0, off_Wk = kW, off_TY = 2 * kW, off_TX = 2 * kW + kT, off_vec = 2 * kW + 2 * kT;
  static constexpr size_t bytes = off_vec + sizeof(Vec) + 1024;
};
constexpr uint32_t kACC = 0, kOPA = 64, kRW = 128;      // tensor-memory columns (256 allocated: two CTAs per SM)

// Node attributes (node_pre_backward with Fa > 0): block at.blk (Uh) also adds dU1att += X^T a (NodeAttrArgs) -- a column
// walk over the X tile weighted by the attribute rows, fp32, like the bias sums.  Only the kAttr instantiations use it.
struct AttrBlk {
  NodeAttrArgs at;
  int blk;
};
__host__ __device__ constexpr int attr_off(size_t base) { return (int)((base + 15) / 16 * 16); }

template <int CG, bool kAttr>
__global__ void __launch_bounds__(128 * CG, 2) dense_bwd_tc_kernel(const __grid_constant__ Args a, const AttrBlk ab) {
  constexpr int NT = 128 * CG, CPT = kH / CG;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
  pdl_trigger();
  Vec* v = reinterpret_cast<Vec*>(smem + Smem::off_vec);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int quarter = warp & 3, cg = warp >> 2, row = quarter * 32 + lane, c0 = cg * CPT;
  const int bid = blockIdx.x % a.nblk, cta = blockIdx.x / a.nblk, nctas = gridDim.x / a.nblk;
  const Blk& b = a.blk[bid];
  uint8_t *Wm = smem + Smem::off_Wm, *Wk = smem + Smem::off_Wk, *TY = smem + Smem::off_TY, *TX = smem + Smem::off_TX;
  [[maybe_unused]] const bool attr = kAttr && bid == ab.blk;         // uniform over the CTA
  [[maybe_unused]] float* sA = reinterpret_cast<float*>(smem + attr_off(Smem::off_vec + sizeof(Vec)));
  [[maybe_unused]] float* sRed = sA + kTM * kMaxFa;
  [[maybe_unused]] float sa[kMaxFa];
  if constexpr (kAttr) {
#pragma unroll
    for (int f = 0; f < kMaxFa; ++f) sa[f] = 0.f;
    for (int i = t; i < kMaxFa * kH; i += NT) sRed[i] = 0.f;
  }

  // ---- prologue: weight block in both layouts (MN-major for X W; K-major only for the head recompute), vectors
  {
    float w[kH * kH / NT];                       // every load in flight before the first store: one L2 round trip
#pragma unroll
    for (int j = 0; j < kH * kH / NT; ++j) {
      const int i = t + j * NT, n = i >> 6, k = i & 63;
      w[j] = b.W[(size_t)n * b.ldw + (size_t)k * b.wks];
    }
#pragma unroll
    for (int j = 0; j < kH * kH / NT; ++j) {
      const int i = t + j * NT, n = i >> 6, k = i & 63;
      *reinterpret_cast<float*>(Wm + mn_off(n, k, kH)) = w[j];
      if (b.head) *reinterpret_cast<float*>(Wk + umma::tile_off(n, k, kH)) = w[j];
    }
  }
  for (int i = t; i < kH; i += NT) {
    v->hb[i] = b.head ? b.hb[i] : 0.f;
    v->hw2[i] = b.head ? b.hw2[i] : 0.f;
    v->cb[i] = 0.f;
    v->cw2[i] = 0.f;
  }
  if (t == 0) {
    v->cb2 = 0.f;
#pragma unroll
    for (int i = 0; i < 3; ++i) umma::mbar_init(&v->bar[i], 1);
    umma::mbar_fence_init();
  }
  if (warp == 0) umma::tmem_alloc<256>(&v->tmem_slot);
  umma::fence_smem_to_async();
  umma::fence_before();
  __syncthreads();
  umma::fence_after();
  pdl_wait();
  const uint32_t tmem = v->tmem_slot;
  const uint32_t tlane = tmem + ((uint32_t)(quarter * 32) << 16) + c0;
  const uint32_t id_ts_k = idesc_tf32(128, 64, 0, 0), id_ts_mn = idesc_tf32(128, 64, 0, 1), id_wg = idesc_tf32(64, 64, 1, 1);
  const uint64_t dWm = make_desc_mn(umma::smem_u32(Wm), kH * 128), dWk = umma::make_desc(umma::smem_u32(Wk));
  const uint64_t dTX = make_desc_mn(umma::smem_u32(TX), kTM * 128), dTY = make_desc_mn(umma::smem_u32(TY), kTM * 128);
  uint32_t ph_r = 0, ph_d = 0, ph_w = 0;
  bool first = true;
  const bool want_w = b.gW != nullptr;

  const int ntiles = (a.N + kTM - 1) / kTM;
  for (int tile = cta; tile < ntiles; tile += nctas) {
    const int i0 = tile * kTM, r = i0 + row;
    const bool valid = r < a.N;
    if (!first && want_w) {                       // the previous tile's weight-gradient GEMM still reads TX / TY
      umma::mbar_wait(&v->bar[2], ph_w);
      umma::fence_after();
      ph_w ^= 1;
    }
    // ---- Y row -> registers -> TY (and tensor memory for the head recompute)
    float y[CPT], x[CPT];
    if (valid) {
      const float4* src = reinterpret_cast<const float4*>(b.Y + (size_t)r * b.ldy + c0);
      const float s = b.yscale != nullptr ? b.yscale[r] : 1.f;
#pragma unroll
      for (int ch = 0; ch < CPT / 4; ++ch) {
        const float4 q = src[ch];
        y[ch * 4] = q.x * s; y[ch * 4 + 1] = q.y * s; y[ch * 4 + 2] = q.z * s; y[ch * 4 + 3] = q.w * s;
      }
      if (b.ysilu) {
#pragma unroll
        for (int j = 0; j < CPT; ++j) y[j] = silu_f(y[j]);
      }
    } else {
#pragma unroll
      for (int j = 0; j < CPT; ++j) y[j] = 0.f;
    }
    mn_store_row<CPT>(TY, row, cg, y);
    if (b.head) {
      tmem_st<CPT>(tlane + kOPA, y);
      tmem_st_wait();
      umma::fence_before();
      __syncthreads();
      if (warp == 0) {
        umma::fence_after();
        if (umma::elect_one()) {
          gemm_ts_kmajor(tmem + kACC, tmem + kOPA, dWk, id_ts_k);           // z = Y W^T
          umma::commit(&v->bar[0]);
        }
        __syncwarp();
      }
      umma::mbar_wait(&v->bar[0], ph_r);
      umma::fence_after();
      ph_r ^= 1;
      tmem_ld<CPT>(tlane + kACC, x);
      const float g = valid ? b.gs[r] : 0.f;
      float aw[CPT];
#pragma unroll
      for (int j = 0; j < CPT; ++j) {
        float av, d;
        silu_grad_f(x[j] + v->hb[c0 + j], av, d);
        aw[j] = g * av;
        x[j] = g * v->hw2[c0 + j] * d;
      }
      // g_hw2 += sum_rows gs * silu(z): warp-reduce over the 32 rows of this warp, one shared-memory atomic per column
#pragma unroll
      for (int j = 0; j < CPT; ++j) {
        float s = aw[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) atomicAdd(&v->cw2[c0 + j], s);
      }
      if (cg == 0) {
        float s = g;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) atomicAdd(&v->cb2, s);
      }
    } else if (valid) {
      const float4* src = reinterpret_cast<const float4*>(b.X + (size_t)r * b.ldx + c0);
      const float s = b.xscale != nullptr ? b.xscale[r] : 1.f;
#pragma unroll
      for (int ch = 0; ch < CPT / 4; ++ch) {
        const float4 q = src[ch];
        x[ch * 4] = q.x * s; x[ch * 4 + 1] = q.y * s; x[ch * 4 + 2] = q.z * s; x[ch * 4 + 3] = q.w * s;
      }
    } else {
#pragma unroll
      for (int j = 0; j < CPT; ++j) x[j] = 0.f;
    }
    if (b.gb != nullptr) {                         // bias gradient: column sums of X in fp32 (not through the TF32 MMA)
#pragma unroll
      for (int j = 0; j < CPT; ++j) {
        float s = x[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) atomicAdd(&v->cb[c0 + j], s);
      }
    }
    tmem_st<CPT>(tlane + kOPA, x);
    mn_store_row<CPT>(TX, row, cg, x);
    if constexpr (kAttr) {
      if (attr) attr_load_tile(sA, ab.at, i0, min(kTM, a.N - i0), NT);
    }
    tmem_st_wait();
    umma::fence_smem_to_async();
    umma::fence_before();
    __syncthreads();
    if constexpr (kAttr) {
      if (attr) {                                  // TX is rewritten by the next tile only after the barrier below
        attr_wgrad_walk(sa, sA, ab.at.Fa, [&](int rr, int c) { return *reinterpret_cast<const float*>(TX + mn_off(rr, c, kTM)); });
        __syncthreads();
      }
    }
    if (warp == 0) {
      umma::fence_after();
      if (umma::elect_one()) {
        if (b.dmode != 0) {
          gemm_ts_mn(tmem + kACC, tmem + kOPA, dWm, id_ts_mn);               // D = X W
          umma::commit(&v->bar[1]);
        }
        if (want_w) {
#pragma unroll
          for (int ks = 0; ks < 16; ++ks)                                     // dW (+)= X^T Y over the 128 rows
            umma::mma_tf32(tmem + kRW, desc_advance(dTX, ks * 1024), desc_advance(dTY, ks * 1024), id_wg,
                           (ks > 0 || !first) ? 1u : 0u);
          umma::commit(&v->bar[2]);
        }
      }
      __syncwarp();
    }
    if (b.dmode != 0) {
      umma::mbar_wait(&v->bar[1], ph_d);
      umma::fence_after();
      ph_d ^= 1;
      float d[CPT];
      tmem_ld<CPT>(tlane + kACC, d);
      if (valid) {
        if (b.dz != nullptr) {
          const float4* zr = reinterpret_cast<const float4*>(b.dz + (size_t)r * kH + c0);
#pragma unroll
          for (int ch = 0; ch < CPT / 4; ++ch) {
            const float4 z = zr[ch];
            float av, e0, e1, e2, e3;
            silu_grad_f(z.x, av, e0); silu_grad_f(z.y, av, e1); silu_grad_f(z.z, av, e2); silu_grad_f(z.w, av, e3);
            d[ch * 4] *= e0; d[ch * 4 + 1] *= e1; d[ch * 4 + 2] *= e2; d[ch * 4 + 3] *= e3;
          }
        }
        const float s = b.dscale != nullptr ? b.dscale[r] : 1.f;
        float4* dst = reinterpret_cast<float4*>(b.D + (size_t)r * b.ldd + c0);
#pragma unroll
        for (int ch = 0; ch < CPT / 4; ++ch) {
          const float4 q = make_float4(d[ch * 4] * s, d[ch * 4 + 1] * s, d[ch * 4 + 2] * s, d[ch * 4 + 3] * s);
          if (b.dmode == 2) atomicAdd(dst + ch, q);
          else dst[ch] = q;
        }
      }
      umma::fence_before();                        // ACC / OPA are rewritten by the next tile
    }
    first = false;
  }
  // ---- flush: weight gradient (M = 64 layout: row n in lane (n / 16) * 32 + n % 16), bias sums
  if (!first && want_w) {
    umma::mbar_wait(&v->bar[2], ph_w);
    umma::fence_after();
  }
  __syncthreads();
  if (!first && want_w) {
    float w[CPT];
    tmem_ld<CPT>(tlane + kRW, w);
    if (lane < 16) {
      const int n = quarter * 16 + lane;
      float* dst = b.gW + (size_t)n * b.ldw + (size_t)c0 * b.wks;
      if (b.wks == 1 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
        for (int j = 0; j < CPT; j += 4) atomicAdd(reinterpret_cast<float4*>(dst + j), make_float4(w[j], w[j + 1], w[j + 2], w[j + 3]));
      } else {
#pragma unroll
        for (int j = 0; j < CPT; ++j) atomicAdd(dst + (size_t)j * b.wks, w[j]);
      }
    }
  }
  if (!first && t < kH) {
    if (b.gb != nullptr) atomicAdd(b.gb + t, v->cb[t]);
    if (b.head && b.g_hw2 != nullptr) atomicAdd(b.g_hw2 + t, v->cw2[t]);
    if (b.head && t == 0 && b.g_hb2 != nullptr) atomicAdd(b.g_hb2, v->cb2);
  }
  if constexpr (kAttr) {
    if (attr && !first) attr_wgrad_flush(sa, sRed, ab.at);
  }
  umma::fence_before();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc<256>(tmem);
}


// ------------------------------------------------------------------------------------------------- small-N form
// The (tile, block) decomposition above pays its fixed costs per work item: at 8 000 nodes (63 tiles) every CTA stages a weight
// block, allocates tensor memory, handles ONE tile and flushes 4 096 weight-gradient atomics -- and `gh += G_b W_b` goes through
// global atomics once per block.  Here a CTA owns a node tile and WALKS the blocks:
//   * the data gradients of consecutive blocks that add into the same D (node_pre_backward: gh) accumulate in ONE tensor-memory
//     accumulator across the blocks -- one epilogue per tile instead of one red.add pass per block;
//   * Y (= h for every node_pre block) is loaded once per tile when consecutive blocks share it;
//   * software pipeline over the blocks: the weight block and the X / Y rows of block b + 1 are in flight (registers) while the
//     MMAs of block b run and the weight gradient of block b - 1 is flushed; weight tiles, X tiles, Y tiles and the weight-gradient
//     accumulators are double-buffered;
//   * bias column sums come from a column walk over the X tile under the MMA (was 160 shuffles per thread).
// Used below kRowsMaxTiles tiles per SM-pair (small graphs); the (tile, block) kernel stays for large N, where its weights are
// staged once per CTA for many tiles.
struct VecR {
  float hb[kH], hw2[kH];
  float cb[2][kH], cw2[kH];
  float cb2;
  uint64_t bar[4];                // 0 head recompute, 1 data gradient, 2 / 3 weight gradient of slot 0 / 1
  uint32_t tmem_slot;
};
struct SmemR {
  static constexpr int kW = kH * kH * 4, kT = kTM * kH * 4;
  static constexpr int kFS = kH * 65 * 4;          // weight-gradient staging [64][65] (transposed through shared memory)
  static constexpr int off_Wm = 0;                 // [2] MN-major weight tiles
  static constexpr int off_Wk = 2 * kW;            // K-major copy (head recompute only)
  static constexpr int off_TY = 3 * kW;            // [2]
  static constexpr int off_TX = 3 * kW + 2 * kT;   // [2]
  static constexpr int off_FS = 3 * kW + 4 * kT;
  static constexpr int off_vec = off_FS + ((kFS + 15) / 16) * 16;
  static constexpr size_t bytes = off_vec + sizeof(VecR) + 1024;
};
constexpr uint32_t kR_ACC = 0, kR_OPA = 64, kR_RW = 128;      // + 64 * slot ; 256 columns

__device__ __forceinline__ void gemm_ts_mn_acc(uint32_t tmem_d, uint32_t tmem_a, uint64_t dW, uint32_t idesc, bool accumulate) {
#pragma unroll
  for (int ks = 0; ks < 8; ++ks)
    bwd2::mma_ts(tmem_d, tmem_a + ks * 8, desc_advance(dW, ks * 1024), idesc, (ks > 0 || accumulate) ? 1u : 0u);
}
#ifdef FEGNN_TRACE
#define TR(i) do { if (threadIdx.x == 0 && blockIdx.x == 1 && blockIdx.y == 0) tr_[(i)] = clock64(); } while (0)
#else
#define TR(i) do { } while (0)
#endif
// Data movement (measured with clock64 stamps, tools/gpu_r2_ab.sh: the row-owner form -- every thread loading / storing ITS
// row -- made each warp-wide 16-byte access touch 32 cache lines; the LSU spent ~4 000 cycles per operand tile pair and as
// many per weight-gradient flush, two thirds of the kernel at 8 000 nodes):
//   * operand rows travel global -> shared with cp.async in row-chunk order (a warp-wide copy covers 2 rows x 256 contiguous
//     bytes) straight into the swizzled MN-major tiles; the row owner then reads ITS row back from shared memory
//     (conflict-free) for the tensor-memory A operand and rewrites it only where a scale / SiLU applies;
//   * the weight gradient leaves tensor memory through a [64][65] staging tile and goes out with the lanes along k
//     (128 contiguous bytes per warp-wide reduction for wks = 1);
//   * silu'(Y) of a block whose output gate reads the same rows (dz == Y: node_h stage 1) stays in registers.
template <bool kAttr>
__global__ void __launch_bounds__(256, 1) dense_bwd_tc_rows_kernel(const __grid_constant__ Args a, const AttrBlk ab) {
  constexpr int NT = 256, CG = 2, CPT = kH / CG, NWR = kH * kH / NT;     // 16 weight words per thread and block
#ifdef FEGNN_TRACE
  long long tr_[48];
  for (int i = 0; i < 48; ++i) tr_[i] = 0;
#endif
  TR(0);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
  pdl_trigger();
  VecR* v = reinterpret_cast<VecR*>(smem + SmemR::off_vec);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;

  const int quarter = warp & 3, cg = warp >> 2, row = quarter * 32 + lane, c0 = cg * CPT;
  uint8_t* Wk = smem + SmemR::off_Wk;
  float* FS = reinterpret_cast<float*>(smem + SmemR::off_FS);
  auto Wm = [&](int s_) { return smem + SmemR::off_Wm + s_ * SmemR::kW; };
  auto TY = [&](int s_) { return smem + SmemR::off_TY + s_ * SmemR::kT; };
  auto TX = [&](int s_) { return smem + SmemR::off_TX + s_ * SmemR::kT; };

  // block range of this CTA (blockIdx.y): at a few dozen tiles the SMs left over take a share of the blocks instead of idling
  const int b0 = a.nsplit > 1 ? a.split[blockIdx.y] : 0, b1 = a.nsplit > 1 ? a.split[blockIdx.y + 1] : a.nblk;
  [[maybe_unused]] const bool attr = kAttr && ab.blk >= b0 && ab.blk < b1;     // uniform over the CTA
  [[maybe_unused]] float* sA = reinterpret_cast<float*>(smem + attr_off(SmemR::off_vec + sizeof(VecR)));
  [[maybe_unused]] float* sRed = sA + kTM * kMaxFa;
  [[maybe_unused]] float sa[kMaxFa];
  if constexpr (kAttr) {
#pragma unroll
    for (int f = 0; f < kMaxFa; ++f) sa[f] = 0.f;
    for (int i = t; i < kMaxFa * kH; i += NT) sRed[i] = 0.f;
  }
  float wreg[NWR];
  auto load_w = [&](const Blk& b) {             // every load in flight before anything is stored
#pragma unroll
    for (int j = 0; j < NWR; ++j) {
      const int i = t + j * NT, n = i >> 6, k = i & 63;
      wreg[j] = b.W[(size_t)n * b.ldw + (size_t)k * b.wks];
    }
  };
  auto store_w = [&](const Blk& b, int s_) {
#pragma unroll
    for (int j = 0; j < NWR; ++j) {
      const int i = t + j * NT, n = i >> 6, k = i & 63;
      *reinterpret_cast<float*>(Wm(s_) + mn_off(n, k, kH)) = wreg[j];
      if (b.head) *reinterpret_cast<float*>(Wk + umma::tile_off(n, k, kH)) = wreg[j];
    }
  };
  // ---- prologue (weights only): the first block's weight tile, vectors, barriers, tensor memory
  load_w(a.blk[b0]);
  for (int i = t; i < kH; i += NT) {
    v->cb[0][i] = 0.f; v->cb[1][i] = 0.f; v->cw2[i] = 0.f;
  }
  if (t == 0) {
    v->cb2 = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) umma::mbar_init(&v->bar[i], 1);
    umma::mbar_fence_init();
  }
  if (warp == 0) umma::tmem_alloc<256>(&v->tmem_slot);
  store_w(a.blk[b0], 0);
  umma::fence_smem_to_async();
  umma::fence_before();
  __syncthreads();
  umma::fence_after();
  TR(1);
  pdl_wait();
  TR(2);
  const uint32_t tmem = v->tmem_slot;
  const uint32_t tlane = tmem + ((uint32_t)(quarter * 32) << 16) + c0;
  const uint32_t id_ts_k = idesc_tf32(128, 64, 0, 0), id_ts_mn = idesc_tf32(128, 64, 0, 1), id_wg = idesc_tf32(64, 64, 1, 1);
  const uint64_t dWk = umma::make_desc(umma::smem_u32(Wk));
  uint32_t ph_r = 0, ph_d = 0, ph_w[2] = {0, 0};
  float dmx = 0.f;                 // running max |D| of the block that carries a dmax pointer
  unsigned* dmx_ptr = nullptr;

  // rows r0 .. r0 + 127 of a [N][64] operand (row stride ld) -> an MN-major tile, 16-byte chunks in (row, chunk) order
  auto fetch_tile = [&](uint8_t* dst, const float* src, int ld, int r0) {
#pragma unroll
    for (int j = 0; j < kTM * 16 / NT; ++j) {
      const int i = t + j * NT, rr = i >> 4, c16 = i & 15;
      const bool ok = r0 + rr < a.N;
      cp_async16(dst + mn_chunk_off(rr, c16, kTM), src + (size_t)(ok ? r0 + rr : 0) * ld + 4 * c16, ok ? 16 : 0);
    }
  };
  auto same_y = [&](int b) { return b != b0 && ((a.same_y_mask >> b) & 1u); };      // block b reads the Y tile block b - 1 left
  auto chain = [&](int b) { return b + 1 < b1 && ((a.chain_mask >> b) & 1u); };       // block b + 1 adds to the same D as block b
  // weight gradient of block b (slot s_): wait for its MMAs (which also frees TX[s_] and the Y tile it read)
  auto wait_w = [&](int b, int s_) {
    if (a.blk[b].gW != nullptr) {
      umma::mbar_wait(&v->bar[2 + s_], ph_w[s_]);
      umma::fence_after();
      ph_w[s_] ^= 1;
    }
  };
  // tensor memory -> staging tile (M = 64 layout: row n in lane (n / 16) * 32 + n % 16), then, after a barrier, out with the
  // lanes along k; bias sums
  auto flush_w_stage = [&](int b, int s_) {
    if (a.blk[b].gW != nullptr) {
      float w[CPT];
      tmem_ld<CPT>(tlane + kR_RW + 64 * s_, w);
      if (lane < 16) {
        const int n = quarter * 16 + lane;
#pragma unroll
        for (int j = 0; j < CPT; ++j) FS[n * 65 + c0 + j] = w[j];
      }
      umma::fence_before();
    }
  };
  auto flush_w_out = [&](int b, int s_) {
    const Blk& blk = a.blk[b];
    if (blk.gW != nullptr) {
#pragma unroll
      for (int j = 0; j < kH * kH / NT; ++j) {
        const int i = t + j * NT, n = i >> 6, k = i & 63;
        atomicAdd(blk.gW + (size_t)n * blk.ldw + (size_t)k * blk.wks, FS[n * 65 + k]);
      }
    }
    if (blk.gb != nullptr && t < kH) {
      atomicAdd(blk.gb + t, v->cb[s_][t]);
      v->cb[s_][t] = 0.f;
    }
  };

  const int ntiles = (a.N + kTM - 1) / kTM;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int r0 = tile * kTM, r = r0 + row;
    const bool valid = r < a.N;
    int ys = 0;                                   // Y slot of the current block
    {
      const Blk& f = a.blk[b0];
      fetch_tile(TY(0), f.Y, f.ldy, r0);
      if (!f.head) fetch_tile(TX(0), f.X, f.ldx, r0);
    }
    if (tile != (int)blockIdx.x) {                // a later tile of this CTA: the first block's weights again (slot 0 is free: all flushed)
      load_w(a.blk[b0]);
      store_w(a.blk[b0], 0);
    }
    float dsil[CPT];                              // silu'(Y row) of a block with dz == Y
    for (int b = b0; b < b1; ++b) {
      const Blk& blk = a.blk[b];
      const int s_ = (b - b0) & 1;
      const bool new_y = !same_y(b);
#ifdef FEGNN_TRACE
      const int tb_ = 3 + 9 * (b - b0);
#endif
      TR(tb_);
      if (new_y && b != b0) ys ^= 1;
      cp_async_wait();
      __syncthreads();                            // this block's rows have landed (every thread's copies)
      float xr[CPT], yr[CPT];
      const bool dz_y = new_y && blk.dz != nullptr && blk.dz == blk.Y && blk.ysilu && blk.yscale == nullptr && blk.ldy == kH;
      // ---- Y rows: scale / SiLU in place (row owner)
      if (new_y && (blk.yscale != nullptr || blk.ysilu)) {
        mn_load_row<CPT>(TY(ys), row, cg, yr);
        const float sc = (valid && blk.yscale != nullptr) ? blk.yscale[r] : 1.f;
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
          yr[j] *= sc;
          if (blk.ysilu) {
            float av, d;
            silu_grad_f(yr[j], av, d);
            yr[j] = valid ? av : 0.f;
            dsil[j] = d;
          }
        }
        mn_store_row<CPT>(TY(ys), row, cg, yr);
      }
      const bool more = b + 1 < b1;
      if (blk.head) {
        // z = Y W^T on the tensor core, X = gs w2 silu'(z + b)
        if (t < kH) { v->hb[t] = blk.hb[t]; v->hw2[t] = blk.hw2[t]; }
        mn_load_row<CPT>(TY(ys), row, cg, yr);
        tmem_st<CPT>(tlane + kR_OPA, yr);
        tmem_st_wait();
        umma::fence_smem_to_async();
        umma::fence_before();
        __syncthreads();
        if (warp == 0) {
          umma::fence_after();
          if (umma::elect_one()) {
            // into this slot's weight-gradient columns (free: block b - 2 was flushed) -- the data-gradient accumulator
            // may hold the running sum of a chain
            gemm_ts_kmajor(tmem + kR_RW + 64 * s_, tmem + kR_OPA, dWk, id_ts_k);
            umma::commit(&v->bar[0]);
          }
          __syncwarp();
        }
        umma::mbar_wait(&v->bar[0], ph_r);
        umma::fence_after();
        ph_r ^= 1;
        TR(tb_ + 1);
        tmem_ld<CPT>(tlane + kR_RW + 64 * s_, xr);
        const float g = valid ? blk.gs[r] : 0.f;
        float aw[CPT];
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
          float av, d;
          silu_grad_f(xr[j] + v->hb[c0 + j], av, d);
          aw[j] = g * av;
          xr[j] = g * v->hw2[c0 + j] * d;
        }
        {
          static_assert(CPT == 32, "one 32-column transposed reduction per warp");
          const float tot = warp_colsum32(aw, lane);          // 31 shuffles (a butterfly per column: 160)
          atomicAdd(&v->cw2[c0 + lane], tot);
        }
        if (cg == 0) {
          float sum = g;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
          if (lane == 0) atomicAdd(&v->cb2, sum);
        }
        umma::fence_before();
        mn_store_row<CPT>(TX(s_), row, cg, xr);
      } else {
        mn_load_row<CPT>(TX(s_), row, cg, xr);
        if (blk.xscale != nullptr) {
          const float sc = valid ? blk.xscale[r] : 0.f;
#pragma unroll
          for (int j = 0; j < CPT; ++j) xr[j] *= sc;
          mn_store_row<CPT>(TX(s_), row, cg, xr);
        }
      }
      // ---- X row -> A operand (tensor memory); the data gradient of block b - 1 has left the A operand
      tmem_st<CPT>(tlane + kR_OPA, xr);
      if constexpr (kAttr) {
        if (b == ab.blk) attr_load_tile(sA, ab.at, r0, min(kTM, a.N - r0), NT);
      }
      tmem_st_wait();
      TR(tb_ + 2);
      if (more) load_w(a.blk[b + 1]);             // lands under the MMAs / epilogue of this block
      umma::fence_smem_to_async();
      umma::fence_before();
      __syncthreads();
      TR(tb_ + 3);
      const bool acc_in = b > b0 && chain(b - 1);
      if (warp == 0) {
        umma::fence_after();
        if (umma::elect_one()) {
          const uint64_t dWm = make_desc_mn(umma::smem_u32(Wm(s_)), kH * 128);
          if (blk.dmode != 0) gemm_ts_mn_acc(tmem + kR_ACC, tmem + kR_OPA, dWm, id_ts_mn, acc_in);      // D (+)= X W
          umma::commit(&v->bar[1]);
          if (blk.gW != nullptr) {
            const uint64_t dTX = make_desc_mn(umma::smem_u32(TX(s_)), kTM * 128), dTY = make_desc_mn(umma::smem_u32(TY(ys)), kTM * 128);
#pragma unroll
            for (int ks = 0; ks < 16; ++ks)                                   // dW = X^T Y over the 128 rows
              umma::mma_tf32(tmem + kR_RW + 64 * s_, desc_advance(dTX, ks * 1024), desc_advance(dTY, ks * 1024), id_wg, ks > 0 ? 1u : 0u);
            umma::commit(&v->bar[2 + s_]);
          }
        }
        __syncwarp();
      }
      TR(tb_ + 4);
      // ---- under the MMAs: the weight gradient of block b - 1 has finished -> its X / Y tiles are free: the rows of block
      //      b + 1 go in flight; flush of block b - 1; bias column sums of this block
      if (b > b0) wait_w(b - 1, s_ ^ 1);
      if (more) {
        const Blk& nx = a.blk[b + 1];
        if (!same_y(b + 1)) fetch_tile(TY(ys ^ 1), nx.Y, nx.ldy, r0);
        if (!nx.head) fetch_tile(TX(s_ ^ 1), nx.X, nx.ldx, r0);
      }
      if (b > b0) flush_w_stage(b - 1, s_ ^ 1);
      if (blk.gb != nullptr) {
        const int col = t & 63, part = t >> 6;
        float sum = 0.f;
#pragma unroll 8
        for (int rr = part * 32; rr < part * 32 + 32; ++rr) sum += *reinterpret_cast<const float*>(TX(s_) + mn_off(rr, col, kTM));
        atomicAdd(&v->cb[s_][col], sum);
      }
      if constexpr (kAttr) {
        if (b == ab.blk)
          attr_wgrad_walk(sa, sA, ab.at.Fa, [&](int rr, int c) { return *reinterpret_cast<const float*>(TX(s_) + mn_off(rr, c, kTM)); });
      }
      TR(tb_ + 5);
      if (b > b0) {
        __syncthreads();                           // staging tile complete
        flush_w_out(b - 1, s_ ^ 1);
      }
      TR(tb_ + 6);
      // ---- the data gradient: wait (the A operand and, at the end of a chain, the accumulator are reused next)
      umma::mbar_wait(&v->bar[1], ph_d);
      umma::fence_after();
      ph_d ^= 1;
      TR(tb_ + 7);
      if (blk.dmode != 0 && !chain(b)) {
        float d[CPT];
        tmem_ld<CPT>(tlane + kR_ACC, d);
        if (valid) {
          if (dz_y) {
#pragma unroll
            for (int j = 0; j < CPT; ++j) d[j] *= dsil[j];
          } else if (blk.dz != nullptr) {
            const float4* zr = reinterpret_cast<const float4*>(blk.dz + (size_t)r * kH + c0);
#pragma unroll
            for (int ch = 0; ch < CPT / 4; ++ch) {
              const float4 z = zr[ch];
              float av, e0, e1, e2, e3;
              silu_grad_f(z.x, av, e0); silu_grad_f(z.y, av, e1); silu_grad_f(z.z, av, e2); silu_grad_f(z.w, av, e3);
              d[ch * 4] *= e0; d[ch * 4 + 1] *= e1; d[ch * 4 + 2] *= e2; d[ch * 4 + 3] *= e3;
            }
          }
          const float sc = blk.dscale != nullptr ? blk.dscale[r] : 1.f;
          float4* dst = reinterpret_cast<float4*>(blk.D + (size_t)r * blk.ldd + c0);
          if (blk.dmax != nullptr) {
#pragma unroll
            for (int j = 0; j < CPT; ++j) dmx = fmaxf(dmx, fabsf(d[j] * sc));
          }
#pragma unroll
          for (int ch = 0; ch < CPT / 4; ++ch) {
            const float4 q = make_float4(d[ch * 4] * sc, d[ch * 4 + 1] * sc, d[ch * 4 + 2] * sc, d[ch * 4 + 3] * sc);
            if (blk.dmode == 2) atomicAdd(dst + ch, q);
            else dst[ch] = q;
          }
        }
      }
      if (blk.dmax != nullptr) dmx_ptr = blk.dmax;
      TR(tb_ + 8);
      if (more) store_w(a.blk[b + 1], s_ ^ 1);     // Wm[s_ ^ 1]: last read by the data gradient of block b - 1 (waited)
      umma::fence_before();
      if (blk.head) {
        __syncthreads();                           // cw2 / cb2 complete
        if (t < kH) {
          if (blk.g_hw2 != nullptr) atomicAdd(blk.g_hw2 + t, v->cw2[t]);
          v->cw2[t] = 0.f;
        }
        if (t == 0) {
          if (blk.g_hb2 != nullptr) atomicAdd(blk.g_hb2, v->cb2);
          v->cb2 = 0.f;
        }
      }
    }
    TR(45);
    {
      const int bl = b1 - 1, sl = (b1 - 1 - b0) & 1;
      wait_w(bl, sl);
      flush_w_stage(bl, sl);
      __syncthreads();                             // staging tile and the bias sums of the last block are complete
      flush_w_out(bl, sl);
      __syncthreads();
    }
    TR(46);
  }
  if (dmx_ptr != nullptr) {                       // uniform over the CTA (the block list is)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dmx = fmaxf(dmx, __shfl_xor_sync(0xffffffffu, dmx, o));
    if (lane == 0) atomicMax(dmx_ptr, __float_as_uint(dmx));
  }
  if constexpr (kAttr) {
    if (attr) attr_wgrad_flush(sa, sRed, ab.at);
  }
  umma::fence_before();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc<256>(tmem);
  TR(47);
#ifdef FEGNN_TRACE
  if (threadIdx.x == 0 && blockIdx.x == 1 && blockIdx.y == 0) {
    printf("DTRACE nblk=%d b0=%d b1=%d head0=%d :", a.nblk, b0, b1, a.blk[b0].head);
    for (int i = 1; i < 48; ++i) if (tr_[i]) printf(" %d:%lld", i, tr_[i] - tr_[0]);
    printf("\n");
  }
#endif
}
#undef TR

}  // namespace dtc

static inline int dense_rows_max_tiles_per_sm() {
  static const int v = getenv("FEGNN_DENSE_ROWS_MAX_TILES_PER_SM") ? atoi(getenv("FEGNN_DENSE_ROWS_MAX_TILES_PER_SM"))
                                                                    : dtc::kRowsMaxTilesPerSm;      // experiment switch
  return v;
}
// true when launch_dense_bwd_tc takes the per-tile kernel (the one that honours Blk::dmax)
inline bool dense_bwd_uses_rows(int N, int sms) {
  const int ntiles = (N + kTM - 1) / kTM;
  return (long long)ntiles <= (long long)dense_rows_max_tiles_per_sm() * sms;
}

// ab != nullptr: the attribute instantiation (block ab->blk adds dU1att)
cudaError_t launch_dense_bwd_tc(const dtc::Args& a_in, int sms, cudaStream_t st, const dtc::AttrBlk* ab = nullptr) {
  dtc::Args a = a_in;
  a.nsplit = 1;
  a.same_y_mask = a.chain_mask = 0;
  for (int b = 1; b < a.nblk; ++b) {
    const dtc::Blk &p = a.blk[b - 1], &q = a.blk[b];
    if (p.Y == q.Y && p.ldy == q.ldy && p.yscale == q.yscale && p.ysilu == q.ysilu) a.same_y_mask |= 1u << b;
    if (p.dmode == 2 && q.dmode == 2 && p.D == q.D && p.ldd == q.ldd && p.dz == q.dz && p.dscale == q.dscale)
      a.chain_mask |= 1u << (b - 1);
  }
  static DevOnce attr;
  if (!attr.get()) {
    cudaError_t e = cudaFuncSetAttribute(dtc::dense_bwd_tc_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)dtc::Smem::bytes);
    if (e != cudaSuccess) return e;
    attr.set();
  }
  const int ntiles = (a.N + kTM - 1) / kTM;
  if (ntiles == 0 || a.nblk == 0) return cudaSuccess;
  if (dense_bwd_uses_rows(a.N, sms)) {   // small graphs: one CTA per node tile walks the blocks
    static DevOnce attr2;
    if (!attr2.get()) {
      cudaError_t e = cudaFuncSetAttribute(dtc::dense_bwd_tc_rows_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)dtc::SmemR::bytes);
      if (e != cudaSuccess) return e;
      attr2.set();
    }
    // Fewer tiles than SMs: cut the block list into ranges of about equal cost (a head block counts twice: it has the
    // recompute round in front of its data gradient) and launch one CTA per (tile, range).  Ranges that add into the same D do
    // so with red.add, exactly as consecutive chains of one CTA do.
    int nsplit = ntiles < sms ? sms / ntiles : 1;
    if (nsplit > a.nblk) nsplit = a.nblk;
    if (const char* e = getenv("FEGNN_DENSE_SPLIT")) { const int v_ = atoi(e); if (v_ >= 1 && v_ <= a.nblk) nsplit = v_; }
    if (nsplit > 1) {
      int cost[dtc::kMaxBlk], total = 0;
      for (int b = 0; b < a.nblk; ++b) { cost[b] = a.blk[b].head ? 2 : 1; total += cost[b]; }
      int s_ = 0, acc = 0;
      a.split[0] = 0;
      for (int b = 0; b < a.nblk && s_ + 1 < nsplit; ++b) {
        acc += cost[b];
        // close range s_ after block b once it holds its share, keeping one block for every later range
        if (acc * nsplit >= total * (s_ + 1) || a.nblk - (b + 1) == nsplit - (s_ + 1)) a.split[++s_] = b + 1;
      }
      while (s_ < nsplit) a.split[++s_] = a.nblk;
      a.nsplit = nsplit;
    }
    const dim3 grid(ntiles < sms ? ntiles : sms, a.nsplit);
    if (ab != nullptr) {
      const size_t bytes = dtc::attr_off(dtc::SmemR::bytes) + kAttrGBytes;
      static DevOnce attr3;
      if (!attr3.get()) {
        cudaError_t e = cudaFuncSetAttribute(dtc::dense_bwd_tc_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) return e;
        attr3.set();
      }
      if (cudaError_t e_ = launch_pdl(dtc::dense_bwd_tc_rows_kernel<true>, grid, dim3(256), bytes, st, a, *ab)) return e_;
      return cudaGetLastError();
    }
    if (cudaError_t e_ = launch_pdl(dtc::dense_bwd_tc_rows_kernel<false>, grid, dim3(256), dtc::SmemR::bytes, st, a, dtc::AttrBlk{})) return e_;
    return cudaGetLastError();
  }
  int per = (2 * sms) / a.nblk;                   // CTAs per block at 2 CTAs / SM
  per = per < 1 ? 1 : (per > ntiles ? ntiles : per);
  if (ab != nullptr) {
    const size_t bytes = dtc::attr_off(dtc::Smem::bytes) + kAttrGBytes;
    static DevOnce attr4;
    if (!attr4.get()) {
      cudaError_t e = cudaFuncSetAttribute(dtc::dense_bwd_tc_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
      if (e != cudaSuccess) return e;
      attr4.set();
    }
    if (cudaError_t e_ = launch_pdl(dtc::dense_bwd_tc_kernel<2, true>, per * a.nblk, 256, bytes, st, a, *ab)) return e_;
    return cudaGetLastError();
  }
  if (cudaError_t e_ = launch_pdl(dtc::dense_bwd_tc_kernel<2, false>, per * a.nblk, 256, dtc::Smem::bytes, st, a, dtc::AttrBlk{})) return e_;
  return cudaGetLastError();
}

}  // namespace fegnn
