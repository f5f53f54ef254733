// input_grads.cu -- gradients to the data inputs node_vel and node_attr (include/fegnn.h, fegnn_input_grads).
//
// Both are per-node terms of one layer that the backward already has in HBM when it asks for them, so each is one small
// pass over that layer's buffers, launched only when the caller requests the gradient; the layer kernels of the default
// backward are not touched.  (dL/d edge_attr needs gz1, which the fused edge backward never writes out: it is computed
// there, edge_kernels.cu / edge_tc_bwd4.cu, kEa.)
#pragma once
#include "common.cuh"

namespace fegnn {

// node_vel: the layer adds phi_v(h_i) v_i to the coordinates (models/FastEGNN.py:142), so dL/dv_i += sv_i g_i with g_i the
// gradient of the layer's output coordinates -- gx_new[i] plus, through the next layer's centroid, gxsum_next[batch[i]]:
// the same g the virtual backward forms for gsv.  One thread per (node, component); one owner per element.
__global__ void input_grad_vel_kernel(int N, const float* __restrict__ sv, const float* __restrict__ gx_new,
                                      const float* __restrict__ gxsum_next, const int* __restrict__ batch,
                                      float* __restrict__ gv) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * 3) return;
  const int i = idx / 3, k = idx - i * 3;
  float g = gx_new[idx];
  if (gxsum_next != nullptr) g += gxsum_next[batch[i] * 3 + k];
  gv[idx] += sv[i] * g;
}

// node_attr: Uh_i = U1h h_i + e1 + U1att a_i (node_pre), so dL/da_i += gUh_i U1att, a [64] x [64, Fa] product per row.
// U1att is staged transposed ([k][f], consecutive f in consecutive banks); one thread per (node, attribute).
constexpr int kGaThreads = 256;
__global__ void __launch_bounds__(kGaThreads) input_grad_attr_kernel(int N, int Fa, int ldn, const float* __restrict__ w,
                                                                     const float* __restrict__ gUh, float* __restrict__ ga) {
  __shared__ float sW[kH * FEGNN_MAX_FA];
  for (int i = threadIdx.x; i < kH * Fa; i += kGaThreads) {
    const int k = i / Fa, f = i - k * Fa;
    sW[i] = w[(size_t)k * ldn + f];
  }
  __syncthreads();
  const size_t idx = (size_t)blockIdx.x * kGaThreads + threadIdx.x;
  if (idx >= (size_t)N * Fa) return;
  const int i = (int)(idx / Fa), f = (int)(idx - (size_t)i * Fa);
  const float4* g = reinterpret_cast<const float4*>(gUh + (size_t)i * kH);
  float s = 0.f;
#pragma unroll 4
  for (int k4 = 0; k4 < kH / 4; ++k4) {
    const float4 v = g[k4];
    s = fmaf(v.x, sW[(4 * k4 + 0) * Fa + f], s);
    s = fmaf(v.y, sW[(4 * k4 + 1) * Fa + f], s);
    s = fmaf(v.z, sW[(4 * k4 + 2) * Fa + f], s);
    s = fmaf(v.w, sW[(4 * k4 + 3) * Fa + f], s);
  }
  ga[idx] += s;
}

// Edge lengths of a graph built from positions x (fegnn_edge_length_backward): edge_attr[e, k] = len_e for every k, with
// len_e = |x_row - x_col| the graph's own edge_attr[e, 0] (radius_graph.cu: __fsqrt_rn of the no-FMA d2), so
//   g_x[row_e] += u_e,  g_x[col_e] -= u_e,  u_e = (sum_k g_ea[e, k]) (x_row - x_col) / len_e,  u_e = 0 where len_e == 0
// (coincident distinct nodes: torch's norm subgradient).  One warp per CSR row over rowptr, lanes over its edges: the row
// side is summed in registers and added once per row, the col side with red.global.add per edge.  Persistent grid; kLive
// bounds every row by the live edge count (read after the wait, as live_edges() does), so no edge at or past it is read.
constexpr int kElThreads = 256;
template <bool kLive>
__global__ void __launch_bounds__(kElThreads) edge_length_bwd_kernel(int N, int E, int Fe, const int* __restrict__ rowptr,
                                                                     const int* __restrict__ col, const float* __restrict__ ea,
                                                                     const float* __restrict__ x, const float* __restrict__ g_ea,
                                                                     const int* __restrict__ n_edges, float* __restrict__ g_x) {
  pdl_trigger();
  pdl_wait();
  if constexpr (kLive) {
    const int n = __ldcg(n_edges);
    E = n < 0 ? 0 : (n > E ? E : n);
  }
  const int lane = threadIdx.x & 31;
  const int warps = gridDim.x * (kElThreads / 32);
  for (int i = blockIdx.x * (kElThreads / 32) + (threadIdx.x >> 5); i < N; i += warps) {
    const int e0 = min(rowptr[i], E), e1 = min(rowptr[i + 1], E);
    if (e0 >= e1) continue;
    const float xi0 = x[3 * i], xi1 = x[3 * i + 1], xi2 = x[3 * i + 2];
    float r0 = 0.f, r1 = 0.f, r2 = 0.f;
    for (int e = e0 + lane; e < e1; e += 32) {
      const float len = ea[(size_t)e * Fe];
      if (len == 0.f) continue;
      float s = 0.f;
      for (int k = 0; k < Fe; ++k) s += g_ea[(size_t)e * Fe + k];
      const int j = col[e];
      const float f = s / len;
      const float u0 = f * (xi0 - x[3 * j]), u1 = f * (xi1 - x[3 * j + 1]), u2 = f * (xi2 - x[3 * j + 2]);
      r0 += u0; r1 += u1; r2 += u2;
      atomicAdd(g_x + 3 * j, -u0);
      atomicAdd(g_x + 3 * j + 1, -u1);
      atomicAdd(g_x + 3 * j + 2, -u2);
    }
    r0 = warpsum(r0); r1 = warpsum(r1); r2 = warpsum(r2);
    if (lane == 0) {
      atomicAdd(g_x + 3 * i, r0);          // other rows' col terms land on this row too
      atomicAdd(g_x + 3 * i + 1, r1);
      atomicAdd(g_x + 3 * i + 2, r2);
    }
  }
}

inline cudaError_t launch_edge_length_bwd(int N, int E, int Fe, const int* rowptr, const int* col, const float* ea,
                                          const float* x, const float* g_ea, const int* n_edges, float* g_x, int sms,
                                          cudaStream_t st) {
  if (N == 0 || E == 0) return cudaSuccess;
  const int rows_per_cta = kElThreads / 32;
  const int grid = min(4 * sms, (N + rows_per_cta - 1) / rows_per_cta);
  cudaError_t e = n_edges != nullptr
      ? launch_pdl(edge_length_bwd_kernel<true>, grid, kElThreads, 0, st, N, E, Fe, rowptr, col, ea, x, g_ea, n_edges, g_x)
      : launch_pdl(edge_length_bwd_kernel<false>, grid, kElThreads, 0, st, N, E, Fe, rowptr, col, ea, x, g_ea, n_edges, g_x);
  if (e != cudaSuccess) return e;
  return cudaGetLastError();
}

inline cudaError_t launch_input_grad_vel(int N, const float* sv, const float* gx_new, const float* gxsum_next,
                                         const int* batch, float* gv, cudaStream_t st) {
  if (N == 0) return cudaSuccess;
  input_grad_vel_kernel<<<(unsigned)((N * 3 + 255) / 256), 256, 0, st>>>(N, sv, gx_new, gxsum_next, batch, gv); ++g_launches;
  return cudaGetLastError();
}
// w = node_w0 + (first attribute column), row stride ldn
inline cudaError_t launch_input_grad_attr(int N, int Fa, int ldn, const float* w, const float* gUh, float* ga, cudaStream_t st) {
  const size_t n = (size_t)N * Fa;
  if (n == 0) return cudaSuccess;
  input_grad_attr_kernel<<<(unsigned)((n + kGaThreads - 1) / kGaThreads), kGaThreads, 0, st>>>(N, Fa, ldn, w, gUh, ga); ++g_launches;
  return cudaGetLastError();
}

}  // namespace fegnn
