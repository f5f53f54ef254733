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
