// mmd.cu -- MMD regulariser between sampled real coordinates and virtual coordinates.
//
// Replaces utils/train.py:17-20 (Laplacian kernel on the plain L2 distance) and the
// per-graph Python loop / boolean masking of :111-165.  The random sample is an input
// (global node indices), so torch.randperm stays the caller's RNG.
//   loss = 1/(B C^2) sum_b sum_{c,c'} k(Z_bc, Z_bc') - 2/(B ns C) sum_b sum_{s,c} k(x_s, Z_bc)
//   k(p,q) = exp(-|p-q| / (2 sigma^2)),  d|p-q|/dp = 0 at p == q (torch.cdist convention).
#include "common.cuh"

namespace fegnn {

__global__ void __launch_bounds__(128) mmd_fwd_kernel(int B, int C, int ns, float inv2s2, float svv, float srv, const float* __restrict__ x,
                                                      const float* __restrict__ Z, const int* __restrict__ idx,
                                                      float* __restrict__ loss) {
  const int b = blockIdx.x;
  const float cvv = svv / ((float)B * C * C), crv = ns > 0 ? srv * 2.f / ((float)B * ns * C) : 0.f;
  float acc = 0.f;
  for (int p = threadIdx.x; p < C * C + ns * C; p += blockDim.x) {
    float px, py, pz, w;
    int c;
    if (p < C * C) {
      const int c0 = p / C;
      c = p - c0 * C;
      px = Z[((size_t)b * 3 + 0) * C + c0]; py = Z[((size_t)b * 3 + 1) * C + c0]; pz = Z[((size_t)b * 3 + 2) * C + c0];
      w = cvv;
    } else {
      const int q = p - C * C, s = q / C;
      c = q - s * C;
      const int i = idx[(size_t)b * ns + s];
      px = x[(size_t)i * 3 + 0]; py = x[(size_t)i * 3 + 1]; pz = x[(size_t)i * 3 + 2];
      w = -crv;
    }
    const float dx = px - Z[((size_t)b * 3 + 0) * C + c], dy = py - Z[((size_t)b * 3 + 1) * C + c],
                dz = pz - Z[((size_t)b * 3 + 2) * C + c];
    acc += w * __expf(-sqrtf(dx * dx + dy * dy + dz * dz) * inv2s2);
  }
  acc = warpsum(acc);
  if ((threadIdx.x & 31) == 0) atomicAdd(loss, acc);
}

__global__ void __launch_bounds__(128) mmd_bwd_kernel(int B, int C, int ns, float inv2s2, float svv, float srv, const float* __restrict__ x,
                                                      const float* __restrict__ Z, const int* __restrict__ idx,
                                                      const float* __restrict__ gloss, float* __restrict__ gx,
                                                      float* __restrict__ gZ) {
  __shared__ float gz[3 * FEGNN_MAX_C];
  const int b = blockIdx.x;
  const float gl = gloss[0];
  const float cvv = svv * gl / ((float)B * C * C), crv = ns > 0 ? srv * 2.f * gl / ((float)B * ns * C) : 0.f;
  if (threadIdx.x < 3 * C) gz[threadIdx.x] = 0.f;
  __syncthreads();
  for (int p = threadIdx.x; p < C * C + ns * C; p += blockDim.x) {
    float px, py, pz, w;
    int c, c0 = -1, i = -1;
    if (p < C * C) {
      c0 = p / C;
      c = p - c0 * C;
      px = Z[((size_t)b * 3 + 0) * C + c0]; py = Z[((size_t)b * 3 + 1) * C + c0]; pz = Z[((size_t)b * 3 + 2) * C + c0];
      w = cvv;
    } else {
      const int q = p - C * C, s = q / C;
      c = q - s * C;
      i = idx[(size_t)b * ns + s];
      px = x[(size_t)i * 3 + 0]; py = x[(size_t)i * 3 + 1]; pz = x[(size_t)i * 3 + 2];
      w = -crv;
    }
    const float dx = px - Z[((size_t)b * 3 + 0) * C + c], dy = py - Z[((size_t)b * 3 + 1) * C + c],
                dz = pz - Z[((size_t)b * 3 + 2) * C + c];
    const float dist = sqrtf(dx * dx + dy * dy + dz * dz);
    if (dist > 0.f) {
      // d/dp of w*exp(-dist*inv2s2) = -w*inv2s2*k * (p-q)/dist ; d/dq is the negative
      const float f = -w * inv2s2 * __expf(-dist * inv2s2) / dist;
      const float fx = f * dx, fy = f * dy, fz = f * dz;
      atomicAdd(&gz[0 * C + c], -fx); atomicAdd(&gz[1 * C + c], -fy); atomicAdd(&gz[2 * C + c], -fz);
      if (c0 >= 0) {
        atomicAdd(&gz[0 * C + c0], fx); atomicAdd(&gz[1 * C + c0], fy); atomicAdd(&gz[2 * C + c0], fz);
      } else {
        atomicAdd(gx + (size_t)i * 3 + 0, fx); atomicAdd(gx + (size_t)i * 3 + 1, fy);
        atomicAdd(gx + (size_t)i * 3 + 2, fz);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < 3 * C) gZ[(size_t)b * 3 * C + threadIdx.x] = gz[threadIdx.x];
}

// ------------------------------------------------------------------ the step's loss in one kernel per direction
// utils/train.py:104,163: loss = MSE(x, target) + weight * (l_vv - l_rv).  As torch ops around mmd_loss this was ten small
// kernels between the last forward kernel and the first backward kernel (reduce, mul, add, their backward, the fills), none
// overlapping another.  Here: CTAs [0, B) evaluate the MMD term of one graph each, the remaining CTAs sum (x - target)^2.
//   out[0] = total, out[1] = the MSE term alone (what the reference logs at :107), both zeroed by the launcher.
__global__ void __launch_bounds__(128) mse_mmd_fwd_kernel(int N, int B, int C, int ns, float inv2s2, float weight, float svv,
                                                          float srv, float inv_count, const float* __restrict__ x,
                                                          const float* __restrict__ target, const float* __restrict__ Z,
                                                          const int* __restrict__ idx, float* __restrict__ out_total,
                                                          float* __restrict__ out_mse) {
  if ((int)blockIdx.x < B) {
    const int b = blockIdx.x;
    const float cvv = svv / ((float)B * C * C), crv = ns > 0 ? srv * 2.f / ((float)B * ns * C) : 0.f;
    float acc = 0.f;
    for (int p = threadIdx.x; p < C * C + ns * C; p += blockDim.x) {
      float px, py, pz, w;
      int c;
      if (p < C * C) {
        const int c0 = p / C;
        c = p - c0 * C;
        px = Z[((size_t)b * 3 + 0) * C + c0]; py = Z[((size_t)b * 3 + 1) * C + c0]; pz = Z[((size_t)b * 3 + 2) * C + c0];
        w = cvv;
      } else {
        const int q = p - C * C, s = q / C;
        c = q - s * C;
        const int i = idx[(size_t)b * ns + s];
        px = x[(size_t)i * 3 + 0]; py = x[(size_t)i * 3 + 1]; pz = x[(size_t)i * 3 + 2];
        w = -crv;
      }
      const float dx = px - Z[((size_t)b * 3 + 0) * C + c], dy = py - Z[((size_t)b * 3 + 1) * C + c],
                  dz = pz - Z[((size_t)b * 3 + 2) * C + c];
      acc += w * __expf(-sqrtf(dx * dx + dy * dy + dz * dz) * inv2s2);
    }
    acc = warpsum(acc);
    if ((threadIdx.x & 31) == 0) atomicAdd(out_total, weight * acc);
    return;
  }
  const size_t n = (size_t)N * 3, stride = (size_t)(gridDim.x - B) * blockDim.x;
  float acc = 0.f;
  for (size_t i = (size_t)(blockIdx.x - B) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float d = x[i] - target[i];
    acc = fmaf(d, d, acc);
  }
  acc = warpsum(acc) * inv_count;
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(out_total, acc);
    atomicAdd(out_mse, acc);
  }
}

// gx = (g_total + g_mse) * 2 inv_count (x - target) + g_total * weight * d(MMD)/dx ; gZ = g_total * weight * d(MMD)/dZ.
// Everything that lands in gx is an atomicAdd onto the launcher's zero fill (the MMD term touches the sampled nodes only).
__global__ void __launch_bounds__(128) mse_mmd_bwd_kernel(int N, int B, int C, int ns, float inv2s2, float weight, float svv,
                                                          float srv, float inv_count, const float* __restrict__ x,
                                                          const float* __restrict__ target, const float* __restrict__ Z,
                                                          const int* __restrict__ idx, const float* __restrict__ g_total,
                                                          const float* __restrict__ g_mse, float* __restrict__ gx,
                                                          float* __restrict__ gZ) {
  __shared__ float gz[3 * FEGNN_MAX_C];
  const float gt = g_total != nullptr ? g_total[0] : 0.f, gm = g_mse != nullptr ? g_mse[0] : 0.f;
  if ((int)blockIdx.x < B) {
    const int b = blockIdx.x;
    const float gl = gt * weight;
    const float cvv = svv * gl / ((float)B * C * C), crv = ns > 0 ? srv * 2.f * gl / ((float)B * ns * C) : 0.f;
    if (threadIdx.x < 3 * C) gz[threadIdx.x] = 0.f;
    __syncthreads();
    for (int p = threadIdx.x; p < C * C + ns * C; p += blockDim.x) {
      float px, py, pz, w;
      int c, c0 = -1, i = -1;
      if (p < C * C) {
        c0 = p / C;
        c = p - c0 * C;
        px = Z[((size_t)b * 3 + 0) * C + c0]; py = Z[((size_t)b * 3 + 1) * C + c0]; pz = Z[((size_t)b * 3 + 2) * C + c0];
        w = cvv;
      } else {
        const int q = p - C * C, s = q / C;
        c = q - s * C;
        i = idx[(size_t)b * ns + s];
        px = x[(size_t)i * 3 + 0]; py = x[(size_t)i * 3 + 1]; pz = x[(size_t)i * 3 + 2];
        w = -crv;
      }
      const float dx = px - Z[((size_t)b * 3 + 0) * C + c], dy = py - Z[((size_t)b * 3 + 1) * C + c],
                  dz = pz - Z[((size_t)b * 3 + 2) * C + c];
      const float dist = sqrtf(dx * dx + dy * dy + dz * dz);
      if (dist > 0.f) {
        const float f = -w * inv2s2 * __expf(-dist * inv2s2) / dist;
        const float fx = f * dx, fy = f * dy, fz = f * dz;
        atomicAdd(&gz[0 * C + c], -fx); atomicAdd(&gz[1 * C + c], -fy); atomicAdd(&gz[2 * C + c], -fz);
        if (c0 >= 0) {
          atomicAdd(&gz[0 * C + c0], fx); atomicAdd(&gz[1 * C + c0], fy); atomicAdd(&gz[2 * C + c0], fz);
        } else {
          atomicAdd(gx + (size_t)i * 3 + 0, fx); atomicAdd(gx + (size_t)i * 3 + 1, fy);
          atomicAdd(gx + (size_t)i * 3 + 2, fz);
        }
      }
    }
    __syncthreads();
    if (threadIdx.x < 3 * C) gZ[(size_t)b * 3 * C + threadIdx.x] = gz[threadIdx.x];
    return;
  }
  const size_t n = (size_t)N * 3, stride = (size_t)(gridDim.x - B) * blockDim.x;
  const float k = (gt + gm) * 2.f * inv_count;
  for (size_t i = (size_t)(blockIdx.x - B) * blockDim.x + threadIdx.x; i < n; i += stride)
    atomicAdd(gx + i, k * (x[i] - target[i]));
}

// ------------------------------------------------------------------ deterministic forms (fegnn_set_mode("deterministic", 1))
// The kernels above add per-warp partials into one word and scatter the gradient terms of each pair with atomics, so the
// last bits depend on the order in which warps arrive.  The forms below fix every summation order; each term is the same
// expression as above.
//   forward: per-CTA partials in a fixed order, stored in the caller's workspace and added in CTA order by the last CTA
//            (below); the grid depends on N and B only.
//   backward: the MSE term is a plain store (one term per element); then one CTA per graph gathers, per virtual channel, the
//            gradient of every pair it takes part in (lanes strided over the pairs, shuffle tree), and per sampled node the
//            C terms in channel order, added onto the MSE term with one atomic per node.  That atomic is order-free when
//            no node index is sampled by two graphs (each graph samples its own nodes); a node sampled twice within one
//            graph gets the same value twice, which is order-free too.

// gradient of w * exp(-|p - q| inv2s2) with respect to p; 0 at p == q (torch.cdist's convention)
__device__ __forceinline__ float3 mmd_pair_grad(float3 p, float3 q, float w, float inv2s2) {
  const float dx = p.x - q.x, dy = p.y - q.y, dz = p.z - q.z;
  const float dist = sqrtf(dx * dx + dy * dy + dz * dz);
  if (!(dist > 0.f)) return make_float3(0.f, 0.f, 0.f);
  const float f = -w * inv2s2 * __expf(-dist * inv2s2) / dist;
  return make_float3(f * dx, f * dy, f * dz);
}
__device__ __forceinline__ float3 ld_z(const float* __restrict__ Z, int b, int C, int c) {
  return make_float3(Z[((size_t)b * 3 + 0) * C + c], Z[((size_t)b * 3 + 1) * C + c], Z[((size_t)b * 3 + 2) * C + c]);
}
__device__ __forceinline__ float3 ld_x(const float* __restrict__ x, int i) {
  return make_float3(x[(size_t)i * 3 + 0], x[(size_t)i * 3 + 1], x[(size_t)i * 3 + 2]);
}

// Forward: the grid of the default kernel (CTAs [0, B) one graph each, then mse_ctas(N) CTAs striding over the MSE
// operands; a function of N and B only).  Each CTA sums its terms per thread in index order, reduces them with a fixed
// shuffle tree, adds its warp partials in warp order and stores the result in its own slot of the caller's workspace.
// The last CTA to finish (ticket counter in the workspace) adds the slots in CTA order.
__device__ __forceinline__ float block_sum_ordered(float v, float* red /* [blockDim / 32] */) {
  v = warpsum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
  if (threadIdx.x == 0)
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) t += red[k];
  __syncthreads();
  return t;                                   // meaningful in thread 0
}

// ws: [gridDim.x] slots, then one unsigned ticket counter (zeroed by the launcher).
// out_total = inv_count * sum (x - target)^2 + weight * MMD and out_mse = the first term; out_mse NULL: the MMD term alone
// (grid = B, weight 1)
__global__ void __launch_bounds__(128) mse_mmd_fwd_det_kernel(int N, int B, int C, int ns, float inv2s2, float weight,
                                                              float svv, float srv, float inv_count,
                                                              const float* __restrict__ x, const float* __restrict__ target,
                                                              const float* __restrict__ Z, const int* __restrict__ idx,
                                                              float* __restrict__ ws, float* __restrict__ out_total,
                                                              float* __restrict__ out_mse) {
  __shared__ float red[4];
  __shared__ bool last;
  float acc = 0.f;
  if ((int)blockIdx.x < B) {
    const int b = blockIdx.x;
    const float cvv = svv / ((float)B * C * C), crv = ns > 0 ? srv * 2.f / ((float)B * ns * C) : 0.f;
    for (int p = threadIdx.x; p < C * C + ns * C; p += blockDim.x) {
      float3 a;
      float w;
      int c;
      if (p < C * C) {
        const int c0 = p / C;
        c = p - c0 * C;
        a = ld_z(Z, b, C, c0);
        w = cvv;
      } else {
        const int r = p - C * C, s = r / C;
        c = r - s * C;
        a = ld_x(x, idx[(size_t)b * ns + s]);
        w = -crv;
      }
      const float3 z = ld_z(Z, b, C, c);
      const float dx = a.x - z.x, dy = a.y - z.y, dz = a.z - z.z;
      acc += w * __expf(-sqrtf(dx * dx + dy * dy + dz * dz) * inv2s2);
    }
  } else {
    const size_t n = (size_t)N * 3, stride = (size_t)(gridDim.x - B) * blockDim.x;
    for (size_t i = (size_t)(blockIdx.x - B) * blockDim.x + threadIdx.x; i < n; i += stride) {
      const float d = x[i] - target[i];
      acc = fmaf(d, d, acc);
    }
  }
  acc = block_sum_ordered(acc, red);
  unsigned* ticket = reinterpret_cast<unsigned*>(ws + gridDim.x);
  if (threadIdx.x == 0) {
    ws[blockIdx.x] = acc;
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  float m = 0.f, e = 0.f;                     // slots in CTA order, strided over the threads, then the fixed reduction
  for (int k = threadIdx.x; k < (int)gridDim.x; k += blockDim.x) {
    const float v = __ldcg(ws + k);
    if (k < B) m += v; else e += v;
  }
  m = block_sum_ordered(m, red);
  e = block_sum_ordered(e, red);
  if (threadIdx.x == 0) {
    e *= inv_count;
    out_total[0] = out_mse != nullptr ? e + weight * m : m;
    if (out_mse != nullptr) out_mse[0] = e;
  }
}

// gx = k (x - target), k = (g_total + g_mse) 2 inv_count: one term per element, a plain store
__global__ void __launch_bounds__(128) mse_bwd_det_kernel(int N, float inv_count, const float* __restrict__ x,
                                                          const float* __restrict__ target, const float* __restrict__ g_total,
                                                          const float* __restrict__ g_mse, float* __restrict__ gx) {
  const float gt = g_total != nullptr ? g_total[0] : 0.f, gm = g_mse != nullptr ? g_mse[0] : 0.f;
  const float k = (gt + gm) * 2.f * inv_count;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)N * 3; i += (size_t)gridDim.x * blockDim.x)
    gx[i] = k * (x[i] - target[i]);
}

// one CTA per graph: gZ[b] written, MMD gradient of the sampled nodes added onto gx.  gl = g[0] * weight.
__global__ void __launch_bounds__(128) mmd_bwd_det_kernel(int B, int C, int ns, float inv2s2, float weight, float svv, float srv,
                                                          const float* __restrict__ x, const float* __restrict__ Z,
                                                          const int* __restrict__ idx, const float* __restrict__ g,
                                                          float* __restrict__ gx, float* __restrict__ gZ) {
  const int b = blockIdx.x, lane = threadIdx.x & 31;
  const float gl = (g != nullptr ? g[0] : 0.f) * weight;
  const float cvv = svv * gl / ((float)B * C * C), crv = ns > 0 ? srv * 2.f * gl / ((float)B * ns * C) : 0.f;
  // channel c takes part in pairs (c0, c) as q, (c, c1) as p and (s, c) as q
  for (int c = threadIdx.x >> 5; c < C; c += blockDim.x >> 5) {
    const float3 zc = ld_z(Z, b, C, c);
    float ax = 0.f, ay = 0.f, az = 0.f;
    for (int j = lane; j < 2 * C + ns; j += 32) {
      float3 t;
      if (j < C) {
        t = mmd_pair_grad(ld_z(Z, b, C, j), zc, cvv, inv2s2);
        t = make_float3(-t.x, -t.y, -t.z);
      } else if (j < 2 * C) {
        t = mmd_pair_grad(zc, ld_z(Z, b, C, j - C), cvv, inv2s2);
      } else {
        t = mmd_pair_grad(ld_x(x, idx[(size_t)b * ns + (j - 2 * C)]), zc, -crv, inv2s2);
        t = make_float3(-t.x, -t.y, -t.z);
      }
      ax += t.x; ay += t.y; az += t.z;
    }
    ax = warpsum(ax); ay = warpsum(ay); az = warpsum(az);
    if (lane == 0) {
      gZ[((size_t)b * 3 + 0) * C + c] = ax;
      gZ[((size_t)b * 3 + 1) * C + c] = ay;
      gZ[((size_t)b * 3 + 2) * C + c] = az;
    }
  }
  for (int s = threadIdx.x; s < ns; s += blockDim.x) {
    const int i = idx[(size_t)b * ns + s];
    const float3 p = ld_x(x, i);
    float ax = 0.f, ay = 0.f, az = 0.f;
    for (int c = 0; c < C; ++c) {
      const float3 t = mmd_pair_grad(p, ld_z(Z, b, C, c), -crv, inv2s2);
      ax += t.x; ay += t.y; az += t.z;
    }
    atomicAdd(gx + (size_t)i * 3 + 0, ax);
    atomicAdd(gx + (size_t)i * 3 + 1, ay);
    atomicAdd(gx + (size_t)i * 3 + 2, az);
  }
}

static inline int mse_ctas(int N) {
  const long long n = (long long)N * 3;
  long long c = (n + 128 * 8 - 1) / (128 * 8);
  return (int)(c < 1 ? 1 : (c > 1184 ? 1184 : c));      // at most 8 x 148 CTAs
}
// workspace of the deterministic forward: one slot per CTA and the ticket counter (enough for the MMD term alone too)
static inline size_t loss_det_ws_floats(int N, int B) { return (size_t)B + mse_ctas(N) + 1; }
static cudaError_t launch_loss_fwd_det(int N, int B, int C, int ns, float sigma, float weight, float svv, float srv,
                                       float inv_count, const float* x, const float* target, const float* Z, const int* idx,
                                       float* ws, float* out_total, float* out_mse, cudaStream_t st) {
  const int grid = B + (out_mse != nullptr ? mse_ctas(N) : 0);
  if (grid == 0) return cudaMemsetAsync(out_total, 0, sizeof(float), st);
  cudaError_t e = cudaMemsetAsync(ws + grid, 0, sizeof(unsigned), st);
  if (e != cudaSuccess) return e;
  mse_mmd_fwd_det_kernel<<<grid, 128, 0, st>>>(N, B, C, ns, 1.f / (2.f * sigma * sigma), weight, svv, srv, inv_count, x, target,
                                               Z, idx, ws, out_total, out_mse); ++g_launches;
  return cudaGetLastError();
}
cudaError_t launch_mse_mmd_fwd(int N, int B, int C, int ns, float sigma, float weight, float svv, float srv, float inv_count,
                               const float* x, const float* target, const float* Z, const int* idx, float* out_total,
                               float* out_mse, float* det_ws, cudaStream_t st) {
  if (det_ws != nullptr) return launch_loss_fwd_det(N, B, C, ns, sigma, weight, svv, srv, inv_count, x, target, Z, idx, det_ws,
                                                    out_total, out_mse, st);
  cudaError_t e = cudaMemsetAsync(out_total, 0, sizeof(float), st);
  if (e != cudaSuccess) return e;
  e = cudaMemsetAsync(out_mse, 0, sizeof(float), st);
  if (e != cudaSuccess) return e;
  mse_mmd_fwd_kernel<<<B + mse_ctas(N), 128, 0, st>>>(N, B, C, ns, 1.f / (2.f * sigma * sigma), weight, svv, srv, inv_count, x,
                                                       target, Z, idx, out_total, out_mse); ++g_launches;
  return cudaGetLastError();
}
cudaError_t launch_mse_mmd_bwd(int N, int B, int C, int ns, float sigma, float weight, float svv, float srv, float inv_count,
                               const float* x, const float* target, const float* Z, const int* idx, const float* g_total,
                               const float* g_mse, float* gx, float* gZ, bool det, cudaStream_t st) {
  if (det) {
    if (N > 0) {
      mse_bwd_det_kernel<<<mse_ctas(N), 128, 0, st>>>(N, inv_count, x, target, g_total, g_mse, gx); ++g_launches;
    }
    if (B > 0) {
      mmd_bwd_det_kernel<<<B, 128, 0, st>>>(B, C, ns, 1.f / (2.f * sigma * sigma), weight, svv, srv, x, Z, idx, g_total, gx,
                                            gZ); ++g_launches;
    }
    return cudaGetLastError();
  }
  cudaError_t e = cudaMemsetAsync(gx, 0, sizeof(float) * 3 * (size_t)N, st);
  if (e != cudaSuccess) return e;
  mse_mmd_bwd_kernel<<<B + mse_ctas(N), 128, 0, st>>>(N, B, C, ns, 1.f / (2.f * sigma * sigma), weight, svv, srv, inv_count, x,
                                                       target, Z, idx, g_total, g_mse, gx, gZ); ++g_launches;
  return cudaGetLastError();
}

cudaError_t launch_mmd_fwd(int B, int C, int ns, float sigma, float svv, float srv, const float* x, const float* Z, const int* idx,
                           float* loss, float* det_ws, cudaStream_t st) {
  if (det_ws != nullptr)
    return launch_loss_fwd_det(0, B, C, ns, sigma, 1.f, svv, srv, 0.f, x, nullptr, Z, idx, det_ws, loss, nullptr, st);
  cudaError_t e = cudaMemsetAsync(loss, 0, sizeof(float), st);
  if (e != cudaSuccess || B == 0) return e;
  mmd_fwd_kernel<<<B, 128, 0, st>>>(B, C, ns, 1.f / (2.f * sigma * sigma), svv, srv, x, Z, idx, loss); ++g_launches;
  return cudaGetLastError();
}
cudaError_t launch_mmd_bwd(int N, int B, int C, int ns, float sigma, float svv, float srv, const float* x, const float* Z, const int* idx,
                           const float* gloss, float* gx, float* gZ, bool det, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(gx, 0, sizeof(float) * 3 * (size_t)N, st);
  if (e != cudaSuccess || B == 0) return e;
  if (det) {
    mmd_bwd_det_kernel<<<B, 128, 0, st>>>(B, C, ns, 1.f / (2.f * sigma * sigma), 1.f, svv, srv, x, Z, idx, gloss, gx, gZ);
    ++g_launches;
    return cudaGetLastError();
  }
  mmd_bwd_kernel<<<B, 128, 0, st>>>(B, C, ns, 1.f / (2.f * sigma * sigma), svv, srv, x, Z, idx, gloss, gx, gZ); ++g_launches;
  return cudaGetLastError();
}

}  // namespace fegnn
