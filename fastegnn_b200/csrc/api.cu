// api.cu -- the C ABI of libfegnn.so (include/fegnn.h): argument checking, workspace
// carving, phase launchers and the whole-layer / whole-stack drivers.
// Single translation unit: the kernel files are included below.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "adam.cu"
#include "edge_kernels.cu"
#include "edge_tc.cu"
#include "edge_tc_bwd.cu"
#include "edge_tc_bwd2.cu"
#include "edge_tc_bwd3.cu"
#include "edge_tc_bwd4.cu"
#include "graph_kernels.cu"
#include "graph_prep.cu"
#include "radius_graph.cu"
#include "halo.cu"
#include "mmd.cu"
#include "node_kernels.cu"
#include "virtual_kernels.cu"
#include "virtual_tc.cu"
#include "node_tc.cu"
#include "dense_tc.cu"
#include "segment.cu"
#include "peak_probe.cu"
#include "input_grads.cu"

using namespace fegnn;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CK(expr)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (expr);                                                                      \
    if (e__ != cudaSuccess) return fail(FEGNN_ECUDA, "%s: %s", #expr, cudaGetErrorString(e__));    \
  } while (0)
#define RQ(cond)                                                              \
  do {                                                                        \
    if (!(cond)) return fail(FEGNN_EINVAL, "%s: requirement failed: %s", __func__, #cond); \
  } while (0)
#define NO_DET(why)                                                                                                \
  do {                                                                                                             \
    if (g_det) return fail(FEGNN_EINVAL, "%s has no deterministic form (%s); set mode \"deterministic\" to 0 to run it", \
                           __func__, why);                                                                         \
  } while (0)
// FEGNN_F_RECOMPUTE is read by the fegnn_model_* entries (and selects the saved-only forms of the virtual and phi_h forwards);
// every other per-layer entry refuses it
#define NO_RECOMPUTE(d)                                                                                            \
  do {                                                                                                             \
    if ((d) != nullptr && ((d)->flags & (FEGNN_F_RECOMPUTE | FEGNN_F_REBUILD_ALL)))                                \
      return fail(FEGNN_EINVAL, "%s: FEGNN_F_RECOMPUTE is a flag of the fegnn_model_* entries (and of the saved-only " \
                  "fegnn_virtual_forward / fegnn_node_h_forward)", __func__);                                       \
  } while (0)
#define TRY(expr)            \
  do {                       \
    int rc__ = (expr);       \
    if (rc__ != 0) return rc__; \
  } while (0)

// 0 = fp32 FMA kernels, 1 = tcgen05 single-pass TF32, 3 = tcgen05 3xTF32 (fp32-grade)
int g_edge_fwd_mode = 1;
// 0 = fp32 FMA kernel, 1 = tcgen05 TF32 with shared-memory operands, 2 / 4 = tcgen05 TF32 with tensor-memory A operands
// and MN-major weight-gradient operands (256 / 512 threads per tile), 5 = tcgen05 kind::f16 with two tile streams per CTA,
// 7 / 8 = the same operand format with packed-fp16 epilogue arithmetic, coalesced scatter and next-tile prefetch
// (edge_tc_bwd4.cu; 256 / 512 threads per tile), 6 = auto (default): 7 wherever the tensor-core form applies (measured on
// the B200, per launch: 98 us at 1.8e5 edges and 1.03 ms at 3.6e6 against 116 us / 1.82 ms for mode 4 and 120 us / 1.42 ms
// for mode 5), else 4 / 0
int g_edge_bwd_mode = 6;

// 0 = fp32 FMA kernels, 1 = tcgen05 TF32 kernels (attention=True layers always take 0)
int g_virt_fwd_mode = 1;
int g_virt_bwd_mode = 1;
// per-node dense phases of the forward: 0 = fp32 FMA kernels, 1 = tcgen05 TF32 node_pre.  Opt-in: h is the one operand of the
// path that is neither bounded by an activation nor an invariant the next layer re-derives exactly, so rounding it to
// TF32 turns fp32-level noise between a rotated and an unrotated run into 2^-11 |h| jumps in P / Q / Av / Uh -- measured
// 2.2e-4 on equivariant_test.py's U(0,10) inputs against its atol of 1e-4.
// 3 (default) = node_pre on the fp32 FMA kernel, phi_h (fegnn_node_h_forward) on tcgen05 with the error-compensated 3xTF32
// split (fp32-grade: node_tc.cu); mode 1 takes the same phi_h kernel.
int g_node_fwd_mode = 3;
const bool g_node_pre_tc3 = getenv("FEGNN_NODE_PRE_TC3") == nullptr || atoi(getenv("FEGNN_NODE_PRE_TC3")) != 0;   // experiment switch
// per-node dense phases of the BACKWARD pass (node_pre_backward, node_h_backward): 0 = fp32 FMA kernels, 1 = tcgen05 TF32
// (dense_tc.cu; gradients do not enter the forward equivariance), 2 = auto (default) = 1 today: the per-tile kernel that
// walks the weight blocks, at every size (measured at 8 000 nodes: step 1.380 ms against 1.416 ms with the fp32 kernels; at
// 160 000 nodes 11.95 ms against 12.89 ms with the (tile, block) kernel, which stays selectable by environment).
int g_node_bwd_mode = 2;
// "deterministic" (fegnn_set_mode): 1 = bit-reproducible forms of the entries that have one; every entry that sums floats
// across CTAs in arrival order and has no such form refuses to run (NO_DET) instead of running nondeterministically
int g_det = 0;
// "layer_overlap" (fegnn_set_mode; environment FEGNN_LAYER_OVERLAP): in fegnn_model_backward_inputs each layer's virtual
// backward runs on a second stream next to its edge backward (DESIGN 3.7) -- 2 = at every size, 1 = auto (default: where
// it measured faster), 0 = never (the two one after the other)
int g_layer_overlap = getenv("FEGNN_LAYER_OVERLAP") ? atoi(getenv("FEGNN_LAYER_OVERLAP")) : 1;
// SMs of the virtual backward in that arrangement (the edge backward gets the rest): 0 = its share of the layer's SM time
const int g_overlap_vsms = getenv("FEGNN_OVERLAP_VSMS") ? atoi(getenv("FEGNN_OVERLAP_VSMS")) : 0;   // experiment switch
constexpr int kNodeTcMinN = 0;
inline bool node_bwd_tc(int N) { return g_node_bwd_mode == 1 || (g_node_bwd_mode == 2 && N >= kNodeTcMinN); }

// "grid_sms" (fegnn_set_mode; test-only): 0 = the device's SM count (default), n >= 2 = min(n, that count).  sm_count()
// sizes launch shapes only (persistent grids, the layer_overlap SM split), never a workspace, so a small cap makes every
// persistent kernel run many tiles per CTA at sizes where the fp64 reference is instant.
int g_grid_sms = 0;

int sm_count() {
  static int sms[64] = {};                  // per device ordinal (a process may drive several GPUs)
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return g_grid_sms > 0 ? min(g_grid_sms, 148) : 148;
  if (sms[dev] == 0) {
    if (cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms[dev] <= 0) sms[dev] = 148;
  }
  return g_grid_sms > 0 ? min(g_grid_sms, sms[dev]) : sms[dev];
}

// the deterministic loss forward keeps per-CTA partials in the caller's workspace (fegnn_loss_workspace_floats)
int check_loss_ws(int N, int B, const float* ws, size_t floats) {
  if (!g_det) return 0;
  const size_t need = loss_det_ws_floats(N, B);
  if (ws == nullptr || floats < need) return fail(FEGNN_ENOMEM, "loss workspace %zu < %zu floats", ws ? floats : 0, need);
  return 0;
}

int check_dims(const fegnn_dims* d) {
  if (d == nullptr) return fail(FEGNN_EINVAL, "dims is null");
  if (d->N < 0 || d->Nl < d->N || d->E < 0 || d->B < 0) return fail(FEGNN_EINVAL, "bad sizes N=%d Nl=%d E=%d B=%d", d->N, d->Nl, d->E, d->B);
  if (d->C < 1 || d->C > FEGNN_MAX_C) return fail(FEGNN_EINVAL, "virtual_channels C=%d outside [1,%d]", d->C, FEGNN_MAX_C);
  if (d->Fe < 0 || d->Fe > FEGNN_MAX_FE) return fail(FEGNN_EINVAL, "edge_attr width Fe=%d outside [0,%d]", d->Fe, FEGNN_MAX_FE);
  if (d->Fa < 0 || d->Fa > FEGNN_MAX_FA) return fail(FEGNN_EINVAL, "node_attr width Fa=%d outside [0,%d]", d->Fa, FEGNN_MAX_FA);
  if ((d->Fa == 0) != (d->node_attr == nullptr))
    return fail(FEGNN_EINVAL, "node_attr must be %s with Fa=%d", d->Fa == 0 ? "NULL" : "non-NULL", d->Fa);
  if (d->Fa > 0 && (d->flags & FEGNN_F_RF)) return fail(FEGNN_EINVAL, "FEGNN_F_RF layers have no phi_h: Fa must be 0");
  return 0;
}

// Requested input gradients (fegnn_input_grads): refused before any launch where the layer has no such input or the
// selected kernel cannot form the gradient.  The edge_attr gradient needs gz1, which only the fp32 kernel (mode 0) and the
// packed-fp16 kernel with 256 threads per tile (mode 7, and 6 = auto) form it from; auto then picks 7 where it applies,
// else 0.  The environment-only tensor-core forms (1, 2, 4, 5, 8) refuse a request.
int check_input_grads(const fegnn_dims* d, const fegnn_input_grads* ig) {
  if (ig == nullptr) return 0;
  if (ig->node_attr != nullptr && d->Fa == 0) return fail(FEGNN_EINVAL, "node_attr gradient requested with Fa = 0");
  if (ig->edge_attr != nullptr && d->Fe == 0) return fail(FEGNN_EINVAL, "edge_attr gradient requested with Fe = 0");
  if (ig->node_vel != nullptr && (d->flags & FEGNN_F_RF))
    return fail(FEGNN_EINVAL, "node_vel gradient requested on FEGNN_F_RF layers (v enters through |v|; not implemented)");
  const bool tc_ok = d->Fe <= kTcMaxFe && !(d->flags & FEGNN_F_ATTENTION);
  const int m = g_edge_bwd_mode;
  if (ig->edge_attr != nullptr && tc_ok && m != 0 && m != 6 && m != 7)
    return fail(FEGNN_EINVAL, "edge_backward mode %d has no edge_attr gradient (modes 0, 6 = auto and 7 have)", m);
  return 0;
}

// FEGNN_F_LIVE_EDGES: the graph must carry its live edge count, and the edge backward (edge_bwd) must have a kernel with a
// live form -- modes 1, 2, 4 and 5 have none and refuse the flag.  Checked before any launch of an entry.
int check_live(const fegnn_dims* d, const fegnn_graph* g, bool edge_bwd) {
  if (d == nullptr || !(d->flags & FEGNN_F_LIVE_EDGES)) return 0;
  if (g == nullptr || g->n_edges == nullptr)
    return fail(FEGNN_EINVAL, "FEGNN_F_LIVE_EDGES is set but fegnn_graph.n_edges is NULL (the live edge count is required)");
  const int m = g_edge_bwd_mode;
  if (edge_bwd && (m == 1 || m == 2 || m == 4 || m == 5))
    return fail(FEGNN_EINVAL, "edge_backward mode %d has no form for FEGNN_F_LIVE_EDGES (modes 0, 6 = auto, 7 and 8 have)", m);
  return 0;
}

inline size_t al4(size_t n) { return (n + 3) & ~(size_t)3; }
// Zero two float buffers with ONE memset node when they are neighbours in the caller's block (the model driver's
// workspaces place them so; padding between 16-byte aligned slots is owned by the block), else with two.
cudaError_t zero_pair(float* a, size_t na, float* b, size_t nb, cudaStream_t st) {
  if (na == 0 || nb == 0) {
    if (na) return cudaMemsetAsync(a, 0, sizeof(float) * na, st);
    if (nb) return cudaMemsetAsync(b, 0, sizeof(float) * nb, st);
    return cudaSuccess;
  }
  if (b == a + al4(na)) return cudaMemsetAsync(a, 0, sizeof(float) * (al4(na) + nb), st);
  if (a == b + al4(nb)) return cudaMemsetAsync(b, 0, sizeof(float) * (al4(nb) + na), st);
  cudaError_t e = cudaMemsetAsync(a, 0, sizeof(float) * na, st);
  if (e != cudaSuccess) return e;
  return cudaMemsetAsync(b, 0, sizeof(float) * nb, st);
}
inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline int ld1(const fegnn_dims* d) { return 2 * kH + 1 + d->Fe; }
inline int ldv(const fegnn_dims* d) { return 2 * kH + 1 + d->C; }
inline int ldn(const fegnn_dims* d) { return 2 * kH + kH * d->C + d->Fa; }
// the attribute term of Uh: columns [ldn - Fa, ldn) of node_mlp.0.weight (and of its gradient)
NodeAttrArgs node_attr_args(const fegnn_dims* d, const float* w0, float* gw0) {
  NodeAttrArgs at;
  memset(&at, 0, sizeof(at));
  const int off = ldn(d) - d->Fa;
  at.Fa = d->Fa; at.ldn = ldn(d); at.a = d->node_attr;
  at.w = w0 + off; at.gw = gw0 != nullptr ? gw0 + off : nullptr;
  return at;
}

EdgeArgs edge_args(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* x,
                   const fegnn_layer_saved* sv) {
  EdgeArgs a;
  memset(&a, 0, sizeof(a));   // msum / tsum share their slots with the backward's g_ea / perm (EdgeArgs): set per direction
  a.N = d->N; a.Nl = d->Nl; a.E = d->E; a.Fe = d->Fe; a.ld1 = ld1(d); a.flags = d->flags; a.eps = d->eps;
  a.row = g->row; a.col = g->col; a.ea = g->edge_attr; a.x = x; a.P = sv->P; a.Q = sv->Q;
  a.w1 = p->edge_w0; a.W2 = p->edge_w2; a.b2 = p->edge_b2; a.W3 = p->cr_w0; a.b3 = p->cr_b0; a.w4 = p->cr_w2;
  a.wa = p->att_w; a.ba = p->att_b;
  a.n_edges = (d->flags & FEGNN_F_LIVE_EDGES) ? g->n_edges : nullptr;
  static const unsigned exp_bits = getenv("FEGNN_EXP") ? (unsigned)atoi(getenv("FEGNN_EXP")) : 0u;
  a.exp = exp_bits;
  return a;
}

VirtArgs virt_args(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* x,
                   const float* v, const float* Z, const fegnn_layer_saved* sv) {
  VirtArgs a;
  memset(&a, 0, sizeof(a));
  a.N = d->N; a.B = d->B; a.C = d->C; a.ldv = ldv(d); a.flags = d->flags;
  a.grav[0] = d->gravity[0]; a.grav[1] = d->gravity[1]; a.grav[2] = d->gravity[2];
  a.batch = g->batch; a.x = x; a.v = v; a.Z = Z; a.Av = sv->Av; a.G1 = sv->G1; a.tsum = sv->tsum;
  a.dinv = (d->flags & FEGNN_F_COORDS_SUM) ? nullptr : g->dinv;   // coords_agg='sum': no 1/deg on the coordinate update
  a.sv = sv->sv; a.sg = sv->sg;
  a.wv1 = p->edgev_w0; a.V2 = p->edgev_w2; a.c2 = p->edgev_b2;
  a.Wxv = p->crv_w0; a.bxv = p->crv_b0; a.wxv = p->crv_w2;
  a.WX = p->cvv_w0; a.bX = p->cvv_b0; a.wX = p->cvv_w2;
  a.wav = p->attv_w; a.bav = p->attv_b;
  return a;
}

GraphArgs graph_args(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p) {
  GraphArgs a;
  memset(&a, 0, sizeof(a));
  a.B = d->B; a.C = d->C; a.ldv = ldv(d); a.flags = d->flags; a.inv_nb = g->inv_nb;
  a.wv1 = p->edgev_w0;
  a.nodev_w0 = p->nodev_w0; a.nodev_b0 = p->nodev_b0; a.nodev_w2 = p->nodev_w2; a.nodev_b2 = p->nodev_b2;
  return a;
}

NodePreArgs node_pre_args(const fegnn_dims* d, const fegnn_layer_params* p, const float* h) {
  NodePreArgs a;
  memset(&a, 0, sizeof(a));
  a.N = d->N; a.ld1 = ld1(d); a.ldv = ldv(d); a.ldn = ldn(d); a.flags = d->flags; a.h = h;
  a.edge_w0 = p->edge_w0; a.edge_b0 = p->edge_b0; a.edgev_w0 = p->edgev_w0; a.edgev_b0 = p->edgev_b0;
  a.node_w0 = p->node_w0; a.node_b0 = p->node_b0;
  a.vel_w0 = p->vel_w0; a.vel_b0 = p->vel_b0; a.vel_w2 = p->vel_w2; a.vel_b2 = p->vel_b2;
  a.grav_w0 = p->grav_w0; a.grav_b0 = p->grav_b0; a.grav_w2 = p->grav_w2; a.grav_b2 = p->grav_b2;
  return a;
}

// Scratch of the deterministic forward-only stack (fegnn_model_inference_det_workspace_floats), behind the stack's workspace.
// The phases below take it as `det`: nullptr = the default kernels, else their kDet forms.
struct DetWs {
  float* eslab;   // edge forward: tile-boundary row sums (edge_det_slab_floats)
  float* dval;    // virtual forward: the rows D sX, [N, C, 3]
  float* gslab;   // per-graph sums: chunk-boundary slots (det_graph_slab_floats)
};
inline int det_graph_width(const fegnn_dims* d) { return d->C * kH + 3 * d->C + 3; }   // Usum, Dsum, xsum_new
size_t det_ws_floats(const fegnn_dims* d) {
  return al4(edge_det_slab_floats(d->E)) + al4((size_t)d->N * d->C * 3) + al4(det_graph_slab_floats(d->N, det_graph_width(d)));
}
void det_ws_bind(const fegnn_dims* d, float* p, DetWs* w) {
  w->eslab = p; p += al4(edge_det_slab_floats(d->E));
  w->dval = p; p += al4((size_t)d->N * d->C * 3);
  w->gslab = p;
}

int check_flags_params(const fegnn_dims* d, const fegnn_layer_params* p) {
  if (p == nullptr) return fail(FEGNN_EINVAL, "layer params is null");
  if ((d->flags & FEGNN_F_ATTENTION) && (!p->att_w || !p->att_b || !p->attv_w || !p->attv_b))
    return fail(FEGNN_EINVAL, "attention flag set but att_mlp tensors are null");
  if ((d->flags & FEGNN_F_GRAVITY) && (!p->grav_w0 || !p->grav_b0 || !p->grav_w2 || !p->grav_b2))
    return fail(FEGNN_EINVAL, "gravity flag set but gravity_mlp tensors are null");
  return 0;
}

__global__ void broadcast_vnf_kernel(int B, int C, const float* __restrict__ vnf, float* __restrict__ S) {
  // S[b][c][k] = virtual_node_feat[0][k][c]   (models/FastEGNN.py:268 with channel-major layout)
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)B * C * kH) return;
  int k = (int)(idx & 63), c = (int)((idx >> 6) % C);
  S[idx] = vnf[k * C + c];
}
__global__ void reduce_gS_kernel(int B, int C, const float* __restrict__ gS, float* __restrict__ gvnf) {
  // g_virtual_node_feat[0][k][c] += sum_b gS[b][c][k]
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= C * kH) return;
  int k = idx & 63, c = idx >> 6;
  float acc = 0.f;
  for (int b = 0; b < B; ++b) acc += gS[((size_t)b * C + c) * kH + k];
  atomicAdd(gvnf + k * C + c, acc);
}
__global__ void final_gx_kernel(int N, const float* __restrict__ gx, const float* __restrict__ gxsum,
                                const int* __restrict__ batch, float* __restrict__ out) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * 3) return;
  int i = idx / 3, k = idx - i * 3;
  out[idx] = gx[idx] + gxsum[batch[i] * 3 + k];
}

}  // namespace

namespace {

// The per-graph phases run one CTA per graph.  fegnn_model_forward / backward put them on a second stream (fork / join
// with events, all capturable) so they overlap the node- and edge-parallel kernels instead of idling 147 SMs.
//
// The backward's virtual branch (layer_overlap) runs on a third stream, `vst`, forked and joined with vfork / vjoin.
struct SideStream {
  cudaStream_t st = nullptr, vst = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr, aux = nullptr, vfork = nullptr, vjoin = nullptr;
};
SideStream* side_stream() {
  static SideStream per_dev[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  SideStream* s = &per_dev[dev];
  if (s->st == nullptr) {
    if (cudaStreamCreateWithFlags(&s->st, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&s->fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&s->join, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&s->aux, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaStreamCreateWithFlags(&s->vst, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&s->vfork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&s->vjoin, cudaEventDisableTiming) != cudaSuccess) return nullptr;
  }
  return s;
}
#define FORK(side, main)                                 \
  do {                                                   \
    CK(cudaEventRecord((side)->fork, (main)));           \
    CK(cudaStreamWaitEvent((side)->st, (side)->fork, 0)); \
  } while (0)
#define JOIN(side, main)                                 \
  do {                                                   \
    CK(cudaEventRecord((side)->join, (side)->st));       \
    CK(cudaStreamWaitEvent((main), (side)->join, 0));    \
  } while (0)

}  // namespace

extern "C" {

const char* fegnn_last_error(void) { return g_err; }
int fegnn_version(void) { return 103; }      // 103: fegnn_dims.Fa / .node_attr; 102: "deterministic" mode, loss workspaces
unsigned long long fegnn_launch_count(void) { return g_launches; }
int fegnn_set_mode(const char* phase, int mode) {
  if (phase == nullptr) return fail(FEGNN_EINVAL, "phase is null");
  if (strcmp(phase, "edge_forward") == 0) {
    if (mode != 0 && mode != 1 && mode != 3) return fail(FEGNN_EINVAL, "edge_forward mode must be 0, 1 or 3");
    g_edge_fwd_mode = mode;
    return 0;
  }
  if (strcmp(phase, "edge_backward") == 0) {
    if (mode != 0 && mode != 1 && mode != 2 && (mode < 4 || mode > 8))
      return fail(FEGNN_EINVAL, "edge_backward mode must be 0, 1, 2, 4, 5, 6 (auto), 7 or 8");
    g_edge_bwd_mode = mode;
    return 0;
  }
  if (strcmp(phase, "node_forward") == 0 || strcmp(phase, "node_backward") == 0) {
    const bool fwd = phase[5] == 'f';
    if (mode != 0 && mode != 1 && !(mode == 2 && !fwd) && !(mode == 3 && fwd))
      return fail(FEGNN_EINVAL, "%s mode must be 0 or 1%s", phase, fwd ? " or 3 (3xTF32 phi_h)" : " or 2 (auto)");
    (fwd ? g_node_fwd_mode : g_node_bwd_mode) = mode;
    return 0;
  }
  if (strcmp(phase, "virtual_forward") == 0 || strcmp(phase, "virtual_backward") == 0) {
    if (mode != 0 && mode != 1) return fail(FEGNN_EINVAL, "%s mode must be 0 or 1", phase);
    (phase[8] == 'f' ? g_virt_fwd_mode : g_virt_bwd_mode) = mode;
    return 0;
  }
  if (strcmp(phase, "deterministic") == 0) {
    if (mode != 0 && mode != 1) return fail(FEGNN_EINVAL, "deterministic mode must be 0 or 1");
    g_det = mode;
    return 0;
  }
  if (strcmp(phase, "layer_overlap") == 0) {
    if (mode < 0 || mode > 2) return fail(FEGNN_EINVAL, "layer_overlap mode must be 0, 1 (auto) or 2");
    g_layer_overlap = mode;
    return 0;
  }
  if (strcmp(phase, "grid_sms") == 0) {
    // layer_overlap splits the SMs between two kernels (at least one each): a cap needs two
    if (mode != 0 && mode < 2) return fail(FEGNN_EINVAL, "grid_sms must be 0 (the device's SM count) or at least 2");
    g_grid_sms = mode;
    return 0;
  }
  return fail(FEGNN_EINVAL, "unknown phase '%s'", phase);
}
int fegnn_get_mode(const char* phase) {
  if (phase != nullptr && strcmp(phase, "edge_forward") == 0) return g_edge_fwd_mode;
  if (phase != nullptr && strcmp(phase, "edge_backward") == 0) return g_edge_bwd_mode;
  if (phase != nullptr && strcmp(phase, "node_forward") == 0) return g_node_fwd_mode;
  if (phase != nullptr && strcmp(phase, "node_backward") == 0) return g_node_bwd_mode;
  if (phase != nullptr && strcmp(phase, "virtual_forward") == 0) return g_virt_fwd_mode;
  if (phase != nullptr && strcmp(phase, "virtual_backward") == 0) return g_virt_bwd_mode;
  if (phase != nullptr && strcmp(phase, "deterministic") == 0) return g_det;
  if (phase != nullptr && strcmp(phase, "layer_overlap") == 0) return g_layer_overlap;
  if (phase != nullptr && strcmp(phase, "grid_sms") == 0) return g_grid_sms;
  return -1;
}

// ------------------------------------------------------------------ graph prep
size_t fegnn_graph_prep_workspace_bytes(int32_t N, int32_t E) { return graph_prep_workspace_bytes(N, E); }

int fegnn_graph_prep(int32_t N, int32_t E, int32_t B, int32_t Fe, const int64_t* edge_index, const int64_t* data_batch,
                     const float* edge_attr, int32_t* perm, int32_t* rowptr, int32_t* row, int32_t* col,
                     int32_t* batch, int32_t* gptr, float* edge_attr_sorted, float* dinv, float* inv_nb,
                     void* workspace, size_t workspace_bytes, void* stream) {
  RQ(N >= 0 && E >= 0 && B >= 0 && Fe >= 0);
  RQ(rowptr && gptr && (N == 0 || (batch && data_batch && dinv)) && (B == 0 || inv_nb));
  RQ(E == 0 || (edge_index && perm && row && col && workspace));
  RQ(E == 0 || Fe == 0 || (edge_attr && edge_attr_sorted));
  if (workspace_bytes < graph_prep_workspace_bytes(N, E))
    return fail(FEGNN_ENOMEM, "graph_prep workspace %zu < %zu bytes", workspace_bytes, graph_prep_workspace_bytes(N, E));
  // the counts chain (rowptr, gptr, reciprocals: 8 small launches) and the radix sort chain (7 launches) are independent:
  // the counts run on the side stream, so the call's critical path is the longer chain, not their sum
  SideStream* sd = E > 0 ? side_stream() : nullptr;
  if (sd != nullptr) FORK(sd, S(stream));
  CK(graph_prep(N, E, B, Fe, edge_index, data_batch, edge_attr, perm, rowptr, row, col, batch, gptr,
                edge_attr_sorted, dinv, inv_nb, workspace, S(stream), sd != nullptr ? sd->st : S(stream)));
  if (sd != nullptr) JOIN(sd, S(stream));
  return 0;
}

int fegnn_graph_prep_live(int32_t N, int32_t E, int32_t B, int32_t Fe, const int64_t* edge_index, const int64_t* data_batch,
                          const float* edge_attr, int32_t* perm, int32_t* rowptr, int32_t* row, int32_t* col,
                          int32_t* batch, int32_t* gptr, float* edge_attr_sorted, float* dinv, float* inv_nb,
                          void* workspace, size_t workspace_bytes, const int32_t* n_edges_in, int32_t* n_edges_out,
                          uint32_t* status, void* stream) {
  RQ(N >= 0 && E >= 0 && B >= 0 && Fe >= 0);
  RQ(n_edges_in && n_edges_out && status);
  RQ(rowptr && gptr && (N == 0 || (batch && data_batch && dinv)) && (B == 0 || inv_nb));
  RQ(E == 0 || (edge_index && perm && row && col && workspace));
  RQ(E == 0 || Fe == 0 || (edge_attr && edge_attr_sorted));
  if (workspace_bytes < graph_prep_workspace_bytes(N, E))
    return fail(FEGNN_ENOMEM, "graph_prep workspace %zu < %zu bytes", workspace_bytes, graph_prep_workspace_bytes(N, E));
  SideStream* sd = E > 0 ? side_stream() : nullptr;
  if (sd != nullptr) FORK(sd, S(stream));
  CK(graph_prep(N, E, B, Fe, edge_index, data_batch, edge_attr, perm, rowptr, row, col, batch, gptr, edge_attr_sorted, dinv,
                inv_nb, workspace, S(stream), sd != nullptr ? sd->st : S(stream), n_edges_in, n_edges_out, status));
  if (sd != nullptr) JOIN(sd, S(stream));
  return 0;
}

// ------------------------------------------------------------------ graph construction (SURVEY.md 8 f2)
size_t fegnn_radius_graph_workspace_bytes(int32_t N, int32_t B) { return radius_graph_workspace_bytes(N, B); }

int fegnn_radius_graph_count(int32_t N, int32_t B, const float* x, const int64_t* data_batch, float r, int32_t* batch,
                             int32_t* gptr, float* inv_nb, int32_t* cand_rowptr, int32_t* n_cand, void* workspace,
                             size_t workspace_bytes, void* stream) {
  RQ(N >= 0 && B >= 0 && r > 0.f);
  RQ(gptr && cand_rowptr && n_cand && (B == 0 || inv_nb) && (N == 0 || (x && data_batch && batch && B >= 1)));
  RQ(workspace != nullptr);
  if (workspace_bytes < radius_graph_workspace_bytes(N, B))
    return fail(FEGNN_ENOMEM, "radius_graph workspace %zu < %zu bytes", workspace_bytes, radius_graph_workspace_bytes(N, B));
  CK(radius_graph_count(N, B, x, data_batch, r, batch, gptr, inv_nb, cand_rowptr, n_cand, workspace, S(stream)));
  return 0;
}

int fegnn_radius_graph_fill(int32_t N, int32_t B, int32_t Fe, float r, double keep_frac, const int32_t* batch,
                            const int32_t* gptr, const int32_t* cand_rowptr, const int32_t* n_cand,
                            int32_t cand_capacity, int32_t* cand_col, float* cand_dist, int32_t* cand_row,
                            int32_t out_capacity, int32_t* rowptr, int32_t* row, int32_t* col, float* edge_attr,
                            float* dinv, int32_t* n_edges, void* workspace, size_t workspace_bytes, void* stream) {
  RQ(N >= 0 && B >= 0 && r > 0.f && Fe >= 0 && Fe <= FEGNN_MAX_FE && cand_capacity >= 0 && out_capacity >= 0);
  RQ(keep_frac >= 0.0);
  RQ(rowptr && n_edges && cand_rowptr && n_cand && (N == 0 || (batch && gptr)));
  RQ(cand_capacity == 0 || (cand_col && cand_dist && cand_row));
  RQ(out_capacity == 0 || (row && col && (Fe == 0 || edge_attr)));
  RQ(workspace != nullptr);
  if (workspace_bytes < radius_graph_workspace_bytes(N, B))
    return fail(FEGNN_ENOMEM, "radius_graph workspace %zu < %zu bytes", workspace_bytes, radius_graph_workspace_bytes(N, B));
  CK(radius_graph_fill(N, B, Fe, r, keep_frac, cand_capacity, batch, gptr, cand_rowptr, n_cand, cand_col, cand_dist,
                       cand_row, out_capacity, rowptr, row, col, edge_attr, dinv, n_edges, workspace, S(stream)));
  return 0;
}

int fegnn_radius_graph_fill_live(int32_t N, int32_t B, int32_t Fe, float r, double keep_frac, const int32_t* batch,
                                 const int32_t* gptr, const int32_t* cand_rowptr, const int32_t* n_cand,
                                 int32_t cand_capacity, int32_t* cand_col, float* cand_dist, int32_t* cand_row,
                                 int32_t out_capacity, int32_t* rowptr, int32_t* row, int32_t* col, float* edge_attr,
                                 float* dinv, int32_t* n_edges, int32_t* n_live, uint32_t* status, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  RQ(n_live && status);
  TRY(fegnn_radius_graph_fill(N, B, Fe, r, keep_frac, batch, gptr, cand_rowptr, n_cand, cand_capacity, cand_col, cand_dist,
                              cand_row, out_capacity, rowptr, row, col, edge_attr, dinv, n_edges, workspace, workspace_bytes,
                              stream));
  rg::live_status_kernel<<<1, 1, 0, S(stream)>>>(n_cand, cand_capacity, n_edges, out_capacity, n_live, status); ++g_launches;
  CK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ small phases
int fegnn_embed_forward(int32_t N, int32_t Fin, const float* node_feat, const float* w, const float* b, float* h,
                        void* stream) {
  RQ(N >= 0 && Fin >= 1 && Fin <= 16 && (N == 0 || (node_feat && w && b && h)));
  CK(launch_embed_fwd(N, Fin, node_feat, w, b, h, S(stream)));
  return 0;
}
int fegnn_embed_backward(int32_t N, int32_t Fin, const float* node_feat, const float* w, const float* gh, float* gw,
                         float* gb, float* gnode_feat, void* stream) {
  NO_DET("weight gradient flushed by many CTAs with float atomics");
  RQ(N >= 0 && Fin >= 1 && Fin <= 16 && (N == 0 || (node_feat && w && gh && gw && gb)));
  CK(launch_embed_bwd(N, Fin, node_feat, w, gh, gw, gb, gnode_feat, S(stream)));
  return 0;
}
}  // extern "C"
namespace {
int graph_xsum_run(int32_t N, int32_t B, const float* x, const int32_t* batch, float* xsum, const DetWs* det, void* stream) {
  RQ(N >= 0 && B >= 0 && (B == 0 || xsum) && (N == 0 || (x && batch)));
  CK(cudaMemsetAsync(xsum, 0, sizeof(float) * 3 * (size_t)B, S(stream)));
  if (det != nullptr) {
    DetSegArgs sa;
    memset(&sa, 0, sizeof(sa));
    sa.N = N; sa.n = 1; sa.batch = batch; sa.slab = det->gslab;
    sa.X[0] = x; sa.W[0] = 3; sa.out[0] = xsum;
    CK(launch_det_graph_sums(sa, S(stream)));
  } else {
    CK(launch_graph_xsum(N, x, batch, xsum, S(stream)));
  }
  return 0;
}
}  // namespace
extern "C" {
int fegnn_graph_xsum(int32_t N, int32_t B, const float* x, const int32_t* batch, float* xsum, void* stream) {
  NO_DET("per-graph sums across CTAs with float atomics");
  return graph_xsum_run(N, B, x, batch, xsum, nullptr, stream);
}

// ------------------------------------------------------------------ forward phases
}  // extern "C"
namespace {
int graph_pre_forward_run(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* Z,
                          const float* Sf, const float* xsum, fegnn_layer_saved* sv, void* stream) {
  TRY(check_dims(d));
  RQ(g && p && Z && Sf && xsum && sv);
  TRY(check_live(d, g, false));
  GraphArgs a = graph_args(d, g, p);
  a.Z = Z; a.S = Sf; a.xsum = xsum; a.M = sv->M; a.Zc = sv->Zc; a.G1 = sv->G1;
  CK(launch_graph_pre_fwd(a, S(stream)));
  return 0;
}

int node_pre_forward_run(const fegnn_dims* d, const fegnn_layer_params* p, const float* h, fegnn_layer_saved* sv,
                         void* stream) {
  TRY(check_dims(d));
  TRY(check_flags_params(d, p));
  RQ(h && sv);
  NodePreArgs a = node_pre_args(d, p, h);
  a.P = sv->P; a.Q = sv->Q; a.Av = sv->Av; a.Uh = sv->Uh; a.sv = sv->sv; a.sg = sv->sg;
  // node attributes enter Uh only; the last layer has none (its phi_h is discarded)
  const NodeAttrArgs at_ = node_attr_args(d, p->node_w0, nullptr);
  const NodeAttrArgs* at = d->Fa > 0 && !(d->flags & FEGNN_F_LAST) ? &at_ : nullptr;
  if (g_node_fwd_mode == 1 && !(d->flags & FEGNN_F_RF)) CK(launch_node_pre_fwd_tc(a, sm_count(), S(stream), at));
  else if (g_node_fwd_mode == 3 && g_node_pre_tc3) CK(launch_node_pre_fwd_tc3(a, sm_count(), S(stream), at));
  else CK(launch_node_pre_fwd(a, sm_count(), S(stream), at));
  return 0;
}

int edge_forward_run(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* x,
                     fegnn_layer_saved* sv, const DetWs* det, void* stream) {
  TRY(check_dims(d));
  TRY(check_flags_params(d, p));
  RQ(g && x && sv);
  TRY(check_live(d, g, false));
  EdgeArgs a = edge_args(d, g, p, x, sv);
  a.msum = sv->msum; a.tsum = sv->tsum;
  if (!(d->flags & FEGNN_F_PREZEROED)) CK(zero_pair(sv->msum, kH * (size_t)d->N, sv->tsum, 3 * (size_t)d->N, S(stream)));
  const int mode = d->Fe <= kTcMaxFe ? g_edge_fwd_mode : 0;
  if (d->flags & FEGNN_F_LIVE_EDGES) {
    // the kLive forms: grids from the capacity d->E, tiles from the live count
    if (det != nullptr) {
      a.slab = det->eslab;
      if (mode == 3) CK((launch_edge_fwd_tc<3, true, true>(a, sm_count(), S(stream))));
      else if (mode == 1) CK((launch_edge_fwd_tc<1, true, true>(a, sm_count(), S(stream))));
      else CK((launch_edge_fwd<true, true>(a, sm_count(), S(stream))));
      return 0;
    }
    if (mode == 3) CK((launch_edge_fwd_tc<3, false, true>(a, sm_count(), S(stream))));
    else if (mode == 1) CK((launch_edge_fwd_tc<1, false, true>(a, sm_count(), S(stream))));
    else CK((launch_edge_fwd<false, true>(a, sm_count(), S(stream))));
    return 0;
  }
  if (det != nullptr) {
    a.slab = det->eslab;
    if (mode == 3) CK((launch_edge_fwd_tc<3, true>(a, sm_count(), S(stream))));
    else if (mode == 1) CK((launch_edge_fwd_tc<1, true>(a, sm_count(), S(stream))));
    else CK(launch_edge_fwd<true>(a, sm_count(), S(stream)));
    return 0;
  }
  if (mode == 3) CK(launch_edge_fwd_tc<3>(a, sm_count(), S(stream)));
  else if (mode == 1) CK(launch_edge_fwd_tc<1>(a, sm_count(), S(stream)));
  else CK(launch_edge_fwd(a, sm_count(), S(stream)));
  return 0;
}

int virtual_forward_run(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* x,
                        const float* v, const float* Z, fegnn_layer_saved* sv, float* x_new, float* xsum_new,
                        const DetWs* det, void* stream) {
  TRY(check_dims(d));
  TRY(check_flags_params(d, p));
  // FEGNN_F_RECOMPUTE: the saved-only form (u, Dsum, Usum; x' and xsum_new are the next layer's state already)
  const bool saved_only = d->flags & FEGNN_F_RECOMPUTE;
  RQ(g && x && v && Z && sv && (saved_only || (x_new && xsum_new)));
  RQ(!saved_only || det == nullptr);
  TRY(check_live(d, g, false));
  VirtArgs a = virt_args(d, g, p, x, v, Z, sv);
  a.u = sv->u; a.x_new = x_new; a.Dsum = sv->Dsum; a.Usum = sv->Usum; a.xsum_new = xsum_new;
  if (!(d->flags & FEGNN_F_PREZEROED)) {
    CK(zero_pair(sv->Dsum, 3 * d->C * (size_t)d->B, sv->Usum, kH * d->C * (size_t)d->B, S(stream)));
    if (!saved_only) CK(cudaMemsetAsync(xsum_new, 0, sizeof(float) * 3 * (size_t)d->B, S(stream)));
  }
  const bool tc = g_virt_fwd_mode == 1 && !(d->flags & FEGNN_F_ATTENTION);
  if (saved_only) {
    a.x_new = nullptr; a.xsum_new = nullptr;
    if (tc) CK((launch_virtual_fwd_tc<2, false, true>(a, sm_count(), S(stream))));
    else CK((launch_virtual_fwd<false, true>(a, sm_count(), S(stream))));
    return 0;
  }
  if (det != nullptr) {
    // the kernel writes u, x_new and the rows D sX (into the Dsum slot); their per-graph sums follow in graph order
    a.Dsum = det->dval;
    if (tc) CK((launch_virtual_fwd_tc<2, true>(a, sm_count(), S(stream))));
    else CK(launch_virtual_fwd<true>(a, sm_count(), S(stream)));
    DetSegArgs sa;
    memset(&sa, 0, sizeof(sa));
    sa.N = d->N; sa.n = 3; sa.batch = g->batch; sa.slab = det->gslab;
    sa.X[0] = sv->u; sa.W[0] = d->C * kH; sa.out[0] = sv->Usum;
    sa.X[1] = det->dval; sa.W[1] = 3 * d->C; sa.out[1] = sv->Dsum; sa.remapC[1] = d->C;
    sa.X[2] = x_new; sa.W[2] = 3; sa.out[2] = xsum_new;
    CK(launch_det_graph_sums(sa, S(stream)));
    return 0;
  }
  if (tc) CK(launch_virtual_fwd_tc<2>(a, sm_count(), S(stream)));
  else CK(launch_virtual_fwd(a, sm_count(), S(stream)));
  return 0;
}

int node_h_forward_run(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* h,
                       fegnn_layer_saved* sv, float* h_new, const DetWs* det, void* stream) {
  TRY(check_dims(d));
  // FEGNN_F_RECOMPUTE: the saved-only form (zh1; h' is the next layer's state already)
  const bool saved_only = d->flags & FEGNN_F_RECOMPUTE;
  RQ(g && p && h && sv && (saved_only || h_new));
  RQ(!saved_only || det == nullptr);
  TRY(check_live(d, g, false));
  NodeHArgs a;
  memset(&a, 0, sizeof(a));
  a.N = d->N; a.C = d->C; a.ldn = ldn(d);
  a.h = h; a.Uh = sv->Uh; a.msum = sv->msum; a.u = sv->u;
  a.dinv = (d->flags & FEGNN_F_NODE_SUM) ? nullptr : g->dinv;     // VNEGNN's A2A stage sums the messages (models/VNEGNN.py:87)
  a.node_w0 = p->node_w0; a.node_w2 = p->node_w2; a.node_b2 = p->node_b2;
  a.zh1 = sv->zh1; a.h_new = h_new;
  a.wimg = sv->wimg;
  if (g_node_fwd_mode != 0 && sv->wimg != nullptr) {
    if (!(d->flags & FEGNN_F_WIMG_READY)) {
      const float *w0 = p->node_w0, *w2 = p->node_w2;
      float* img = sv->wimg;
      CK(launch_node_h_wprep(d->C, ldn(d), 1, &w0, &w2, &img, S(stream)));
    }
    if (saved_only) CK(launch_node_h_fwd_tc<true>(a, sm_count(), S(stream)));
    else CK(launch_node_h_fwd_tc(a, sm_count(), S(stream)));
  }
  else if (saved_only) CK((launch_node_h_fwd<false, true>(a, sm_count(), S(stream), !(d->flags & FEGNN_F_PREZEROED))));
  else if (det != nullptr) CK(launch_node_h_fwd<true>(a, sm_count(), S(stream)));
  else CK(launch_node_h_fwd(a, sm_count(), S(stream), !(d->flags & FEGNN_F_PREZEROED)));
  return 0;
}

}  // namespace
extern "C" {
int fegnn_node_h_weight_images(const fegnn_dims* d, int32_t nl, const fegnn_layer_params* layers, float* const* wimg,
                               void* stream) {
  NO_RECOMPUTE(d);
  TRY(check_dims(d));
  RQ(nl >= 0 && nl <= 32 && (nl == 0 || (layers && wimg)));
  const float *w0[32], *w2[32];
  for (int l = 0; l < nl; ++l) {
    RQ(layers[l].node_w0 && layers[l].node_w2 && wimg[l]);
    w0[l] = layers[l].node_w0; w2[l] = layers[l].node_w2;
  }
  CK(launch_node_h_wprep(d->C, ldn(d), nl, w0, w2, wimg, S(stream)));
  return 0;
}
}  // extern "C"
namespace {

int graph_post_forward_run(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* Z,
                           const float* Sf, const fegnn_layer_saved* sv, float* Z_new, float* S_new, void* stream) {
  TRY(check_dims(d));
  RQ(g && p && Z && Sf && sv && Z_new && ((d->flags & FEGNN_F_LAST) || S_new));
  TRY(check_live(d, g, false));
  GraphArgs a = graph_args(d, g, p);
  a.Z = Z; a.S = Sf; a.Dsum = sv->Dsum; a.Usum = sv->Usum; a.Z_new = Z_new; a.S_new = S_new;
  CK(launch_graph_post_fwd(a, S(stream)));
  return 0;
}

}  // namespace
extern "C" {
int fegnn_graph_pre_forward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* Z,
                            const float* Sf, const float* xsum, fegnn_layer_saved* sv, void* stream) {
  NO_RECOMPUTE(d);
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  return graph_pre_forward_run(d, g, p, Z, Sf, xsum, sv, stream);
}

int fegnn_node_pre_forward(const fegnn_dims* d, const fegnn_layer_params* p, const float* h, fegnn_layer_saved* sv,
                           void* stream) {
  NO_RECOMPUTE(d);
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  return node_pre_forward_run(d, p, h, sv, stream);
}

int fegnn_edge_forward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* x,
                       fegnn_layer_saved* sv, void* stream) {
  NO_RECOMPUTE(d);
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  return edge_forward_run(d, g, p, x, sv, nullptr, stream);
}

int fegnn_virtual_forward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* x,
                          const float* v, const float* Z, fegnn_layer_saved* sv, float* x_new, float* xsum_new,
                          void* stream) {
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  return virtual_forward_run(d, g, p, x, v, Z, sv, x_new, xsum_new, nullptr, stream);
}

int fegnn_node_h_forward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* h,
                         fegnn_layer_saved* sv, float* h_new, void* stream) {
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  return node_h_forward_run(d, g, p, h, sv, h_new, nullptr, stream);
}

int fegnn_graph_post_forward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* Z,
                             const float* Sf, const fegnn_layer_saved* sv, float* Z_new, float* S_new, void* stream) {
  NO_RECOMPUTE(d);
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  return graph_post_forward_run(d, g, p, Z, Sf, sv, Z_new, S_new, stream);
}

// ------------------------------------------------------------------ backward phases
int fegnn_graph_post_backward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                              fegnn_layer_grads* gr, const float* Sf, const fegnn_layer_saved* sv,
                              const float* gZ_new, const float* gS_new, float* gZ, float* gS, float* gDsum,
                              float* gUsum, void* stream) {
  NO_RECOMPUTE(d);
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  TRY(check_dims(d));
  const bool last = d->flags & FEGNN_F_LAST;
  RQ(g && p && gr && sv && gZ_new && gZ && gS && gDsum && gUsum && (last || (Sf && gS_new)));
  TRY(check_live(d, g, false));
  GraphArgs a = graph_args(d, g, p);
  a.S = Sf; a.Usum = sv->Usum; a.gZ_new = gZ_new; a.gS_new = gS_new;
  a.gZ = gZ; a.gS = gS; a.gDsum = gDsum; a.gUsum = gUsum;
  a.g_nodev_w0 = gr->nodev_w0; a.g_nodev_b0 = gr->nodev_b0; a.g_nodev_w2 = gr->nodev_w2; a.g_nodev_b2 = gr->nodev_b2;
  CK(launch_graph_post_bwd(a, S(stream)));
  return 0;
}

int fegnn_node_h_backward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                          fegnn_layer_grads* gr, const fegnn_layer_saved* sv, const float* gh_new, float* gzh1,
                          float* gm, float* gu, void* stream) {
  NO_RECOMPUTE(d);
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  TRY(check_dims(d));
  RQ(g && p && gr && sv && gh_new && gzh1 && gm && gu);
  TRY(check_live(d, g, false));
  NodeHArgs a;
  memset(&a, 0, sizeof(a));
  a.N = d->N; a.C = d->C; a.ldn = ldn(d);
  a.msum = sv->msum; a.u = sv->u; a.zh1 = sv->zh1;
  a.dinv = (d->flags & FEGNN_F_NODE_SUM) ? nullptr : g->dinv;
  a.node_w0 = p->node_w0; a.node_w2 = p->node_w2; a.node_b2 = p->node_b2;
  a.gh_new = gh_new; a.gzh1 = gzh1; a.gm = gm; a.gu = gu;
  a.g_node_w0 = gr->node_w0; a.g_node_w2 = gr->node_w2; a.g_node_b2 = gr->node_b2;
  if (node_bwd_tc(d->N)) {
    // tcgen05: (1) gzh1 = (gh' U2) * silu'(zh1), dU2 += gh'^T silu(zh1), de2 += sum gh' ; (2) per K-block of the first
    // Linear: gm = (gzh1 U1a) / deg, gu_c = gzh1 U1u_c, dU1 blocks += gzh1^T [msum / deg | u_c]
    dtc::Args t1;
    memset(&t1, 0, sizeof(t1));
    t1.N = d->N; t1.nblk = 1;
    dtc::Blk& b = t1.blk[0];
    b.X = gh_new; b.ldx = kH; b.Y = sv->zh1; b.ldy = kH; b.ysilu = 1; b.W = p->node_w2; b.ldw = kH; b.wks = 1;
    b.D = gzh1; b.ldd = kH; b.dmode = 1; b.dz = sv->zh1; b.gW = gr->node_w2; b.gb = gr->node_b2;
    CK(launch_dense_bwd_tc(t1, sm_count(), S(stream)));
    dtc::Args t2;
    memset(&t2, 0, sizeof(t2));
    t2.N = d->N; t2.nblk = d->C + 1;
    for (int k = 0; k <= d->C; ++k) {
      dtc::Blk& q = t2.blk[k];
      q.X = gzh1; q.ldx = kH; q.ldw = a.ldn; q.dmode = 1;
      if (k == 0) {
        q.Y = sv->msum; q.ldy = kH; q.yscale = a.dinv; q.W = p->node_w0 + kH; q.wks = 1;
        q.D = gm; q.ldd = kH; q.dscale = a.dinv; q.gW = gr->node_w0 ? gr->node_w0 + kH : nullptr;
        q.dmax = sv->scratch != nullptr ? reinterpret_cast<unsigned*>(sv->scratch) + 1 : nullptr;   // max|gm| (FEGNN_F_STATS_READY)
      } else {
        const int c = k - 1;
        q.Y = sv->u + (size_t)c * kH; q.ldy = d->C * kH; q.W = p->node_w0 + 2 * kH + c; q.wks = d->C;
        q.D = gu + (size_t)c * kH; q.ldd = d->C * kH; q.gW = gr->node_w0 ? gr->node_w0 + 2 * kH + c : nullptr;
      }
    }
    CK(launch_dense_bwd_tc(t2, sm_count(), S(stream)));
    return 0;
  }
  CK(launch_node_h_bwd(a, sm_count(), S(stream)));
  return 0;
}

int fegnn_virtual_backward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                           fegnn_layer_grads* gr, const float* x, const float* v, const float* Z,
                           const fegnn_layer_saved* sv, const float* gx_new, const float* gxsum_next,
                           const float* gDsum, const float* gUsum, const float* gu, float* gAv, float* gG1, float* gx,
                           float* gZ, float* gsv, float* gsg, float* gt, void* stream) {
  return fegnn_virtual_backward_inputs(d, g, p, gr, x, v, Z, sv, gx_new, gxsum_next, gDsum, gUsum, gu, gAv, gG1, gx, gZ, gsv,
                                       gsg, gt, nullptr, stream);
}
// the virtual backward runs on its two tensor-core kernels (else on the fp32 kernel)
static bool virt_bwd_tc(const fegnn_dims* d, const float* gu) {
  return g_virt_bwd_mode == 1 && !(d->flags & FEGNN_F_ATTENTION) && gu != nullptr;
}
// gt_ahead: gt and its bound statistics were formed by launch_virtual_bwd_gt (fegnn_model_backward_inputs, layer_overlap;
// tensor-core kernels only), which the heads kernel then skips.  cap: grid cap of the tensor-core kernels.
static int virtual_backward_run(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                                fegnn_layer_grads* gr, const float* x, const float* v, const float* Z,
                                const fegnn_layer_saved* sv, const float* gx_new, const float* gxsum_next,
                                const float* gDsum, const float* gUsum, const float* gu, float* gAv, float* gG1, float* gx,
                                float* gZ, float* gsv, float* gsg, float* gt, const fegnn_input_grads* ig, bool gt_ahead,
                                int cap, void* stream) {
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  TRY(check_dims(d));
  TRY(check_flags_params(d, p));
  TRY(check_input_grads(d, ig));
  RQ(g && gr && x && v && Z && sv && gx_new && gDsum && gAv && gG1 && gx && gZ && gsv && gt);
  TRY(check_live(d, g, false));
  RQ(!gt_ahead || virt_bwd_tc(d, gu));
  RQ(!(d->flags & FEGNN_F_GRAVITY) || gsg);
  VirtArgs a = virt_args(d, g, p, x, v, Z, sv);
  a.gx_new = gx_new; a.gxsum_next = gxsum_next; a.gDsum = gDsum; a.gUsum = gUsum; a.gu = gu;
  a.gAv = gAv; a.gG1 = gG1; a.gx = gx; a.gZ = gZ; a.gsv = gsv; a.gsg = gsg; a.gt = gt;
  a.g_wv1 = gr->edgev_w0; a.g_V2 = gr->edgev_w2; a.g_c2 = gr->edgev_b2;
  a.g_Wxv = gr->crv_w0; a.g_bxv = gr->crv_b0; a.g_wxv = gr->crv_w2;
  a.g_WX = gr->cvv_w0; a.g_bX = gr->cvv_b0; a.g_wX = gr->cvv_w2;
  a.g_wav = gr->attv_w; a.g_bav = gr->attv_b;
  if (!(d->flags & FEGNN_F_PREZEROED)) CK(zero_pair(gG1, kH * d->C * (size_t)d->B, gx, 3 * (size_t)d->Nl, S(stream)));
  // tensor-core form: two kernels; `gu` doubles as the [N,C,H] scratch that carries the total dL/du between them
  if (d->flags & FEGNN_F_LAST) a.gu = nullptr;        // last layer: phi_h is discarded, a gu buffer holds no input
  if (virt_bwd_tc(d, gu)) {
    a.gu_work = const_cast<float*>(gu);
    a.u = sv->u;                                       // the heads are recomputed from the saved u
    a.stats = reinterpret_cast<unsigned*>(sv->scratch);   // max|gt|, max|x - x_0| for the edge backward (FEGNN_F_STATS_READY)
    if (gt_ahead) { a.gt = nullptr; a.stats = nullptr; }
    CK(launch_virtual_bwd_tc<4>(a, cap, S(stream)));
  } else {
    CK(launch_virtual_bwd(a, sm_count(), S(stream)));
  }
  if (ig != nullptr && ig->node_vel != nullptr)
    CK(launch_input_grad_vel(d->N, sv->sv, gx_new, gxsum_next, g->batch, ig->node_vel, S(stream)));
  return 0;
}
int fegnn_virtual_backward_inputs(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                                  fegnn_layer_grads* gr, const float* x, const float* v, const float* Z,
                                  const fegnn_layer_saved* sv, const float* gx_new, const float* gxsum_next,
                                  const float* gDsum, const float* gUsum, const float* gu, float* gAv, float* gG1, float* gx,
                                  float* gZ, float* gsv, float* gsg, float* gt, const fegnn_input_grads* ig, void* stream) {
  NO_RECOMPUTE(d);
  return virtual_backward_run(d, g, p, gr, x, v, Z, sv, gx_new, gxsum_next, gDsum, gUsum, gu, gAv, gG1, gx, gZ, gsv, gsg, gt,
                              ig, false, sm_count(), stream);
}

int fegnn_edge_backward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, fegnn_layer_grads* gr,
                        const float* x, const fegnn_layer_saved* sv, const float* gm, const float* gt, float* gP,
                        float* gQ, float* gx, void* stream) {
  return fegnn_edge_backward_inputs(d, g, p, gr, x, sv, gm, gt, gP, gQ, gx, nullptr, stream);
}
// claim: NULL (static tile split) or a zeroed word from which the packed-fp16 kernels claim their tiles; cap: their grid cap
static int edge_backward_run(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, fegnn_layer_grads* gr,
                             const float* x, const fegnn_layer_saved* sv, const float* gm, const float* gt, float* gP,
                             float* gQ, float* gx, const fegnn_input_grads* ig, unsigned* claim, int cap, void* stream) {
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  TRY(check_dims(d));
  TRY(check_flags_params(d, p));
  TRY(check_input_grads(d, ig));
  RQ(g && gr && x && sv && gt && gP && gQ && gx);
  TRY(check_live(d, g, true));
  EdgeArgs a = edge_args(d, g, p, x, sv);
  a.gm = gm; a.gt = gt; a.gP = gP; a.gQ = gQ; a.gx = gx;
  a.g_w1 = gr->edge_w0; a.g_W2 = gr->edge_w2; a.g_b2 = gr->edge_b2;
  a.g_W3 = gr->cr_w0; a.g_b3 = gr->cr_b0; a.g_w4 = gr->cr_w2; a.g_wa = gr->att_w; a.g_ba = gr->att_b;
  const bool zero = !(d->flags & FEGNN_F_PREZEROED);
  if (zero) CK(zero_pair(gP, kH * (size_t)d->N, gQ, kH * (size_t)d->Nl, S(stream)));
  const bool tc_ok = d->Fe <= kTcMaxFe && !(d->flags & FEGNN_F_ATTENTION);
  int mode = g_edge_bwd_mode;
  // FEGNN_F_LIVE_EDGES: modes 1, 2, 4 and 5 were refused above; where 7 / 8 do not apply the fp32 kernel (0) takes their place
  const bool live = d->flags & FEGNN_F_LIVE_EDGES;
  if (mode == 6) mode = (tc_ok && sv->scratch != nullptr) ? 7 : (live ? 0 : 4);      // auto: the packed-fp16 kernel wherever it applies
  if ((mode == 7 || mode == 8) && (!tc_ok || sv->scratch == nullptr)) mode = live ? 0 : 4;
  const bool pre = !(d->flags & FEGNN_F_STATS_READY);      // the bound pre-pass (its statistics came with the layer's other phases)
  if (ig != nullptr && ig->edge_attr != nullptr) {
    // dL/d edge_attr: the kEa instantiations (modes checked above); the output rides in the slots the forward uses for
    // msum / tsum, so the argument block is the default one's
    a.g_ea = ig->edge_attr;
    a.perm = ig->perm;
    if (live) {
      if (tc_ok && sv->scratch != nullptr && mode == 7)
        CK((launch_edge_bwd_tc4<2, true, true>(a, reinterpret_cast<unsigned*>(sv->scratch), cap, S(stream), zero && pre, pre, claim)));
      else
        CK((launch_edge_bwd<true, true>(a, sm_count(), S(stream))));
      return 0;
    }
    if (tc_ok && sv->scratch != nullptr && mode == 7) {
      CK((launch_edge_bwd_tc4<2, true>(a, reinterpret_cast<unsigned*>(sv->scratch), cap, S(stream), zero && pre, pre, claim)));
    } else {
      CK(launch_edge_bwd<true>(a, sm_count(), S(stream)));
    }
    return 0;
  }
  if (live) {
    if (mode == 7) CK((launch_edge_bwd_tc4<2, false, true>(a, reinterpret_cast<unsigned*>(sv->scratch), cap, S(stream), zero && pre, pre, claim)));
    else if (mode == 8) CK((launch_edge_bwd_tc4<4, false, true>(a, reinterpret_cast<unsigned*>(sv->scratch), cap, S(stream), zero && pre, pre, claim)));
    else CK((launch_edge_bwd<false, true>(a, sm_count(), S(stream))));
    return 0;
  }
  if (mode == 7) CK(launch_edge_bwd_tc4<2>(a, reinterpret_cast<unsigned*>(sv->scratch), cap, S(stream), zero && pre, pre, claim));
  else if (mode == 8) CK(launch_edge_bwd_tc4<4>(a, reinterpret_cast<unsigned*>(sv->scratch), cap, S(stream), zero && pre, pre, claim));
  else if (mode == 5 && tc_ok && sv->scratch != nullptr)
    CK(launch_edge_bwd_tc3(a, reinterpret_cast<unsigned*>(sv->scratch), sm_count(), S(stream), zero));
  else if (mode == 2 && tc_ok) CK(launch_edge_bwd_tc2<2>(a, sm_count(), S(stream)));
  else if ((mode == 4 || mode == 5) && tc_ok) CK(launch_edge_bwd_tc2<4>(a, sm_count(), S(stream)));
  else if (mode == 1 && tc_ok) CK(launch_edge_bwd_tc(a, sm_count(), S(stream)));
  else CK(launch_edge_bwd(a, sm_count(), S(stream)));
  return 0;
}
int fegnn_edge_backward_inputs(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, fegnn_layer_grads* gr,
                               const float* x, const fegnn_layer_saved* sv, const float* gm, const float* gt, float* gP,
                               float* gQ, float* gx, const fegnn_input_grads* ig, void* stream) {
  NO_RECOMPUTE(d);
  return edge_backward_run(d, g, p, gr, x, sv, gm, gt, gP, gQ, gx, ig, nullptr, sm_count(), stream);
}

int fegnn_graph_pre_backward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                             fegnn_layer_grads* gr, const float* Sf, const fegnn_layer_saved* sv, const float* gG1,
                             float* gS, float* gZ, float* gxsum, void* stream) {
  NO_RECOMPUTE(d);
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  TRY(check_dims(d));
  RQ(g && p && gr && Sf && sv && gG1 && gS && gZ && gxsum);
  TRY(check_live(d, g, false));
  GraphArgs a = graph_args(d, g, p);
  a.S = Sf; a.M = sv->M; a.Zc = sv->Zc; a.gG1 = gG1; a.gS = gS; a.gZ = gZ; a.gxsum = gxsum;
  a.g_wv1 = gr->edgev_w0;
  CK(launch_graph_pre_bwd(a, S(stream)));
  return 0;
}

int fegnn_node_pre_backward(const fegnn_dims* d, const fegnn_layer_params* p, fegnn_layer_grads* gr, const float* h,
                            const float* gP, const float* gQ, const float* gAv, const float* gUh, const float* gsv,
                            const float* gsg, float* gh, void* stream) {
  return fegnn_node_pre_backward_inputs(d, p, gr, h, gP, gQ, gAv, gUh, gsv, gsg, gh, nullptr, stream);
}
int fegnn_node_pre_backward_inputs(const fegnn_dims* d, const fegnn_layer_params* p, fegnn_layer_grads* gr, const float* h,
                                   const float* gP, const float* gQ, const float* gAv, const float* gUh, const float* gsv,
                                   const float* gsg, float* gh, const fegnn_input_grads* ig, void* stream) {
  NO_RECOMPUTE(d);
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  TRY(check_dims(d));
  TRY(check_flags_params(d, p));
  TRY(check_input_grads(d, ig));
  // dL/da += gUh U1att: the last layer has no Uh (gUh == NULL) and adds nothing
  const bool want_ga = ig != nullptr && ig->node_attr != nullptr && gUh != nullptr;
  RQ(gr && h && gP && gQ && gAv && gsv && gh);
  RQ(!(d->flags & FEGNN_F_GRAVITY) || gsg);
  NodePreArgs a = node_pre_args(d, p, h);
  a.gP = gP; a.gQ = gQ; a.gAv = gAv; a.gUh = gUh; a.gsv = gsv; a.gsg = gsg; a.gh = gh;
  a.g_edge_w0 = gr->edge_w0; a.g_edge_b0 = gr->edge_b0; a.g_edgev_w0 = gr->edgev_w0; a.g_edgev_b0 = gr->edgev_b0;
  a.g_node_w0 = gr->node_w0; a.g_node_b0 = gr->node_b0;
  a.g_vel_w0 = gr->vel_w0; a.g_vel_b0 = gr->vel_b0; a.g_vel_w2 = gr->vel_w2; a.g_vel_b2 = gr->vel_b2;
  a.g_grav_w0 = gr->grav_w0; a.g_grav_b0 = gr->grav_b0; a.g_grav_w2 = gr->grav_w2; a.g_grav_b2 = gr->grav_b2;
  // dU1att = sum_i gUh_i a_i^T rides on the Uh block (none in the last layer: gUh == NULL)
  const NodeAttrArgs at_ = node_attr_args(d, p->node_w0, gr->node_w0);
  const bool attr = d->Fa > 0 && gUh != nullptr;
  if (node_bwd_tc(d->N)) {
    // tcgen05: gh += G_blk W_blk (red.add), dW_blk += G_blk^T h, db_blk += sum G_blk for P, Q, Av [, Uh] and the phi_v
    // [/ phi_g] heads (whose G is recomputed on the tensor core from h)
    dtc::Args t;
    memset(&t, 0, sizeof(t));
    t.N = d->N;
    auto plain = [&](const float* G, const float* W, int ldw, float* gW, float* gb) {
      dtc::Blk& q = t.blk[t.nblk++];
      q.X = G; q.ldx = kH; q.Y = h; q.ldy = kH; q.W = W; q.ldw = ldw; q.wks = 1;
      q.D = gh; q.ldd = kH; q.dmode = 2; q.gW = gW; q.gb = gb;
    };
    auto head = [&](const float* gs, const float* W, const float* hb, const float* hw2, float* gW, float* gb, float* gw2,
                    float* gb2) {
      dtc::Blk& q = t.blk[t.nblk++];
      q.head = 1; q.Y = h; q.ldy = kH; q.W = W; q.ldw = kH; q.wks = 1; q.gs = gs; q.hb = hb; q.hw2 = hw2;
      q.D = gh; q.ldd = kH; q.dmode = 2; q.gW = gW; q.gb = gb; q.g_hw2 = gw2; q.g_hb2 = gb2;
    };
    plain(gP, p->edge_w0, a.ld1, gr->edge_w0, gr->edge_b0);
    plain(gQ, p->edge_w0 + kH, a.ld1, gr->edge_w0 ? gr->edge_w0 + kH : nullptr, nullptr);
    plain(gAv, p->edgev_w0, a.ldv, gr->edgev_w0, gr->edgev_b0);
    dtc::AttrBlk ab;
    ab.at = at_;
    ab.blk = t.nblk;
    if (gUh != nullptr) plain(gUh, p->node_w0, a.ldn, gr->node_w0, gr->node_b0);
    if (!(d->flags & FEGNN_F_RF)) head(gsv, p->vel_w0, p->vel_b0, p->vel_w2, gr->vel_w0, gr->vel_b0, gr->vel_w2, gr->vel_b2);
    if (d->flags & FEGNN_F_GRAVITY)
      head(gsg, p->grav_w0, p->grav_b0, p->grav_w2, gr->grav_w0, gr->grav_b0, gr->grav_w2, gr->grav_b2);
    CK(launch_dense_bwd_tc(t, sm_count(), S(stream), attr ? &ab : nullptr));
  } else {
    CK(launch_node_pre_bwd(a, sm_count(), S(stream), attr ? &at_ : nullptr));
  }
  if (want_ga) CK(launch_input_grad_attr(d->N, d->Fa, at_.ldn, at_.w, gUh, ig->node_attr, S(stream)));
  return 0;
}

int fegnn_edge_length_backward(const fegnn_dims* d, const fegnn_graph* g, const int32_t* rowptr, const float* x,
                               const float* g_ea, float* g_x, void* stream) {
  NO_DET("the col side of the position gradient is a scatter with float atomics");
  TRY(check_dims(d));
  if (d->Fe == 0) return fail(FEGNN_EINVAL, "fegnn_edge_length_backward: the graph has no edge_attr (Fe = 0)");
  RQ(g != nullptr);
  TRY(check_live(d, g, false));
  RQ(d->N == 0 || d->E == 0 || (rowptr && g->col && g->edge_attr && x && g_ea && g_x));
  CK(launch_edge_length_bwd(d->N, d->E, d->Fe, rowptr, g->col, g->edge_attr, x, g_ea,
                            (d->flags & FEGNN_F_LIVE_EDGES) ? g->n_edges : nullptr, g_x, sm_count(), S(stream)));
  return 0;
}

// ------------------------------------------------------------------ halo exchange over peer memory (partitioned path)
int fegnn_halo_push(int32_t n, const int32_t* src_row, const uint64_t* dst_q, const uint64_t* dst_x, const float* Q,
                    const float* x, void* stream) {
  RQ(n >= 0 && (n == 0 || (src_row && dst_q && dst_x && Q && x)));
  CK(launch_halo_push(n, src_row, reinterpret_cast<const unsigned long long*>(dst_q),
                      reinterpret_cast<const unsigned long long*>(dst_x), Q, x, S(stream)));
  return 0;
}
int fegnn_halo_reduce_push(int32_t n, int32_t first_halo_row, const uint64_t* dst_q, const uint64_t* dst_x, const float* gQ,
                           const float* gx, void* stream) {
  NO_DET("remote float atomics");
  RQ(n >= 0 && first_halo_row >= 0 && (n == 0 || (dst_q && dst_x && gQ && gx)));
  CK(launch_halo_reduce_push(n, first_halo_row, reinterpret_cast<const unsigned long long*>(dst_q),
                             reinterpret_cast<const unsigned long long*>(dst_x), gQ, gx, S(stream)));
  return 0;
}

namespace {
int p2p_args(const fegnn_p2p* p, P2PArgs* a) {
  if (p == nullptr) return fail(FEGNN_EINVAL, "fegnn_p2p is null");
  if (p->world < 1 || p->world > kP2PMaxWorld || p->rank < 0 || p->rank >= p->world)
    return fail(FEGNN_EINVAL, "bad rank / world %d / %d (max %d)", p->rank, p->world, kP2PMaxWorld);
  if (!p->epoch || !p->done || !p->err) return fail(FEGNN_EINVAL, "fegnn_p2p local counters are null");
  for (int i = 0; i < kP2PMaxWorld; ++i) {
    a->sig_peer[i] = i < p->world ? p->sig_peer[i] : 0ull;
    a->ar_peer[i] = i < p->world ? p->ar_peer[i] : 0ull;
    if (i < p->world && p->sig_peer[i] == 0) return fail(FEGNN_EINVAL, "signal pad of rank %d is null", i);
  }
  a->epoch = p->epoch; a->done = p->done; a->err = p->err;
  a->rank = p->rank; a->world = p->world; a->ar_capacity = p->ar_capacity;
  return 0;
}
}  // namespace
static_assert(kP2PMaxWorld == FEGNN_P2P_MAX_WORLD && kP2PChannels == FEGNN_P2P_CHANNELS, "fegnn.h and halo.cu disagree");

int fegnn_halo_push_signal(const fegnn_p2p* p, int32_t channel, int32_t n, const int32_t* src_row, int32_t row0,
                           const uint64_t* dst_q, const uint64_t* dst_x, const float* Q, const float* x, void* stream) {
  P2PArgs a;
  TRY(p2p_args(p, &a));
  RQ(channel >= 0 && channel < kP2PChannels && n >= 0 && row0 >= 0 && (n == 0 || (dst_q && dst_x && Q && x)));
  CK(launch_halo_push_signal(a, channel, n, src_row, row0, reinterpret_cast<const unsigned long long*>(dst_q),
                             reinterpret_cast<const unsigned long long*>(dst_x), Q, x, sm_count(), S(stream)));
  return 0;
}
int fegnn_halo_reduce_apply(int32_t n_rows, const int32_t* rows, const int32_t* ptr, const int32_t* slots,
                            const float* recv_q, const float* recv_x, float* gQ, float* gx, void* stream) {
  RQ(n_rows >= 0 && (n_rows == 0 || (rows && ptr && slots && recv_q && recv_x && gQ && gx)));
  CK(launch_halo_reduce_apply(n_rows, rows, ptr, slots, recv_q, recv_x, gQ, gx, S(stream)));
  return 0;
}
int fegnn_p2p_allreduce(const fegnn_p2p* p, int32_t channel, int32_t nseg, float* const* seg_host, const int32_t* count_host,
                        void* stream) {
  NO_DET("multi-GPU reductions are not covered");
  P2PArgs a;
  TRY(p2p_args(p, &a));
  RQ(channel >= 0 && channel < kP2PChannels && nseg >= 1 && nseg <= 4 && seg_host && count_host);
  P2PSegs g;
  memset(&g, 0, sizeof(g));
  long long tot = 0;
  for (int i = 0; i < nseg; ++i) {
    RQ(count_host[i] >= 0 && (count_host[i] == 0 || seg_host[i] != nullptr));
    g.ptr[i] = seg_host[i]; g.count[i] = count_host[i];
    tot += count_host[i];
  }
  g.nseg = nseg;
  if (tot > a.ar_capacity) return fail(FEGNN_ENOMEM, "all-reduce of %lld floats exceeds the slot capacity %d", tot, a.ar_capacity);
  for (int i = 0; i < a.world; ++i) RQ(a.ar_peer[i] != 0);
  CK(launch_p2p_allreduce(a, channel, g, S(stream)));
  return 0;
}

// ------------------------------------------------------------------ FastRF velocity head (models/FastRF.py:76-80,135)
int fegnn_rf_vel_forward(int32_t N, const float* v, const fegnn_layer_params* p, float* sv, void* stream) {
  RQ(N >= 0 && p && (N == 0 || (v && sv)) && p->vel_w0 && p->vel_b0 && p->vel_w2 && p->vel_b2);
  CK(launch_rf_vel_fwd(N, v, p->vel_w0, p->vel_b0, p->vel_w2, p->vel_b2, sv, S(stream)));
  return 0;
}
int fegnn_rf_vel_backward(int32_t N, const float* v, const fegnn_layer_params* p, fegnn_layer_grads* gr, const float* gsv,
                          void* stream) {
  NO_DET("weight gradient flushed by many CTAs with float atomics");
  RQ(N >= 0 && p && gr && (N == 0 || (v && gsv)) && p->vel_w0 && p->vel_b0 && p->vel_w2);
  CK(launch_rf_vel_bwd(N, v, p->vel_w0, p->vel_b0, p->vel_w2, gsv, gr->vel_w0, gr->vel_b0, gr->vel_w2, gr->vel_b2,
                       sm_count(), S(stream)));
  return 0;
}

// ------------------------------------------------------------------ saved block / workspaces
size_t fegnn_layer_saved_floats(const fegnn_dims* d) {
  const size_t N = d->N, Nl = d->Nl, B = d->B, C = d->C;
  return 3 * al4(N * kH) /*P Av Uh*/ + al4(Nl * kH) /*Q*/ + 2 * al4(N) /*sv sg*/ + al4(B * C * C) + al4(B * 3 * C) +
         al4(B * C * kH) /*M Zc G1*/ + al4(N * kH) + al4(N * 3) /*msum tsum*/ + al4(N * C * kH) /*u*/ +
         al4(N * kH) /*zh1*/ + al4(B * 3 * C) + al4(B * C * kH) /*Dsum Usum*/ + 16 /*scratch*/ +
         (C + 2) * 2 * (size_t)(kH * kH) /*wimg*/;
}
int fegnn_layer_saved_bind(const fegnn_dims* d, float* block, fegnn_layer_saved* out) {
  TRY(check_dims(d));
  RQ(block && out);
  const size_t N = d->N, Nl = d->Nl, B = d->B, C = d->C;
  float* p = block;
  auto take = [&](size_t n) { float* r = p; p += al4(n); return r; };
  // accumulators first and contiguous (one zero-fill per layer and step, fegnn_layer_saved_accum_floats words from msum)
  out->msum = take(N * kH); out->tsum = take(N * 3); out->zh1 = take(N * kH);
  out->Dsum = take(B * 3 * C); out->Usum = take(B * C * kH);
  out->scratch = take(16);
  out->P = take(N * kH); out->Av = take(N * kH); out->Uh = take(N * kH); out->Q = take(Nl * kH);
  out->sv = take(N); out->sg = take(N);
  out->M = take(B * C * C); out->Zc = take(B * 3 * C); out->G1 = take(B * C * kH);
  out->u = take(N * C * kH);
  out->wimg = take((C + 2) * 2 * (size_t)(kH * kH));
  return 0;
}
size_t fegnn_layer_saved_accum_floats(const fegnn_dims* d) {
  const size_t N = d->N, B = d->B, C = d->C;
  return al4(N * kH) + al4(N * 3) + al4(N * kH) + al4(B * 3 * C) + al4(B * C * kH) + 16;
}

}  // extern "C"

namespace {

// A stack's workspace as its drivers see it.  What differs between the training stack and the forward-only stack is
// data here, not code in forward_stack.
struct ModelWs {
  // per layer l in [0, L]: state entering layer l (index L = outputs)
  float *h[33], *x[33], *Z[33], *Sx[33], *xsum[33];
  fegnn_layer_saved saved[32];      // layer l's block is block l % nb of a ring of nb <= L blocks
  int nb;
  bool xsum_ahead;                  // the x sums of all states are distinct and contiguous: ONE zero-fill ahead of the chain
  const DetWs* det;                 // the deterministic forms' scratch (forward-only stack), else nullptr: the default kernels
};

void bind_blocks(const fegnn_dims* d, int L, int nb, float* p, ModelWs* w) {
  w->nb = nb < L ? nb : L;
  for (int l = 0; l < L; ++l) {
    if (l < w->nb) {
      fegnn_layer_saved_bind(d, p, &w->saved[l]);
      p += fegnn_layer_saved_floats(d);
    } else {
      w->saved[l] = w->saved[l % w->nb];
    }
  }
}

// saved blocks of the training stack: one per layer, or with FEGNN_F_RECOMPUTE a ring of min(L, 2) (DESIGN 3.8)
inline int model_blocks(const fegnn_dims* d, int L) { return (d->flags & FEGNN_F_RECOMPUTE) ? (L < 2 ? L : 2) : L; }
// one state: h, x, Z, S and the per-graph x sums
size_t state_floats(const fegnn_dims* d) {
  const size_t N = d->N, Nl = d->Nl, B = d->B, C = d->C;
  return al4(N * kH) + al4(Nl * 3) + al4(B * 3 * C) + al4(B * C * kH) + al4(B * 3);
}
size_t model_ws_floats(const fegnn_dims* d, int L) {
  return (size_t)(L + 1) * state_floats(d) + (size_t)model_blocks(d, L) * fegnn_layer_saved_floats(d);
}
void model_ws_bind(const fegnn_dims* d, int L, float* base, ModelWs* w) {
  const size_t N = d->N, Nl = d->Nl, B = d->B, C = d->C;
  float* p = base;
  auto take = [&](size_t n) { float* r = p; p += al4(n); return r; };
  for (int l = 0; l <= L; ++l) w->xsum[l] = take(B * 3);       // contiguous: ONE zero-fill per step for all of them
  for (int l = 0; l <= L; ++l) {
    w->h[l] = take(N * kH); w->x[l] = take(Nl * 3); w->Z[l] = take(B * 3 * C); w->Sx[l] = take(B * C * kH);
  }
  w->xsum_ahead = true;
  w->det = nullptr;
  bind_blocks(d, L, model_blocks(d, L), p, w);
}

// Forward-only stack (rollout / evaluation; utils/train.py:24-27,191-192: validation and test run the model with
// backprop=False).  Nothing is kept for a backward: the layers ping-pong between two state slots and share ONE block of
// per-layer intermediates, so the workspace is 3 states + 1 block instead of (L + 1) states + L blocks (3.4 GB instead of
// 13.4 GB at 1 M nodes, C = 8, L = 4).  Small graphs get a RING of kInferBlocks blocks (a stack of up to that many layers
// has a block per layer): with ONE block the per-graph kernels of layer l + 1 (side stream) must not start before layer
// l's node phase has read u / msum, and the next main-stream kernels not before graph_post(l) has read Dsum / Usum -- a
// join + fork per layer that puts 12 us of one-CTA kernels on the chain -- and every layer needs its accumulator fill and
// its phi_h weight images inside the chain.  With the ring the stack has the training forward's structure: fills and
// weight images ahead of the first kernel, one fork / join pair per layer.  Large graphs keep one block: there all of this
// is noise and the block is gigabytes.
constexpr int kInferRingMaxN = 65536, kInferBlocks = 4;      // 4 = n_layers of every reference main
inline int infer_blocks(const fegnn_dims* d) { return d->N <= kInferRingMaxN ? kInferBlocks : 1; }
void infer_ws_bind(const fegnn_dims* d, int L, float* base, const DetWs* det, ModelWs* w) {
  const size_t N = d->N, Nl = d->Nl, B = d->B, C = d->C;
  float* p = base;
  auto take = [&](size_t n) { float* r = p; p += al4(n); return r; };
  float *h[3], *x[3], *Z[3], *Sx[3], *xsum[3];
  for (int i = 0; i < 3; ++i) {
    h[i] = take(N * kH); x[i] = take(Nl * 3); Z[i] = take(B * 3 * C); Sx[i] = take(B * C * kH); xsum[i] = take(B * 3);
  }
  // slot 2 keeps the embedding state (h0, S0), which FastRF reads in every layer; the layers' outputs alternate 0, 1, 0, ...
  for (int l = 0; l <= L; ++l) {
    const int s = l == 0 ? 2 : (l - 1) & 1;
    w->h[l] = h[s]; w->x[l] = x[s]; w->Z[l] = Z[s]; w->Sx[l] = Sx[s]; w->xsum[l] = xsum[s];
  }
  w->xsum_ahead = false;
  w->det = det;
  bind_blocks(d, L, infer_blocks(d), p, w);
}

struct BwdScratch {
  float *gh, *gx[2], *gZ[2], *gS[2], *gxsum[2], *gDsum, *gUsum, *gzh1, *gm, *gu, *gAv, *gG1[2], *gsv, *gsg, *gt, *gP[2], *gQ[2];
  unsigned* claim[2];                     // the edge backward's tile counter (layer_overlap)
  size_t set_a_floats, set_b_floats;      // [gG1 | gx] and [gP | gQ | claim] of one set, each contiguous (one zero-fill)
};
size_t bwd_scratch_floats(const fegnn_dims* d) {
  const size_t N = d->N, Nl = d->Nl, B = d->B, C = d->C;
  return al4(N * kH) + 2 * al4(Nl * 3) + 2 * al4(B * 3 * C) + 2 * al4(B * C * kH) + 2 * al4(B * 3) + al4(B * 3 * C) +
         al4(B * C * kH) + 2 * al4(N * kH) + al4(N * C * kH) + al4(N * kH) + 2 * al4(B * C * kH) + 2 * al4(N) +
         al4(N * 3) + 2 * (al4(N * kH) + al4(Nl * kH) + 4);
}
void bwd_scratch_bind(const fegnn_dims* d, float* base, BwdScratch* s) {
  const size_t N = d->N, Nl = d->Nl, B = d->B, C = d->C;
  float* p = base;
  auto take = [&](size_t n) { float* r = p; p += al4(n); return r; };
  s->gh = take(N * kH);
  for (int k = 0; k < 2; ++k) { s->gG1[k] = take(B * C * kH); s->gx[k] = take(Nl * 3); }    // set k: [gG1 | gx] contiguous
  s->set_a_floats = al4(B * C * kH) + Nl * 3;
  s->gZ[0] = take(B * 3 * C); s->gZ[1] = take(B * 3 * C);
  s->gS[0] = take(B * C * kH); s->gS[1] = take(B * C * kH);
  s->gxsum[0] = take(B * 3); s->gxsum[1] = take(B * 3);
  s->gDsum = take(B * 3 * C); s->gUsum = take(B * C * kH);
  s->gzh1 = take(N * kH); s->gm = take(N * kH); s->gu = take(N * C * kH);
  s->gAv = take(N * kH);
  s->gsv = take(N); s->gsg = take(N); s->gt = take(N * 3);
  for (int k = 0; k < 2; ++k) {                                                             // set k: [gP | gQ | claim]
    s->gP[k] = take(N * kH); s->gQ[k] = take(Nl * kH); s->claim[k] = reinterpret_cast<unsigned*>(take(4));
  }
  s->set_b_floats = al4(N * kH) + al4(Nl * kH) + 4;
}

// every layer's parameters against the flags, before a stack's first launch
int check_layers(const fegnn_dims* d, int L, const fegnn_layer_params* layers) {
  char why[sizeof(g_err)];
  for (int l = 0; l < L; ++l) {
    if (check_flags_params(d, &layers[l]) == 0) continue;
    memcpy(why, g_err, sizeof(why));
    return fail(FEGNN_EINVAL, "layer %d: %s", l, why);
  }
  return 0;
}

// the dims of layer l's phases in a stack: their full forms (FEGNN_F_RECOMPUTE is the stack's flag), accumulators
// zero-filled by the stack, FEGNN_F_LAST on the last layer and on every FastRF layer (h passes through: models/FastRF.py:186)
fegnn_dims layer_dims(const fegnn_dims* d, int L, int l) {
  fegnn_dims dl = *d;
  dl.flags &= ~(FEGNN_F_RECOMPUTE | FEGNN_F_REBUILD_ALL);
  dl.flags |= FEGNN_F_PREZEROED;
  if ((d->flags & FEGNN_F_RF) || l == L - 1) dl.flags |= FEGNN_F_LAST;
  return dl;
}

// the accumulator head of a saved block (fegnn_layer_saved_accum_floats words from msum)
cudaError_t fill_block(const fegnn_dims* d, const fegnn_layer_saved& sv, cudaStream_t s) {
  return cudaMemsetAsync(sv.msum, 0, sizeof(float) * fegnn_layer_saved_accum_floats(d), s);
}

// phi_h on the tensor cores: the operand-tile images of layers l0 .. l0 + n - 1 into their blocks, in one launch
cudaError_t weight_images(const fegnn_dims* d, const fegnn_layer_params* layers, const ModelWs& w, int l0, int n,
                          cudaStream_t s) {
  const float *w0[32], *w2[32];
  float* img[32];
  for (int l = 0; l < n; ++l) { w0[l] = layers[l0 + l].node_w0; w2[l] = layers[l0 + l].node_w2; img[l] = w.saved[l0 + l].wimg; }
  return launch_node_h_wprep(d->C, ldn(d), n, w0, w2, img, s);
}

// The ring block that layer l reuses, filled on the side stream behind its last readers (a memset node between two kernels
// of the chain would cut their programmatic overlap); the main stream waits for `aux` before layer l (layer_forward)
int ring_fill(const fegnn_dims* d, const fegnn_layer_saved& sv, SideStream* sd) {
  CK(fill_block(d, sv, sd->st));
  CK(cudaEventRecord(sd->aux, sd->st));
  return 0;
}

// Layer l's forward on the main stream, from state l to state l + 1: [the wait for its ring block's fill,] node_pre,
// FastRF's velocity head, the edge forward, the join (the virtual forward reads graph_pre's M and G1), the virtual
// forward, the fork and phi_h.  The caller puts graph_pre on the side stream ahead of it and graph_post (the backward's
// rebuild: graph_post_backward) behind it.  With FEGNN_F_RECOMPUTE in dl the saved-only forms run: x', xsum' and h' are
// state l + 1 already.
int layer_forward(const fegnn_dims* dl, const fegnn_graph* g, const fegnn_layer_params* p, const float* v, ModelWs& w, int l,
                  bool ring_wait, bool node_pre, SideStream* sd, void* stream) {
  cudaStream_t st = S(stream);
  const bool rf = dl->flags & FEGNN_F_RF, saved_only = dl->flags & FEGNN_F_RECOMPUTE;
  fegnn_layer_saved* sv = &w.saved[l];
  if (ring_wait) CK(cudaStreamWaitEvent(st, sd->aux, 0));
  if (node_pre) TRY(node_pre_forward_run(dl, p, w.h[rf ? 0 : l], sv, stream));
  if (rf) TRY(fegnn_rf_vel_forward(dl->N, v, p, sv->sv, stream));
  TRY(edge_forward_run(dl, g, p, w.x[l], sv, w.det, stream));
  JOIN(sd, st);
  TRY(virtual_forward_run(dl, g, p, w.x[l], v, w.Z[l], sv, saved_only ? nullptr : w.x[l + 1],
                          saved_only ? nullptr : w.xsum[l + 1], w.det, stream));
  FORK(sd, st);
  if (!(dl->flags & FEGNN_F_LAST)) TRY(node_h_forward_run(dl, g, p, w.h[l], sv, saved_only ? nullptr : w.h[l + 1], w.det, stream));
  return 0;
}

// The forward of both stacks (fegnn_model_forward, fegnn_model_forward_inference): the prologue, the layer loop and the
// output copies.  The per-graph phases run one CTA per graph on the side stream, under the main chain.
int forward_stack(const fegnn_dims* d, int L, int Fin, const fegnn_graph* g, const fegnn_layer_params* layers,
                  const float* embed_w, const float* embed_b, const float* vnf, const float* node_feat, const float* x0,
                  const float* v, const float* loc_mean, float* x_out, float* Z_out, ModelWs& w, void* stream) {
  cudaStream_t st = S(stream);
  const size_t N = d->N, B = d->B, C = d->C;
  const bool rf = d->flags & FEGNN_F_RF;          // FastRF: h and S of state 0 enter every layer
  const int nb = w.nb;
  TRY(fegnn_embed_forward(d->N, Fin, node_feat, embed_w, embed_b, w.h[0], stream));
  CK(cudaMemcpyAsync(w.x[0], x0, sizeof(float) * 3 * N, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(w.Z[0], loc_mean, sizeof(float) * 3 * C * B, cudaMemcpyDeviceToDevice, st));
  if (B > 0) {
    broadcast_vnf_kernel<<<(unsigned)((B * C * kH + 255) / 256), 256, 0, st>>>(d->B, d->C, vnf, w.Sx[0]); ++g_launches;
    CK(cudaGetLastError());
  }
  // the accumulators are zero-filled ahead of the kernel chain (the phases then skip their own fills): the x sums of every
  // state where the states are distinct, and the accumulator head of every block.  A ring (nb > 1) refills the block of a
  // layer l >= nb on the side stream during layer l - 1; a single block is refilled in the chain in front of each layer.
  if (w.xsum_ahead) CK(cudaMemsetAsync(w.xsum[0], 0, sizeof(float) * ((size_t)L * al4(B * 3) + B * 3), st));
  for (int l = 0; l < nb; ++l) CK(fill_block(d, w.saved[l], st));
  // phi_h on the tensor cores with a ring: the first blocks' weight images in ONE launch here -- weights only, so it runs
  // ahead of the chain and (graph_pending) under the CSR sort -- and layer l + 1 >= nb's on the side stream next to
  // graph_post(l) (its block's images were last read by phi_h of layer l + 1 - nb, ahead of the fork).  A single block:
  // phi_h writes its own images in the chain.
  const bool img_ahead = nb > 1 && g_node_fwd_mode != 0 && !rf;
  const int nimg_top = nb < L - 1 ? nb : L - 1;   // the last layer has no phi_h
  if (img_ahead) CK(weight_images(d, layers, w, 0, nimg_top, st));
  const bool graph_pending = g->ready_event != nullptr;
  if (graph_pending) {
    // the CSR sort is still running on another stream: everything above and the first layer's node phase read no graph
    // array and run under it; this stream joins the sort here
    const fegnn_dims d0 = layer_dims(d, L, 0);
    TRY(node_pre_forward_run(&d0, &layers[0], w.h[0], &w.saved[0], stream));
    CK(cudaStreamWaitEvent(st, static_cast<cudaEvent_t>(g->ready_event), 0));
  }
  if (w.xsum_ahead) CK(launch_graph_xsum(d->N, w.x[0], g->batch, w.xsum[0], st));
  else TRY(graph_xsum_run(d->N, d->B, w.x[0], g->batch, w.xsum[0], w.det, stream));
  SideStream* sd = side_stream();
  RQ(sd != nullptr);
  void* side = sd->st;
  FORK(sd, st);                                   // side: graph_pre(0)
  for (int l = 0; l < L; ++l) {
    fegnn_dims dl = layer_dims(d, L, l);
    if (img_ahead) dl.flags |= FEGNN_F_WIMG_READY;
    const fegnn_layer_params* p = &layers[l];
    fegnn_layer_saved* sv = &w.saved[l];
    const int ls = rf ? 0 : l;                    // layer whose (h, S) state this layer reads
    if (nb == 1 && l > 0) CK(fill_block(d, *sv, st));
    // states in shared slots: the x sums of the state this layer produces, on the side stream (last read by the per-graph
    // kernels of the layer that consumed that slot's state, earlier on the same stream; joined in front of virtual_forward)
    if (!w.xsum_ahead) CK(cudaMemsetAsync(w.xsum[l + 1], 0, sizeof(float) * 3 * B, S(side)));
    TRY(graph_pre_forward_run(&dl, g, p, w.Z[l], w.Sx[ls], w.xsum[l], sv, side));
    TRY(layer_forward(&dl, g, p, v, w, l, nb > 1 && l >= nb, !(graph_pending && l == 0), sd, stream));
    // side: [the fill of the block layer l + 1 reuses,] graph_post(l) [-> graph_pre(l + 1)] under phi_h(l), node_pre(l + 1),
    // edge(l + 1).  The fill's block was last read by layer l + 1 - nb: its node phase on the main stream ahead of the
    // fork, its per-graph kernels earlier on the side stream.
    if (nb > 1 && l + 1 >= nb && l + 1 < L) TRY(ring_fill(d, w.saved[l + 1], sd));
    TRY(graph_post_forward_run(&dl, g, p, w.Z[l], w.Sx[ls], sv, w.Z[l + 1], w.Sx[l + 1], side));
    if (img_ahead && l + 2 < L && l + 1 >= nimg_top) CK(weight_images(d, layers, w, l + 1, 1, S(side)));
    // a single block is rewritten by the next layer: its per-graph kernels (side) must not start before this layer's
    // phi_h (main) has read u / msum, and its main-stream kernels not before this layer's graph_post (side) has read
    // Dsum / Usum.  (Ring: block l % nb is next written by layer l + nb, whose kernels are ordered behind both by the
    // joins in front of the virtual forwards in between.)
    if (nb == 1 && l + 1 < L) {
      JOIN(sd, st);
      FORK(sd, st);
    }
  }
  JOIN(sd, st);
  CK(cudaMemcpyAsync(x_out, w.x[L], sizeof(float) * 3 * N, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(Z_out, w.Z[L], sizeof(float) * 3 * C * B, cudaMemcpyDeviceToDevice, st));
  return 0;
}

}  // namespace

extern "C" {

size_t fegnn_model_workspace_floats(const fegnn_dims* d, int32_t L) { return model_ws_floats(d, L); }
size_t fegnn_model_backward_scratch_floats(const fegnn_dims* d) { return bwd_scratch_floats(d); }

int fegnn_model_forward(const fegnn_dims* d, int32_t L, int32_t Fin, const fegnn_graph* g,
                        const fegnn_layer_params* layers, const float* embed_w, const float* embed_b,
                        const float* vnf, const float* node_feat, const float* x0, const float* v,
                        const float* loc_mean, float* x_out, float* Z_out, float* workspace, size_t workspace_floats,
                        void* stream) {
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  TRY(check_dims(d));
  RQ(L >= 1 && L <= 32 && g && layers && embed_w && embed_b && vnf && workspace && x_out && Z_out);
  RQ(d->Nl == d->N);   // the partitioned path drives the phases itself (halo rows come from peers)
  TRY(check_live(d, g, false));
  if (workspace_floats < model_ws_floats(d, L))
    return fail(FEGNN_ENOMEM, "model workspace %zu < %zu floats", workspace_floats, model_ws_floats(d, L));
  TRY(check_layers(d, L, layers));
  ModelWs w;
  model_ws_bind(d, L, workspace, &w);
  return forward_stack(d, L, Fin, g, layers, embed_w, embed_b, vnf, node_feat, x0, v, loc_mean, x_out, Z_out, w, stream);
}

// ------------------------------------------------------------------ forward-only stack (rollout / evaluation)
size_t fegnn_model_inference_workspace_floats(const fegnn_dims* d) {
  // two ping-pong states + the (h, S) of the embedding (FastRF) + the shared block(s) of per-layer intermediates
  return 3 * state_floats(d) + infer_blocks(d) * fegnn_layer_saved_floats(d);
}
// the deterministic forms' scratch (DetWs), which follows that workspace
size_t fegnn_model_inference_det_workspace_floats(const fegnn_dims* d) {
  return g_det && d != nullptr && check_dims(d) == 0 ? det_ws_floats(d) : 0;
}

int fegnn_model_forward_inference(const fegnn_dims* d, int32_t L, int32_t Fin, const fegnn_graph* g,
                                  const fegnn_layer_params* layers, const float* embed_w, const float* embed_b,
                                  const float* vnf, const float* node_feat, const float* x0, const float* v,
                                  const float* loc_mean, float* x_out, float* Z_out, float* workspace,
                                  size_t workspace_floats, void* stream) {
  TRY(check_dims(d));
  RQ(L >= 1 && L <= 32 && g && layers && embed_w && embed_b && vnf && workspace && x_out && Z_out);
  RQ(d->Nl == d->N);
  TRY(check_live(d, g, false));
  // deterministic mode: the kDet forms of the phases, with their scratch behind the workspace
  const size_t base_floats = fegnn_model_inference_workspace_floats(d);
  const size_t need = base_floats + fegnn_model_inference_det_workspace_floats(d);
  if (workspace_floats < need) return fail(FEGNN_ENOMEM, "inference workspace %zu < %zu floats", workspace_floats, need);
  TRY(check_layers(d, L, layers));
  DetWs det;
  if (g_det) det_ws_bind(d, workspace + base_floats, &det);
  ModelWs w;                                      // FEGNN_F_RECOMPUTE is a training-stack flag: nothing is kept here anyway
  infer_ws_bind(d, L, workspace, g_det ? &det : nullptr, &w);
  return forward_stack(d, L, Fin, g, layers, embed_w, embed_b, vnf, node_feat, x0, v, loc_mean, x_out, Z_out, w, stream);
}

int fegnn_model_backward(const fegnn_dims* d, int32_t L, int32_t Fin, const fegnn_graph* g,
                         const fegnn_layer_params* layers, fegnn_layer_grads* grads, const float* embed_w,
                         float* g_embed_w, float* g_embed_b, float* g_vnf, const float* node_feat, const float* v,
                         const float* gx_out, const float* gZ_out, float* g_x0, float* g_loc_mean,
                         float* g_node_feat, const float* workspace, float* scratch, size_t scratch_floats,
                         void* stream) {
  return fegnn_model_backward_inputs(d, L, Fin, g, layers, grads, embed_w, g_embed_w, g_embed_b, g_vnf, node_feat, v, gx_out,
                                     gZ_out, g_x0, g_loc_mean, g_node_feat, workspace, scratch, scratch_floats, nullptr, stream);
}
int fegnn_model_backward_inputs(const fegnn_dims* d, int32_t L, int32_t Fin, const fegnn_graph* g,
                                const fegnn_layer_params* layers, fegnn_layer_grads* grads, const float* embed_w,
                                float* g_embed_w, float* g_embed_b, float* g_vnf, const float* node_feat, const float* v,
                                const float* gx_out, const float* gZ_out, float* g_x0, float* g_loc_mean,
                                float* g_node_feat, const float* workspace, float* scratch, size_t scratch_floats,
                                const fegnn_input_grads* ig, void* stream) {
  NO_DET("the layer kernels add edge, node and graph sums across CTAs with float atomics");
  TRY(check_dims(d));
  TRY(check_input_grads(d, ig));
  RQ(L >= 1 && L <= 32 && g && layers && grads && embed_w && g_embed_w && g_embed_b && g_vnf && workspace && scratch);
  RQ(gx_out && gZ_out && g_x0 && g_loc_mean && d->Nl == d->N);
  RQ(!(d->flags & FEGNN_F_REBUILD_ALL) || (d->flags & FEGNN_F_RECOMPUTE));
  TRY(check_live(d, g, true));
  if (scratch_floats < bwd_scratch_floats(d))
    return fail(FEGNN_ENOMEM, "backward scratch %zu < %zu floats", scratch_floats, bwd_scratch_floats(d));
  TRY(check_layers(d, L, layers));
  cudaStream_t st = S(stream);
  ModelWs w;
  model_ws_bind(d, L, const_cast<float*>(workspace), &w);
  BwdScratch s;
  bwd_scratch_bind(d, scratch, &s);
  const size_t N = d->N, B = d->B, C = d->C;
  CK(cudaMemsetAsync(s.gh, 0, sizeof(float) * kH * N, st));
  // the requested input gradients are sums over layers: filled here, then every layer adds its term
  if (ig != nullptr) {
    if (ig->node_vel != nullptr) CK(cudaMemsetAsync(ig->node_vel, 0, sizeof(float) * 3 * N, st));
    if (ig->node_attr != nullptr) CK(cudaMemsetAsync(ig->node_attr, 0, sizeof(float) * d->Fa * N, st));
    if (ig->edge_attr != nullptr) CK(cudaMemsetAsync(ig->edge_attr, 0, sizeof(float) * d->Fe * (size_t)d->E, st));
  }
  // [gG1 | gx] and [gP | gQ] exist twice: layer l accumulates into set `cur` while the side stream zero-fills the other set
  // (whose last readers, virtual_backward(l) and node_pre_backward(l + 1), lie before the fork) for layer l - 1 -- no fill
  // stands between two kernels of the main chain
  CK(cudaMemsetAsync(s.gG1[0], 0, sizeof(float) * s.set_a_floats, st));
  CK(cudaMemsetAsync(s.gP[0], 0, sizeof(float) * s.set_b_floats, st));
  const float* gx_new = gx_out;
  const float* gZ_new = gZ_out;
  const float* gS_new = nullptr;
  const float* gxsum_next = nullptr;
  int cur = 0;
  SideStream* sd = side_stream();
  RQ(sd != nullptr);
  void* side = sd->st;
  FORK(sd, st);                                   // side: graph_post_bwd(L-1)
  const bool rf = d->flags & FEGNN_F_RF;
  // FEGNN_F_RECOMPUTE (DESIGN 3.8): layer l's block is block l % 2.  The forward leaves the blocks of layers L - 1 and L - 2
  // complete (unless a backward has run since: FEGNN_F_REBUILD_ALL); every layer below is rebuilt from its input state just
  // before its backward (recompute(l)).  Its accumulator fill, phi_h weight images and graph_pre run on the side stream during
  // backward(l + 1), behind the last readers of the block (backward(l + 2), ahead of the fork in front of graph_pre_bwd(l + 1)).
  // recompute(l) waits for the fill (aux) before its first kernel and for the rest at its join in front of the virtual forward.
  // A backward leaves the ring blocks holding layers 0 / 1, not L - 1 / L - 2: a further backward over the same forward
  // passes FEGNN_F_REBUILD_ALL and then rebuilds those two as well (the top layer's preparation runs ahead of the loop).
  const bool rc = d->flags & FEGNN_F_RECOMPUTE;
  const bool rebuild_all = d->flags & FEGNN_F_REBUILD_ALL;
  const bool rc_img = g_node_fwd_mode != 0 && !rf;
  auto recomputed = [&](int l) { return rc && l >= 0 && (rebuild_all || l + 2 < L); };
  // side stream, ahead of recompute(l): the block's accumulator fill, layer l's phi_h weight images and graph_pre(l)
  auto prepare = [&](int l) -> int {
    const fegnn_dims dp = layer_dims(d, L, l);
    TRY(ring_fill(d, w.saved[l], sd));
    if (rc_img && !(dp.flags & FEGNN_F_LAST)) CK(weight_images(d, layers, w, l, 1, S(side)));
    TRY(graph_pre_forward_run(&dp, g, &layers[l], w.Z[l], w.Sx[rf ? 0 : l], w.xsum[l], &w.saved[l], side));
    return 0;
  };
  if (recomputed(L - 1)) TRY(prepare(L - 1));     // rebuild_all: behind the fork above (the caller's stream order)
  for (int l = L - 1; l >= 0; --l) {
    fegnn_dims dl = layer_dims(d, L, l);
    const bool last = rf || l == L - 1;
    const fegnn_layer_params* p = &layers[l];
    fegnn_layer_grads* gr = &grads[l];
    fegnn_layer_saved* sv = &w.saved[l];
    const int ls = rf ? 0 : l;
    if (recomputed(l)) {
      // recompute(l): node_pre, edge, virtual (u, Dsum, Usum) and phi_h (zh1) forwards of layer l from state l.  graph_post's
      // forward is not rerun: it writes only Z' / S' (state l + 1), and its backward reads S, Usum and the gradients.
      fegnn_dims ds = dl;
      ds.flags |= FEGNN_F_RECOMPUTE;                              // the saved-only forms
      if (rc_img) ds.flags |= FEGNN_F_WIMG_READY;
      TRY(layer_forward(&ds, g, p, v, w, l, true, true, sd, stream));    // its fork: graph_post_bwd(l) reads Usum
    }
    // the edge backward's bound statistics come out of this layer's virtual backward (max|gt|, max|x - x_0|) and node_h
    // backward (max|gm|; the last layer has no gm) when those run on their tensor-core kernels: no pre-pass kernel on the chain
    static const bool stats_fused = getenv("FEGNN_STATS_FUSED") == nullptr || atoi(getenv("FEGNN_STATS_FUSED")) != 0;   // experiment switch
    if (stats_fused && !rf && g_virt_bwd_mode == 1 && !(d->flags & FEGNN_F_ATTENTION) && sv->scratch != nullptr &&
        (last || (node_bwd_tc(d->N) && dense_bwd_uses_rows(d->N, sm_count()))))
      dl.flags |= FEGNN_F_STATS_READY;
    // FastRF: S is one tensor read by every layer, so dL/dS of the layers above passes through (gS = gS_new)
    TRY(fegnn_graph_post_backward(&dl, g, p, gr, w.Sx[ls], sv, gZ_new, gS_new, s.gZ[cur], s.gS[cur], s.gDsum, s.gUsum,
                                  side));                                                   // side, under node_h_bwd
    if (!last) TRY(fegnn_node_h_backward(&dl, g, p, gr, sv, s.gh, s.gzh1, s.gm, s.gu, stream));
    JOIN(sd, st);
    // layer_overlap: gt on this stream, then the virtual backward on `vst` next to the edge backward here (they share
    // only gx, to which both add); vst is joined in front of node_pre_bwd, which reads gAv / gsv / gsg
    // Auto: only where the virtual backward's tiles leave most of a second wave idle (more than one and at most 1.5 waves
    // of one CTA per SM).  In one wave there is no idle wave to fill and the extra launch and events cost (N-body-5: +2 %
    // per step); with more (N-body-100: 1.6 waves, protein batch: 6.9) both kernels fill the machine anyway and the split
    // measured slower than one after the other (B200: +1.0 % / +1.9 %; config 5 at 1 M nodes -1.2 %; DESIGN 3.7).
    const int vtiles = (d->N + kTM / d->C - 1) / (kTM / d->C);
    const bool overlap = virt_bwd_tc(&dl, s.gu) &&
                         (g_layer_overlap == 2 || (g_layer_overlap == 1 && vtiles > sm_count() && 2 * vtiles <= 3 * sm_count()));
    void* vstream = overlap ? static_cast<void*>(sd->vst) : stream;
    // Each kernel takes one CTA per SM and a whole SM's shared memory, so the two share the machine by SMs: the first
    // launched would hold every SM it can fill.  The virtual backward gets `vsms` persistent CTAs, the edge backward the
    // remaining SMs -- in proportion to their SM time (B200, Water-3D: one (node, channel) tile through the heads and trunk
    // kernels costs about as much as 2.9 edge tiles; DESIGN 3.7).
    int vsms = g_overlap_vsms;
    if (overlap && vsms <= 0) {
      const double wv = 2.9 * vtiles, we = (double)((d->E + kTM - 1) / kTM);
      vsms = (int)(sm_count() * wv / (wv + we) + 0.5);
    }
    vsms = min(max(vsms, 1), sm_count() - 1);
    if (overlap) {
      VirtArgs ga = virt_args(&dl, g, p, w.x[l], v, w.Z[l], sv);
      ga.gx_new = gx_new; ga.gxsum_next = gxsum_next; ga.gt = s.gt;
      CK(launch_virtual_bwd_gt(ga, reinterpret_cast<unsigned*>(sv->scratch), st));
      CK(cudaEventRecord(sd->vfork, st));                  // after gt: the set fills forked from vst below overwrite gx_new
      CK(cudaStreamWaitEvent(sd->vst, sd->vfork, 0));
    }
    TRY(virtual_backward_run(&dl, g, p, gr, w.x[l], v, w.Z[l], sv, gx_new, gxsum_next, s.gDsum, last ? nullptr : s.gUsum, s.gu,
                             s.gAv, s.gG1[cur], s.gx[cur], s.gZ[cur], s.gsv, s.gsg, s.gt, ig, overlap,
                             overlap ? vsms : sm_count(), vstream));
    // side: graph_pre_bwd(l) -> graph_post_bwd(l-1), under edge_bwd, node_pre_bwd
    CK(cudaEventRecord(sd->fork, S(vstream)));
    CK(cudaStreamWaitEvent(sd->st, sd->fork, 0));
    TRY(fegnn_graph_pre_backward(&dl, g, p, gr, w.Sx[ls], sv, s.gG1[cur], s.gS[cur], s.gZ[cur], s.gxsum[cur], side));
    if (l > 0) {                                  // side: the other set, for layer l - 1
      CK(cudaMemsetAsync(s.gG1[cur ^ 1], 0, sizeof(float) * s.set_a_floats, S(side)));
      CK(cudaMemsetAsync(s.gP[cur ^ 1], 0, sizeof(float) * s.set_b_floats, S(side)));
    }
    if (recomputed(l - 1)) TRY(prepare(l - 1));   // side: into the block backward(l + 1) has left
    TRY(edge_backward_run(&dl, g, p, gr, w.x[l], sv, last ? nullptr : s.gm, s.gt, s.gP[cur], s.gQ[cur], s.gx[cur], ig,
                          overlap ? s.claim[cur] : nullptr, overlap ? sm_count() - vsms : sm_count(), stream));
    if (overlap) {
      CK(cudaEventRecord(sd->vjoin, sd->vst));
      CK(cudaStreamWaitEvent(st, sd->vjoin, 0));
    }
    if (rf) TRY(fegnn_rf_vel_backward(d->N, v, p, gr, s.gsv, stream));
    TRY(fegnn_node_pre_backward_inputs(&dl, p, gr, w.h[ls], s.gP[cur], s.gQ[cur], s.gAv, last ? nullptr : s.gzh1, s.gsv, s.gsg,
                                       s.gh, ig, stream));
    gx_new = s.gx[cur]; gZ_new = s.gZ[cur]; gS_new = s.gS[cur]; gxsum_next = s.gxsum[cur];
    cur ^= 1;
  }
  // tail: the input-coordinate gradient, dL/d loc_mean and dL/d virtual_node_feat (short kernels on the per-graph results) run
  // on the side stream next to the embedding backward instead of in front of and behind it
  FORK(sd, st);                                   // gx of layer 0 is complete on the main stream (edge, virtual backward)
  if (N > 0) {
    final_gx_kernel<<<(unsigned)((N * 3 + 255) / 256), 256, 0, S(side)>>>(d->N, gx_new, gxsum_next, g->batch, g_x0); ++g_launches;
    CK(cudaGetLastError());
  }
  CK(cudaMemcpyAsync(g_loc_mean, gZ_new, sizeof(float) * 3 * C * B, cudaMemcpyDeviceToDevice, S(side)));
  if (B > 0) {
    reduce_gS_kernel<<<(unsigned)((C * kH + 255) / 256), 256, 0, S(side)>>>(d->B, d->C, gS_new, g_vnf); ++g_launches;
    CK(cudaGetLastError());
  }
  TRY(fegnn_embed_backward(d->N, Fin, node_feat, embed_w, s.gh, g_embed_w, g_embed_b, g_node_feat, stream));
  JOIN(sd, st);
  return 0;
}

// ------------------------------------------------------------------ roofline probes (measurement, not the path)
int fegnn_peak_probe(int32_t kind, int32_t iters, float* sink, double* ops_host, void* stream) {
  RQ(kind >= 0 && kind <= 3 && iters >= 8 && sink && ops_host);
  CK(launch_peak_probe(kind, iters, sink, ops_host, sm_count(), S(stream)));
  return 0;
}

// ------------------------------------------------------------------ unsorted_segment_sum / _mean (models/FastEGNN.py:279-294)
int fegnn_segment_reduce(int64_t E, int32_t K, int32_t S_, const float* data, const int64_t* segment_ids, int32_t mean,
                         float* out, float* count, void* stream) {
  NO_DET("scatter by segment id with float atomics");
  RQ(E >= 0 && K >= 1 && S_ >= 0 && (S_ == 0 || out) && (E == 0 || (data && segment_ids)) && (!mean || S_ == 0 || count));
  CK(launch_segment_reduce(E, K, S_, data, reinterpret_cast<const long long*>(segment_ids), mean != 0, out, count,
                           sm_count(), S(stream)));
  return 0;
}
int fegnn_segment_reduce_backward(int64_t E, int32_t K, int32_t S_, const float* g_out, const int64_t* segment_ids,
                                  const float* count, float* g_data, void* stream) {
  RQ(E >= 0 && K >= 1 && S_ >= 0 && (E == 0 || (g_out && segment_ids && g_data)));
  CK(launch_segment_gather(E, K, S_, g_out, reinterpret_cast<const long long*>(segment_ids), count, g_data, sm_count(),
                           S(stream)));
  return 0;
}

// ------------------------------------------------------------------ optimizer step (utils/train.py:168-170)
int fegnn_adam_step(int64_t n, float* p, const float* g, float* m, float* v, const unsigned char* live, float* step,
                    float lr, double beta1, double beta2, float eps, float weight_decay, void* stream) {
  RQ(n >= 0 && (n & 3) == 0 && step);
  RQ(n == 0 || (p && g && m && v && live));
  RQ(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
       reinterpret_cast<uintptr_t>(v)) & 15) == 0 && (reinterpret_cast<uintptr_t>(live) & 3) == 0);
  CK(launch_adam(n, p, g, m, v, live, step, lr, beta1, beta2, eps, weight_decay, sm_count(), S(stream)));
  return 0;
}

// ------------------------------------------------------------------ MMD
size_t fegnn_loss_workspace_floats(int32_t N, int32_t B) {
  return g_det && N >= 0 && B >= 0 ? loss_det_ws_floats(N, B) : 0;
}
int fegnn_mmd_forward(int32_t B, int32_t C, int32_t ns, float sigma, float scale_vv, float scale_rv, const float* x,
                      const float* Z, const int32_t* sample_idx, float* loss, float* workspace, size_t workspace_floats,
                      void* stream) {
  RQ(B >= 0 && C >= 1 && C <= FEGNN_MAX_C && ns >= 0 && sigma > 0.f && loss && (B == 0 || Z));
  RQ(B == 0 || ns == 0 || (x && sample_idx));
  TRY(check_loss_ws(0, B, workspace, workspace_floats));
  CK(launch_mmd_fwd(B, C, ns, sigma, scale_vv, scale_rv, x, Z, sample_idx, loss, g_det ? workspace : nullptr, S(stream)));
  return 0;
}
int fegnn_mmd_backward(int32_t N, int32_t B, int32_t C, int32_t ns, float sigma, float scale_vv, float scale_rv,
                       const float* x, const float* Z, const int32_t* sample_idx, const float* gloss, float* gx,
                       float* gZ, void* stream) {
  RQ(N >= 0 && B >= 0 && C >= 1 && C <= FEGNN_MAX_C && ns >= 0 && sigma > 0.f && gloss && gx && gZ);
  RQ(B == 0 || (Z && (ns == 0 || (x && sample_idx))));
  CK(launch_mmd_bwd(N, B, C, ns, sigma, scale_vv, scale_rv, x, Z, sample_idx, gloss, gx, gZ, g_det != 0, S(stream)));
  return 0;
}

int fegnn_mse_mmd_forward(int32_t N, int32_t B, int32_t C, int32_t ns, float sigma, float weight, float scale_vv,
                          float scale_rv, float inv_count, const float* x, const float* target, const float* Z,
                          const int32_t* sample_idx, float* out_total, float* out_mse, float* workspace,
                          size_t workspace_floats, void* stream) {
  RQ(N >= 0 && B >= 0 && C >= 1 && C <= FEGNN_MAX_C && ns >= 0 && sigma > 0.f && out_total && out_mse && (B == 0 || Z));
  RQ((N == 0 || (x && target)) && (B == 0 || ns == 0 || (x && sample_idx)));
  TRY(check_loss_ws(N, B, workspace, workspace_floats));
  CK(launch_mse_mmd_fwd(N, B, C, ns, sigma, weight, scale_vv, scale_rv, inv_count, x, target, Z, sample_idx, out_total,
                        out_mse, g_det ? workspace : nullptr, S(stream)));
  return 0;
}
int fegnn_mse_mmd_backward(int32_t N, int32_t B, int32_t C, int32_t ns, float sigma, float weight, float scale_vv,
                           float scale_rv, float inv_count, const float* x, const float* target, const float* Z,
                           const int32_t* sample_idx, const float* g_total, const float* g_mse, float* gx, float* gZ,
                           void* stream) {
  RQ(N >= 0 && B >= 0 && C >= 1 && C <= FEGNN_MAX_C && ns >= 0 && sigma > 0.f && gx && (B == 0 || (Z && gZ)));
  RQ((N == 0 || (x && target)) && (B == 0 || ns == 0 || (x && sample_idx)));
  CK(launch_mse_mmd_bwd(N, B, C, ns, sigma, weight, scale_vv, scale_rv, inv_count, x, target, Z, sample_idx, g_total, g_mse,
                        gx, gZ, g_det != 0, S(stream)));
  return 0;
}

}  // extern "C"
