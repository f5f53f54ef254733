/* fegnn.h -- C ABI of the B200-native FastEGNN layer path (libfegnn.so).
 *
 * The reference (GLAD-RUC/FastEGNN) has no FFI: its "operator interface" for this
 * path is the Python class API of models/FastEGNN.py (FastEGNN.forward :265-276,
 * E_GCL_vel.forward :192-223) plus the MMD block of utils/train.py:111-165.
 * Every entry point below states which reference lines it replaces.  A binding
 * (ctypes) lives in fastegnn_b200/_lib.py; INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the
 *     name ends in _host; `stream` is a cudaStream_t passed as void*.
 *   - no allocation, no synchronisation, no host<->device copies inside any call
 *     (fegnn_graph_prep_* use the caller's workspace); safe for CUDA-graph capture.
 *   - return 0 on success, negative FEGNN_E* otherwise; fegnn_last_error() gives a
 *     thread-local message.
 *   - fp32 everywhere, indices int32 after graph prep (the reference's int64
 *     edge_index / data_batch are converted once by fegnn_graph_prep).
 *   - H (hidden_nf) must be 64; 1 <= C <= FEGNN_MAX_C; 0 <= Fe <= FEGNN_MAX_FE; 0 <= Fa <= FEGNN_MAX_FA.
 *   - "reference layout" = torch.nn.Linear weight [out, in] row-major, the tensors
 *     of the reference state_dict, untouched.  Kernels re-tile them in shared memory.
 */
#ifndef FEGNN_H_
#define FEGNN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FEGNN_H 64
#define FEGNN_MAX_C 16
#define FEGNN_MAX_FE 8
#define FEGNN_MAX_FA 16

#define FEGNN_OK 0
#define FEGNN_EINVAL (-1)   /* bad argument (shape / flag / null pointer)  */
#define FEGNN_ECUDA (-2)    /* a CUDA runtime call or launch failed        */
#define FEGNN_ENOMEM (-3)   /* caller workspace too small                  */

/* flag word (reference ctor kwargs, models/FastEGNN.py:11-12,227-228) */
#define FEGNN_F_ATTENTION 1u
#define FEGNN_F_NORMALIZE 2u
#define FEGNN_F_TANH 4u
#define FEGNN_F_GRAVITY 8u
#define FEGNN_F_LAST 16u      /* last layer of the stack: phi_h / phi_hv outputs are discarded (:276) */
#define FEGNN_F_RF 32u        /* FastRF sibling (models/FastRF.py:6-186): the layer has no phi_h / phi_hv (h and S pass
                                 through every layer unchanged, :186) and phi_v acts on |v_i| (Linear(1,H), :76-80,135):
                                 vel_w0 is [H,1] and the head is evaluated by fegnn_rf_vel_forward / _backward instead
                                 of fegnn_node_pre_*.  Understood by fegnn_node_pre_* and fegnn_model_*.            */

#define FEGNN_F_COORDS_SUM 64u /* E_GCL_vel(coords_agg='sum') (:124-125): d_e * phi_x(m_e) is summed, not averaged, over
                                 the edges of a row.  Understood by fegnn_virtual_forward / _backward (the phase that
                                 applies 1/deg to tsum); FastEGNN itself never sets it (:261).                          */

#define FEGNN_F_NODE_SUM 128u  /* phi_h takes the SUM of a row's messages instead of their mean (the A2A stage of the VNEGNN
                                 sibling, models/VNEGNN.py:85-96).  Understood by fegnn_node_h_forward / _backward.            */

#define FEGNN_F_PREZEROED 256u /* the caller has already zero-filled every accumulator a phase adds into (msum | tsum | zh1 | Dsum |
                                 Usum | scratch of the saved block -- contiguous from .msum, fegnn_layer_saved_accum_floats() words --
                                 xsum_new, gG1, gx, gP, gQ): the phase skips its own fills.  fegnn_model_forward / _backward set it
                                 and issue the fills once per step, off the kernel chain.                                         */
#define FEGNN_F_WIMG_READY 512u /* fegnn_node_h_forward: the weight-block images in saved.wimg are current (written by
                                  fegnn_node_h_weight_images for this layer's parameters): skip the in-call pre-pass */
#define FEGNN_F_STATS_READY 1024u /* fegnn_edge_backward (tensor-core modes 7 / 8): saved.scratch[0..2] already hold the bound
                                    statistics (max|gt|, max|gm|, max|x - x_0|) -- written by fegnn_virtual_backward and
                                    fegnn_node_h_backward of the same layer on their tensor-core kernels: skip the pre-pass */
#define FEGNN_F_RECOMPUTE 2048u /* recompute ("activation checkpointing") for the training stack: fegnn_model_workspace_floats,
                                  fegnn_model_forward and fegnn_model_backward[_inputs] keep the L + 1 layer states and min(L, 2)
                                  saved blocks instead of L; the backward rebuilds a layer's block from its input state just
                                  before that layer's backward (DESIGN 3.8).  On fegnn_virtual_forward / fegnn_node_h_forward it
                                  selects the saved-only forms of a recompute: u, Dsum, Usum (resp. zh1) are written, x',
                                  xsum_new (resp. h') are not (x_new, xsum_new, h_new may be NULL).  Every other per-layer phase
                                  and fegnn_node_h_weight_images return FEGNN_EINVAL with it; fegnn_model_forward_inference
                                  ignores it (it keeps no blocks). */
#define FEGNN_F_REBUILD_ALL 4096u /* with FEGNN_F_RECOMPUTE, read by fegnn_model_backward[_inputs] only: the saved blocks are not as
                                    fegnn_model_forward left them, so rebuild every layer.  A recompute backward rebuilds the
                                    lower layers into the two blocks the forward left holding layers L - 1 and L - 2 (for L >= 3),
                                    so a SECOND backward over the same forward (autograd's retain_graph) must pass this flag, or
                                    it reads the wrong layers' intermediates.  The first backward after a forward may pass it
                                    too (it then also rebuilds the top two layers).  Without FEGNN_F_RECOMPUTE the backward
                                    refuses it with FEGNN_EINVAL; the forward entries ignore it; every other per-layer entry
                                    refuses it like FEGNN_F_RECOMPUTE. */

typedef struct fegnn_dims {
  int32_t N;        /* owned real nodes                                             */
  int32_t Nl;       /* rows of x / Q: owned + halo (== N on one GPU)                */
  int32_t E;        /* directed real edges owned (row < N, col < Nl)                */
  int32_t B;        /* graphs                                                       */
  int32_t C;        /* virtual channels                                             */
  int32_t Fe;       /* edge_attr width                                              */
  uint32_t flags;   /* FEGNN_F_*                                                    */
  float gravity[3]; /* models/FastEGNN.py:258-259                                   */
  float eps;        /* normalize epsilon, :21                                       */
  int32_t Fa;       /* node_attr width (node_attr_nf, :89-93); 0 = no node attributes (FastRF: must be 0) */
  const float* node_attr; /* [N,Fa] fp32, NULL iff Fa == 0: the last Fa columns of node_mlp.0's input (:159), read
                             by fegnn_node_pre_forward / _backward (Uh += U1att a) and the fegnn_model_* entries */
} fegnn_dims;

/* CSR-by-row graph, produced by fegnn_graph_prep (all int32 / fp32, device). */
typedef struct fegnn_graph {
  const int32_t* row;     /* [E] sorted ascending (stable)                          */
  const int32_t* col;     /* [E] col[perm]                                          */
  const int32_t* batch;   /* [N] graph id per node, non-decreasing                  */
  const float* edge_attr; /* [E,Fe] edge_attr[perm]                                 */
  const float* dinv;      /* [N]  1 / max(1, deg_row)        (:294 clamp(min=1))    */
  const float* inv_nb;    /* [B]  1 / max(1, nodes in graph) (global_mean_pool)     */
  void* ready_event;      /* optional cudaEvent_t recorded behind a fegnn_graph_prep that runs on ANOTHER stream: fegnn_model_forward
                             waits for it right before its first use of the arrays above (the embedding and the first layer's
                             node phase run under the sort), fegnn_model_forward_inference at its start; NULL = same stream.
                             Every other entry point ignores it: the caller orders them (ops.CsrGraph.wait)                    */
} fegnn_graph;

/* One layer's parameters in reference layout (models/FastEGNN.py:28-99).
 * att_* may be NULL without FEGNN_F_ATTENTION, gravity_* without FEGNN_F_GRAVITY. */
typedef struct fegnn_layer_params {
  const float *edge_w0, *edge_b0, *edge_w2, *edge_b2;         /* edge_mlp.{0,2}           [H,2H+1+Fe],[H],[H,H],[H] */
  const float *edgev_w0, *edgev_b0, *edgev_w2, *edgev_b2;     /* edge_mlp_virtual.{0,2}   [H,2H+1+C],...            */
  const float *cr_w0, *cr_b0, *cr_w2;                         /* coord_mlp_r.{0,2}        [H,H],[H],[1,H]           */
  const float *crv_w0, *crv_b0, *crv_w2;                      /* coord_mlp_r_virtual                                 */
  const float *cvv_w0, *cvv_b0, *cvv_w2;                      /* coord_mlp_v_virtual                                 */
  const float *vel_w0, *vel_b0, *vel_w2, *vel_b2;             /* coord_mlp_vel.{0,2}      [H,H],[H],[1,H],[1]       */
  const float *grav_w0, *grav_b0, *grav_w2, *grav_b2;         /* gravity_mlp.{0,2}                                   */
  const float *node_w0, *node_b0, *node_w2, *node_b2;         /* node_mlp.{0,2}           [H,2H+H*C+Fa],[H],[H,H],[H] */
  const float *nodev_w0, *nodev_b0, *nodev_w2, *nodev_b2;     /* node_mlp_virtual.{0,2}   [H,2H],[H],[H,H],[H]      */
  const float *att_w, *att_b, *attv_w, *attv_b;               /* att_mlp.0, att_mlp_virtual.0  [1,H],[1]            */
} fegnn_layer_params;
#define FEGNN_LAYER_NPTR 37

/* Same member order; gradients are ACCUMULATED (+=) into these buffers, which the
 * caller zero-fills once per backward.  A NULL member means "no gradient wanted". */
typedef struct fegnn_layer_grads {
  float *edge_w0, *edge_b0, *edge_w2, *edge_b2;
  float *edgev_w0, *edgev_b0, *edgev_w2, *edgev_b2;
  float *cr_w0, *cr_b0, *cr_w2;
  float *crv_w0, *crv_b0, *crv_w2;
  float *cvv_w0, *cvv_b0, *cvv_w2;
  float *vel_w0, *vel_b0, *vel_w2, *vel_b2;
  float *grav_w0, *grav_b0, *grav_w2, *grav_b2;
  float *node_w0, *node_b0, *node_w2, *node_b2;
  float *nodev_w0, *nodev_b0, *nodev_w2, *nodev_b2;
  float *att_w, *att_b, *attv_w, *attv_b;
} fegnn_layer_grads;

/* Per-layer activations kept from forward for backward (all device, caller-owned;
 * fegnn_layer_saved_floats() gives the size of one contiguous block and
 * fegnn_layer_saved_bind() carves it). */
typedef struct fegnn_layer_saved {   /* the accumulators msum, tsum, zh1, Dsum, Usum, scratch lie first and contiguously */
  float *P, *Q, *Av, *Uh;   /* [N,H] [Nl,H] [N,H] [N,H] first-layer products of h        */
  float *sv, *sg;           /* [N] phi_v(h), phi_g(h)                                     */
  float *M, *Zc, *G1;       /* [B,C,C] [B,3,C] [B,C,H] per-graph terms                    */
  float *msum, *tsum;       /* [N,H] [N,3] row sums of m_e and d_e*phi_x(m_e)             */
  float *u;                 /* [N,C,H] real->virtual messages                             */
  float *zh1;               /* [N,H] phi_h pre-activation                                 */
  float *Dsum, *Usum;       /* [B,3,C] [B,C,H] per-graph partial sums (all-reduced when partitioned) */
  float *scratch;           /* [16] words of per-layer kernel scratch (edge backward mode 5: the bound pre-pass)  */
  float *wimg;              /* [(C+2), 2, 64*64] phi_h weight blocks as tcgen05 operand-tile images (3xTF32 hi | lo),
                               rewritten by every fegnn_node_h_forward on the tensor cores (node_forward mode 1 / 3) */
} fegnn_layer_saved;

const char* fegnn_last_error(void);
int fegnn_version(void);   /* 103 (102: before fegnn_dims.Fa / .node_attr; 101: before the "deterministic" mode and the loss forwards' workspace; 100: before
                              fegnn_layer_saved.wimg / fegnn_node_h_weight_images / FEGNN_F_WIMG_READY) */
/* kernels launched by this library so far in this process (host-side counter; bench.py reports it) */
unsigned long long fegnn_launch_count(void);
/* Arithmetic mode of a phase.  "edge_forward": 0 = fp32 FMA kernel, 1 = tcgen05 single-pass TF32 tiles (default),
 * 3 = tcgen05 error-compensated 3xTF32 tiles (fp32-grade).  "edge_backward": 0 = fp32 FMA kernel, 1 = tcgen05 TF32 with
 * shared-memory operands, 2 / 4 = tcgen05 TF32 with tensor-memory A operands and MN-major weight-gradient operands,
 * 256 / 512 threads per 128-edge tile, 5 = tcgen05 kind::f16 (fp16 operands with one power-of-two scale per launch and
 * gradient tensor, fp32 accumulation; same 10-bit mantissa as TF32) with two 128-edge tiles in flight per SM, 7 / 8 = the
 * same operands with packed-fp16 epilogue arithmetic (SiLU on fp16 pairs), 256 / 512 threads per tile, 6 = auto (default):
 * 7 wherever the tensor-core form applies, else 4 / 0.  Layers with attention=True or Fe > 4 always take mode 0 in
 * the backward (Fe > 4 also in the forward).  "virtual_forward" / "virtual_backward": 0 = fp32 FMA kernels, 1 = tcgen05
 * TF32 kernels (default; attention=True layers always take 0).  "node_forward": 0 = fp32 FMA kernels, 3 (default) = fegnn_node_h_forward
 * on tcgen05 error-compensated 3xTF32 tiles (fp32-grade) with fegnn_node_pre_forward on the fp32 FMA kernel, 1 = that plus
 * single-pass tcgen05 TF32 for fegnn_node_pre_forward (opt-in: rounding the unbounded h to TF32 costs equivariant_test.py's
 * atol 1e-4 on its U(0,10) inputs).  "node_backward": 0 = fp32 FMA kernels, 1 = tcgen05 TF32, 2 = auto (default; = 1 today)
 * for fegnn_node_pre_backward and fegnn_node_h_backward (gradients do not enter the forward equivariance).  Process-wide.
 * "deterministic": 0 (default) or 1.  Under 1, fegnn_mmd_forward / _backward and fegnn_mse_mmd_forward / _backward run
 * forms whose every sum has a fixed order: repeated calls with the same inputs on the same device model and SM count give
 * bitwise identical results, whatever the timing (eager or graph replay, other work on other streams, a fresh process);
 * the forwards take a workspace of fegnn_loss_workspace_floats.  fegnn_adam_step, fegnn_graph_prep and the radius graph are deterministic in either mode.
 * fegnn_model_forward_inference runs the same way under 1, with the extra workspace of
 * fegnn_model_inference_det_workspace_floats.
 * Every entry that adds floats across CTAs in arrival order and has no such form -- the layer phases, fegnn_model_forward,
 * fegnn_model_backward[_inputs],
 * fegnn_embed_backward, fegnn_graph_xsum, fegnn_rf_vel_backward, fegnn_segment_reduce, fegnn_halo_reduce_push and
 * fegnn_p2p_allreduce -- returns FEGNN_EINVAL under 1, naming the reason, instead of running.
 * "layer_overlap": 1 (default, auto), 2 or 0; the environment variable FEGNN_LAYER_OVERLAP sets the starting value.
 * Under 2, fegnn_model_backward(_inputs) runs each layer's virtual backward on a second internal stream next to its edge
 * backward (the edge backward's tiles are then claimed dynamically); under 0 the two run one after the other on `stream`;
 * under 1 the first where the virtual backward has more than one and at most 1.5 waves of tiles (one CTA per SM), else
 * the second.  Both arrangements run the same arithmetic; float sums are added in arrival order either way. */
int fegnn_set_mode(const char* phase, int mode);
int fegnn_get_mode(const char* phase);

/* ------------------------------------------------------------------ graph prep
 * Replaces, for the whole stack, what the reference redoes in every layer with
 * int64 gathers / scatter_add (models/FastEGNN.py:182,210,283-294) and
 * global_mean_pool's counting (:148,170,212).  Stable sort of edges by row
 * (== torch.sort(row, stable=True)): perm, rowptr, sorted row/col as int32,
 * gathered edge_attr, clamped inverse degrees and inverse graph sizes.          */
size_t fegnn_graph_prep_workspace_bytes(int32_t N, int32_t E);
int fegnn_graph_prep(int32_t N, int32_t E, int32_t B, int32_t Fe,
                     const int64_t* edge_index /*[2,E]*/, const int64_t* data_batch /*[N]*/,
                     const float* edge_attr /*[E,Fe] or NULL*/,
                     int32_t* perm /*[E]*/, int32_t* rowptr /*[N+1]*/, int32_t* row /*[E]*/, int32_t* col /*[E]*/,
                     int32_t* batch /*[N]*/, int32_t* gptr /*[B+1]*/, float* edge_attr_sorted /*[E,Fe]*/,
                     float* dinv /*[N]*/, float* inv_nb /*[B]*/,
                     void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ graph construction on the device
 * Replaces the step right before the path: torch_cluster.radius_graph + cutoff_edge (torch.sort of the lengths, keep
 * the int(E (1 - cutoff_rate)) shortest) + torch.norm of datasets/simulation/dataset.py:80-82,96-101, the complete-graph
 * / topk variant of datasets/nbody/dataset.py:102-113 (r = +inf) and the contact graph of
 * datasets/protein/dataset.py:146-156,208-213 -- and emits the result directly as the CSR-by-row graph of
 * fegnn_graph_prep (same arrays, same order: rows ascending, inside a row ascending (length, col), which is what a
 * stable sort by row of the reference's length-ordered edge list gives).
 *   candidates: ordered pairs (i,j), i != j, same graph, d2 < r*r, d2 = (dx*dx + dy*dy) + dz*dz in fp32 without FMA;
 *   selection : per graph the int(E_b * keep_frac) first candidates in (length, col, row) order; keep_frac >= 1 keeps all;
 *   edge_attr : every one of the Fe columns holds length = sqrtf(d2)  (dataset edge_attr + utils/train.py:41-43).
 * Two calls, because the edge count is data dependent and nothing here allocates or synchronises:
 *   fegnn_radius_graph_count -> batch / gptr / inv_nb, cand_rowptr [N+1] (exclusive) and *n_cand (device);
 *   the caller reads *n_cand, provides candidate scratch (3 x cand_capacity words) and outputs of out_capacity
 *   entries (out_capacity >= the final edge count, cand_capacity >= *n_cand always suffices), then
 *   fegnn_radius_graph_fill -> rowptr [N+1], row / col / edge_attr / dinv and *n_edges (device).
 * The workspace must be the same, untouched block in both calls. */
size_t fegnn_radius_graph_workspace_bytes(int32_t N, int32_t B);
int fegnn_radius_graph_count(int32_t N, int32_t B, const float* x /*[N,3]*/, const int64_t* data_batch /*[N]*/, float r,
                             int32_t* batch /*[N]*/, int32_t* gptr /*[B+1]*/, float* inv_nb /*[B]*/,
                             int32_t* cand_rowptr /*[N+1]*/, int32_t* n_cand /*[1]*/,
                             void* workspace, size_t workspace_bytes, void* stream);
int fegnn_radius_graph_fill(int32_t N, int32_t B, int32_t Fe, float r, double keep_frac,
                            const int32_t* batch, const int32_t* gptr, const int32_t* cand_rowptr, const int32_t* n_cand,
                            int32_t cand_capacity, int32_t* cand_col, float* cand_dist, int32_t* cand_row,
                            int32_t out_capacity, int32_t* rowptr /*[N+1]*/, int32_t* row, int32_t* col,
                            float* edge_attr /*[out_capacity,Fe]*/, float* dinv /*[N]*/, int32_t* n_edges /*[1]*/,
                            void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ phases of one layer (forward)
 * Names follow oracle/staged.py, which spells the same pipeline out on the CPU.  */

/* embedding_in (models/FastEGNN.py:271) and per-graph coordinate sums for xbar (:212). */
int fegnn_embed_forward(int32_t N, int32_t Fin, const float* node_feat, const float* w /*[H,Fin]*/, const float* b,
                        float* h, void* stream);
int fegnn_embed_backward(int32_t N, int32_t Fin, const float* node_feat, const float* w, const float* gh,
                         float* gw, float* gb, float* gnode_feat /*or NULL*/, void* stream);
int fegnn_graph_xsum(int32_t N, int32_t B, const float* x, const int32_t* batch, float* xsum /*[B,3] zeroed here*/,
                     void* stream);

/* xbar, centred Gram M and G1 = V1s S_c + V1m M[:,c]        (:212-214, per-graph part of :112-115) */
int fegnn_graph_pre_forward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                            const float* Z, const float* S, const float* xsum, fegnn_layer_saved* sv, void* stream);
/* P,Q,Av,Uh and phi_v / phi_g heads: the h-dependent half of every first Linear (:104,115,139,142,162); with Fa > 0
 * Uh also carries the node-attribute term U1att a_i (columns [2H + H*C, 2H + H*C + Fa) of node_mlp.0.weight) */
int fegnn_node_pre_forward(const fegnn_dims* d, const fegnn_layer_params* p, const float* h, fegnn_layer_saved* sv,
                           void* stream);
/* fused real-edge phase: gather, phi_e, phi_x, segment sums by row (:102-108,:125-129,:156) */
int fegnn_edge_forward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* x,
                       fegnn_layer_saved* sv, void* stream);
/* dense N x C real<->virtual phase + new coordinates + per-graph partial sums (:111-119,:133-150) */
int fegnn_virtual_forward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* x,
                          const float* v, const float* Z, fegnn_layer_saved* sv, float* x_new /*[N,3]*/,
                          float* xsum_new /*[B,3]*/, void* stream);
/* phi_h (:153-166) */
int fegnn_node_h_forward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* h,
                         fegnn_layer_saved* sv, float* h_new, void* stream);
/* Operand-tile images (3xTF32 hi | lo, K-major SWIZZLE_128B) of the phi_h weight blocks of nl layers, one launch: layer l
 * reads node_w0 / node_w2 of layers[l] and writes wimg[l] ([(C+2), 2, 64*64] floats, e.g. saved.wimg).  Weights only: a
 * caller may run it once per step next to the kernel chain and pass FEGNN_F_WIMG_READY to fegnn_node_h_forward. */
int fegnn_node_h_weight_images(const fegnn_dims* d, int32_t nl, const fegnn_layer_params* layers, float* const* wimg,
                               void* stream);
/* Z' and S' (:146-150,:168-177) */
int fegnn_graph_post_forward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p, const float* Z,
                             const float* S, const fegnn_layer_saved* sv, float* Z_new, float* S_new, void* stream);

/* ------------------------------------------------------------------ phases of one layer (backward)
 * Hand-written adjoints of the phases above; per-edge / per-(node,channel)
 * activations are recomputed, never stored.                                     */
int fegnn_graph_post_backward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                              fegnn_layer_grads* gr, const float* S, const fegnn_layer_saved* sv,
                              const float* gZ_new, const float* gS_new,
                              float* gZ /*[B,3,C] =*/, float* gS /*[B,C,H] =*/, float* gDsum /*[B,3,C] =*/,
                              float* gUsum /*[B,C,H] =*/, void* stream);
int fegnn_node_h_backward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                          fegnn_layer_grads* gr, const fegnn_layer_saved* sv, const float* gh_new,
                          float* gzh1 /*[N,H] =*/, float* gm /*[N,H] =*/, float* gu /*[N,C,H] =*/, void* stream);
int fegnn_virtual_backward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                           fegnn_layer_grads* gr, const float* x, const float* v, const float* Z,
                           const fegnn_layer_saved* sv, const float* gx_new /*[N,3]*/,
                           const float* gxsum_next /*[B,3] or NULL*/, const float* gDsum, const float* gUsum,
                           const float* gu /*[N,C,H] or NULL; input dL/du from phi_h (ignored with FEGNN_F_LAST).  With
                                             the tensor-core mode a non-NULL buffer is also used as scratch and OVERWRITTEN
                                             (it carries the total dL/du between the two kernels); NULL selects the fp32 kernel*/,
                           float* gAv /*[N,H] =*/, float* gG1 /*[B,C,H] zeroed here, +=*/, float* gx /*[Nl,3] zeroed here, owned rows =*/,
                           float* gZ /*[B,3,C] +=*/, float* gsv /*[N] =*/, float* gsg /*[N] =*/, float* gt /*[N,3] =*/,
                           void* stream);
int fegnn_edge_backward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                        fegnn_layer_grads* gr, const float* x, const fegnn_layer_saved* sv,
                        const float* gm /*[N,H] or NULL*/, const float* gt /*[N,3]*/,
                        float* gP /*[N,H] zeroed here, +=*/, float* gQ /*[Nl,H] zeroed here, +=*/, float* gx /*[Nl,3] +=*/,
                        void* stream);
int fegnn_graph_pre_backward(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                             fegnn_layer_grads* gr, const float* S, const fegnn_layer_saved* sv, const float* gG1,
                             float* gS /*[B,C,H] +=*/, float* gZ /*[B,3,C] +=*/, float* gxsum /*[B,3] =*/, void* stream);
int fegnn_node_pre_backward(const fegnn_dims* d, const fegnn_layer_params* p, fegnn_layer_grads* gr, const float* h,
                            const float* gP, const float* gQ, const float* gAv, const float* gUh /*or NULL*/,
                            const float* gsv, const float* gsg, float* gh /*[N,H] in: dL/dh' (residual), out: dL/dh*/,
                            void* stream);

/* ------------------------------------------------------------------ gradients to the data inputs
 * The reference's autograd reaches node_vel, node_attr and edge_attr (models/FastEGNN.py:104,142,159); these entries add
 * those gradients.  A NULL member is not requested; when nothing is requested the _inputs forms run exactly the kernels
 * of the plain forms, which are these entries called with NULL.
 *   node_vel  [N,3]  : sum over layers of phi_v(h_i) dL/dx'_i (the layer adds phi_v(h) v to x, :142)
 *   node_attr [N,Fa] : sum over the layers with a Uh block (all but the last) of dL/dUh_i U1att
 *   edge_attr [E,Fe] : sum over layers of dL/dz1_e W1[:, 2H+1 ..] (edge_attr enters phi_e's first Linear only, :104), in
 *                      the CALLER's edge order: row perm[e] receives CSR edge e (perm of fegnn_graph_prep), or CSR order
 *                      when perm is NULL (fegnn_radius_graph_fill has no other order)
 * The per-phase forms ADD (+=) their layer's term, one owner per element (no atomics); fegnn_model_backward_inputs fills
 * the requested buffers.  Refused with FEGNN_EINVAL before any launch: node_attr with Fa == 0, edge_attr with Fe == 0,
 * node_vel on FEGNN_F_RF layers (v enters FastRF through |v|), and edge_attr under an "edge_backward" mode whose kernel
 * has no such term (1, 2, 4, 5, 8; modes 0, 6 = auto and 7 have it).  With edge_attr requested, auto and mode 7 take the
 * fp32 kernel (mode 0) wherever the packed-fp16 kernel does not apply (attention, Fe > 4, no saved scratch).          */
typedef struct fegnn_input_grads {
  float* node_vel;       /* [N,3]  or NULL */
  float* node_attr;      /* [N,Fa] or NULL */
  float* edge_attr;      /* [E,Fe] or NULL */
  const int32_t* perm;   /* [E] CSR edge -> caller edge, or NULL (CSR order) */
} fegnn_input_grads;
int fegnn_virtual_backward_inputs(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                                  fegnn_layer_grads* gr, const float* x, const float* v, const float* Z,
                                  const fegnn_layer_saved* sv, const float* gx_new, const float* gxsum_next,
                                  const float* gDsum, const float* gUsum, const float* gu, float* gAv, float* gG1,
                                  float* gx, float* gZ, float* gsv, float* gsg, float* gt,
                                  const fegnn_input_grads* ig /*node_vel +=*/, void* stream);
int fegnn_edge_backward_inputs(const fegnn_dims* d, const fegnn_graph* g, const fegnn_layer_params* p,
                               fegnn_layer_grads* gr, const float* x, const fegnn_layer_saved* sv, const float* gm,
                               const float* gt, float* gP, float* gQ, float* gx,
                               const fegnn_input_grads* ig /*edge_attr +=, perm*/, void* stream);
int fegnn_node_pre_backward_inputs(const fegnn_dims* d, const fegnn_layer_params* p, fegnn_layer_grads* gr,
                                   const float* h, const float* gP, const float* gQ, const float* gAv,
                                   const float* gUh, const float* gsv, const float* gsg, float* gh,
                                   const fegnn_input_grads* ig /*node_attr +=*/, void* stream);

/* ------------------------------------------------------------------ halo exchange over peer memory
 * Multi-GPU form of the layer (one big graph in spatial slabs, fastegnn_b200/partitioned.py): a node is owned by one
 * rank; rows [N, Nl) of Q / x are copies of remote neighbours ("halo").  These two calls move the rows over NVLink
 * with direct peer stores / remote atomics instead of pack + all-to-all + unpack.  dst_q[k] / dst_x[k] are DEVICE
 * ADDRESSES IN THE PEER's mapping of its Q (resp. x) array (torch symmetric memory gives the base pointers), fixed by
 * the partition plan.  Ordering between ranks (a barrier on the stream) is the caller's.
 *   fegnn_halo_push:        for k < n: Q_peer[dst row k] = Q[src_row[k]], x_peer[...] = x[src_row[k]]     (forward)
 *   fegnn_halo_reduce_push: for k < n: Q_owner[dst row k] += gQ[first_halo_row + k], same for gx          (backward) */
int fegnn_halo_push(int32_t n, const int32_t* src_row /*[n]*/, const uint64_t* dst_q /*[n]*/, const uint64_t* dst_x /*[n]*/,
                    const float* Q /*[Nl,H]*/, const float* x /*[Nl,3]*/, void* stream);
int fegnn_halo_reduce_push(int32_t n, int32_t first_halo_row, const uint64_t* dst_q /*[n]*/, const uint64_t* dst_x /*[n]*/,
                           const float* gQ /*[Nl,H]*/, const float* gx /*[Nl,3]*/, void* stream);

/* Second generation: payload + inter-rank ordering in ONE kernel (no NCCL, no separate barrier launch).  Every rank owns
 * a signal pad and a set of all-reduce slots in symmetric memory; fegnn_p2p carries the peers' addresses of both.
 * A call stores its payload into the peers' memory, then its last CTA signals `epoch + 1` to every rank
 * (st.release.sys) and waits for every rank's signal (ld.acquire.sys): when the kernel completes, everything destined for
 * this rank has arrived, and stream order does the rest.  All ranks must issue the same sequence of calls per channel.
 * A wait is bounded (~4 s); on timeout *err becomes 1 + channel and the kernel returns instead of hanging the GPU.
 *   fegnn_halo_push_signal : src_row != NULL -> rows src_row[k] (forward: owners' (Q_j, x_j) into the users' halo rows);
 *                            src_row == NULL -> rows row0 + k (backward: this rank's halo rows of dQ / dx into the OWNER's
 *                            receive buffer, one slot per (user, row): plain stores, no remote atomics).
 *   fegnn_halo_reduce_apply: local; owned boundary row rows[k] adds its received slots[ptr[k] .. ptr[k+1]) in that fixed
 *                            order -> a deterministic reverse halo.
 *   fegnn_p2p_allreduce    : one-shot sum over ranks, IN PLACE, of up to 4 device vectors (total <= ar_capacity floats;
 *                            the <= 2 KB per-graph sums): slot [rank] of every peer is written, signal / wait, then the
 *                            slots are added in rank order, so every rank gets bitwise the same result. */
#define FEGNN_P2P_MAX_WORLD 16
#define FEGNN_P2P_CHANNELS 4
typedef struct fegnn_p2p {
  uint64_t sig_peer[FEGNN_P2P_MAX_WORLD]; /* device address of rank p's signal pad: uint32 [CHANNELS][MAX_WORLD], zeroed once */
  uint64_t ar_peer[FEGNN_P2P_MAX_WORLD];  /* device address of rank p's all-reduce slots: float [2][world][ar_capacity]       */
  uint32_t* epoch;                        /* [CHANNELS] local device counters, zeroed once                                    */
  uint32_t* done;                         /* [CHANNELS] local CTA counters, zeroed once                                       */
  int32_t* err;                           /* [1] local sticky error word                                                      */
  int32_t rank, world, ar_capacity;
} fegnn_p2p;
int fegnn_halo_push_signal(const fegnn_p2p* p, int32_t channel, int32_t n, const int32_t* src_row /*[n] or NULL*/,
                           int32_t row0, const uint64_t* dst_q /*[n]*/, const uint64_t* dst_x /*[n]*/,
                           const float* Q /*[.,H]*/, const float* x /*[.,3]*/, void* stream);
int fegnn_halo_reduce_apply(int32_t n_rows, const int32_t* rows, const int32_t* ptr /*[n_rows+1]*/, const int32_t* slots,
                            const float* recv_q /*[slots,H]*/, const float* recv_x /*[slots,3]*/, float* gQ, float* gx,
                            void* stream);
int fegnn_p2p_allreduce(const fegnn_p2p* p, int32_t channel, int32_t nseg, float* const* seg_host /*[nseg] device ptrs*/,
                        const int32_t* count_host /*[nseg]*/, void* stream);

/* FastRF's velocity head (models/FastRF.py:76-80,135,165): sv_i = w2 . silu(w0 |v_i| + b0) + b2 with
 * |v_i| = sqrt(vx^2 + vy^2 + vz^2) (detached data).  The backward accumulates (+=) into gr->vel_*. */
int fegnn_rf_vel_forward(int32_t N, const float* v /*[N,3]*/, const fegnn_layer_params* p, float* sv /*[N]*/, void* stream);
int fegnn_rf_vel_backward(int32_t N, const float* v, const fegnn_layer_params* p, fegnn_layer_grads* gr,
                          const float* gsv /*[N]*/, void* stream);

/* ------------------------------------------------------------------ whole layer / whole stack
 * fegnn_layer_forward == one E_GCL_vel.forward (:192-223) with S in [B,C,H];
 * fegnn_model_forward == FastEGNN.forward (:265-276) after graph prep; with FEGNN_F_RF in d->flags it is
 * FastRF.forward (models/FastRF.py:228-240): every layer reads the embedding h and the initial S.
 * Workspace layout is private; sizes come from the *_floats queries.            */
size_t fegnn_layer_saved_floats(const fegnn_dims* d);
/* words of the accumulator head of a saved block (from .msum): what FEGNN_F_PREZEROED expects zero-filled */
size_t fegnn_layer_saved_accum_floats(const fegnn_dims* d);
int fegnn_layer_saved_bind(const fegnn_dims* d, float* block, fegnn_layer_saved* out);
/* (L + 1) states + L saved blocks; with FEGNN_F_RECOMPUTE in d->flags (L + 1) states + min(L, 2) saved blocks.  The forward
 * and the backward of one step must see the same flag. */
size_t fegnn_model_workspace_floats(const fegnn_dims* d, int32_t L);
size_t fegnn_model_backward_scratch_floats(const fegnn_dims* d);

int fegnn_model_forward(const fegnn_dims* d, int32_t L, int32_t Fin, const fegnn_graph* g,
                        const fegnn_layer_params* layers_host /*[L]*/, const float* embed_w, const float* embed_b,
                        const float* virtual_node_feat /*[1,H,C] reference layout*/,
                        const float* node_feat /*[N,Fin]*/, const float* x0 /*[N,3]*/, const float* v /*[N,3]*/,
                        const float* loc_mean /*[B,3,C]*/, float* x_out /*[N,3]*/, float* Z_out /*[B,3,C]*/,
                        float* workspace, size_t workspace_floats, void* stream);
/* Forward-only stack for evaluation / rollout (utils/train.py:24-27,191-192: backprop=False): same arguments and results
 * as fegnn_model_forward, but nothing is kept for a backward -- the layers ping-pong between two state sets and share ONE
 * block of per-layer intermediates (workspace = 3 states + 1 block instead of (L + 1) states + L blocks); up to 65 536 nodes
 * a ring of FOUR blocks (layer l uses block l % 4), which takes the per-layer join + fork, the accumulator fills and the
 * phi_h weight images out of the kernel chain.
 * Under the "deterministic" mode the phases run their deterministic forms, which need workspace_floats >= the sum of the two
 * queries below (FEGNN_ENOMEM before any launch otherwise); their scratch lies behind the first query's floats. */
size_t fegnn_model_inference_workspace_floats(const fegnn_dims* d);
/* 0 with the "deterministic" mode off; with it on, the scratch of the deterministic forms (edge tile-boundary row sums, the
 * virtual phase's per-row D sX and the per-graph chunk sums) */
size_t fegnn_model_inference_det_workspace_floats(const fegnn_dims* d);
int fegnn_model_forward_inference(const fegnn_dims* d, int32_t L, int32_t Fin, const fegnn_graph* g,
                                  const fegnn_layer_params* layers_host, const float* embed_w, const float* embed_b,
                                  const float* virtual_node_feat, const float* node_feat, const float* x0, const float* v,
                                  const float* loc_mean, float* x_out, float* Z_out, float* workspace,
                                  size_t workspace_floats, void* stream);
int fegnn_model_backward(const fegnn_dims* d, int32_t L, int32_t Fin, const fegnn_graph* g,
                         const fegnn_layer_params* layers_host, fegnn_layer_grads* grads_host /*[L]*/,
                         const float* embed_w, float* g_embed_w, float* g_embed_b, float* g_virtual_node_feat,
                         const float* node_feat, const float* v,
                         const float* gx_out /*[N,3]*/, const float* gZ_out /*[B,3,C]*/,
                         float* g_x0 /*[N,3]*/, float* g_loc_mean /*[B,3,C]*/, float* g_node_feat /*[N,Fin] or NULL*/,
                         const float* workspace, float* scratch, size_t scratch_floats, void* stream);
/* fegnn_model_backward plus the requested input gradients (fegnn_input_grads above; the buffers are filled here).
 * With FEGNN_F_RECOMPUTE both backward entries rewrite the saved blocks of the workspace (the states are only read). */
int fegnn_model_backward_inputs(const fegnn_dims* d, int32_t L, int32_t Fin, const fegnn_graph* g,
                                const fegnn_layer_params* layers_host, fegnn_layer_grads* grads_host /*[L]*/,
                                const float* embed_w, float* g_embed_w, float* g_embed_b, float* g_virtual_node_feat,
                                const float* node_feat, const float* v, const float* gx_out, const float* gZ_out,
                                float* g_x0, float* g_loc_mean, float* g_node_feat, const float* workspace, float* scratch,
                                size_t scratch_floats, const fegnn_input_grads* ig, void* stream);

/* ------------------------------------------------------------------ MMD regulariser
 * utils/train.py:17-20,111-165 with the random sample made explicit:
 * sample_idx[b*ns + s] is a GLOBAL node index (graph offset already added).
 * loss = scale_vv * (1/(B C^2)) sum k(Z_bc,Z_bc') - scale_rv * (2/(B ns C)) sum k(x_s, Z_bc),
 * k(p,q) = exp(-|p-q| / (2 sigma^2)).  scale_vv = scale_rv = 1 is the reference; the partitioned
 * path evaluates the Z-only term on one rank (scale_vv = 0 elsewhere) and weights each rank's share of
 * the samples (scale_rv = ns_local / ns_total; ns == 0 is allowed).
 * Under the "deterministic" mode the forward keeps one partial per CTA in `workspace` (at least
 * fegnn_loss_workspace_floats(N, B) floats; pass N = 0 for fegnn_mmd_forward) and the backward is bitwise reproducible
 * provided no node index is sampled by two different graphs (sampling within each graph, as the reference does).  With
 * the mode off the query returns 0 and workspace may be NULL.                                                      */
size_t fegnn_loss_workspace_floats(int32_t N, int32_t B);
int fegnn_mmd_forward(int32_t B, int32_t C, int32_t ns, float sigma, float scale_vv, float scale_rv,
                      const float* x /*[N,3]*/, const float* Z /*[B,3,C]*/, const int32_t* sample_idx,
                      float* loss /*[1] zeroed here*/, float* workspace, size_t workspace_floats, void* stream);
int fegnn_mmd_backward(int32_t N, int32_t B, int32_t C, int32_t ns, float sigma, float scale_vv, float scale_rv,
                       const float* x, const float* Z, const int32_t* sample_idx, const float* gloss /*[1]*/,
                       float* gx /*[N,3] zeroed here*/, float* gZ /*[B,3,C] =*/, void* stream);

/* The step's loss (utils/train.py:104,163): total = MSE + weight * MMD in one kernel per direction.
 *   MSE = inv_count * sum (x - target)^2  (inv_count = 1 / (3 N) is torch's mean; a partitioned caller passes 1 / (3 N_global)),
 *   MMD as above.  out_total[0], out_mse[0] (the MSE term alone, what the reference logs at :107) are zeroed here.
 * Backward: g_total / g_mse = dL/d(total), dL/d(mse) (device scalars, either may be NULL);
 *   gx [N,3] (zeroed here) = (g_total + g_mse) * 2 inv_count (x - target) + g_total * weight * dMMD/dx ; gZ [B,3,C] =. */
int fegnn_mse_mmd_forward(int32_t N, int32_t B, int32_t C, int32_t ns, float sigma, float weight, float scale_vv,
                          float scale_rv, float inv_count, const float* x, const float* target, const float* Z,
                          const int32_t* sample_idx, float* out_total, float* out_mse, float* workspace,
                          size_t workspace_floats, void* stream);
int fegnn_mse_mmd_backward(int32_t N, int32_t B, int32_t C, int32_t ns, float sigma, float weight, float scale_vv,
                           float scale_rv, float inv_count, const float* x, const float* target, const float* Z,
                           const int32_t* sample_idx, const float* g_total, const float* g_mse, float* gx, float* gZ,
                           void* stream);

/* ------------------------------------------------------------------ roofline probes (measurement only)
 * One launch of a micro-benchmark for the pipe a kernel of the path is bound by: kind 0 = tcgen05.mma kind::tf32
 * (cta_group::1, M128 N256 K8, shared-memory operands), 1 = tcgen05.mma kind::f16 (K16), 2 = fp32 FMA, 3 = MUFU
 * tanh.approx.  `iters` instructions per issuing thread; *ops_host (HOST pointer) receives the flops (kinds 0-2) or MUFU
 * results (kind 3) of the launch.  The caller times the launch with CUDA events (bench.py: peak_*_measured). */
int fegnn_peak_probe(int32_t kind, int32_t iters, float* sink /*[1] device*/, double* ops_host, void* stream);

/* ------------------------------------------------------------------ segment helpers exported by the reference file
 * unsorted_segment_sum (models/FastEGNN.py:279-284) and unsorted_segment_mean (:287-294) on int64 segment ids, as the
 * reference passes them: out [S,K] (zeroed here) = sum of data rows [E,K] per segment; mean != 0 additionally divides by
 * the per-segment row count clamped to >= 1 (count [S] is written).  The backward gathers g_out rows back to the edges
 * (divided by the same clamped count when count != NULL).  The fused edge kernels do NOT go through these. */
int fegnn_segment_reduce(int64_t E, int32_t K, int32_t S, const float* data /*[E,K]*/, const int64_t* segment_ids /*[E]*/,
                         int32_t mean, float* out /*[S,K]*/, float* count /*[S] or NULL when mean == 0*/, void* stream);
int fegnn_segment_reduce_backward(int64_t E, int32_t K, int32_t S, const float* g_out /*[S,K]*/,
                                  const int64_t* segment_ids, const float* count /*[S] or NULL*/, float* g_data /*[E,K]*/,
                                  void* stream);

/* ------------------------------------------------------------------ optimizer step
 * torch.optim.Adam (amsgrad=False, maximize=False; utils/train.py:168-170, main_*.py optimizer construction) over ONE
 * flat buffer: n floats (multiple of 4, 16-byte aligned pointers).  live[i] == 0 marks elements of parameters that
 * received no gradient this step (torch skips such parameters).  `step` is a device float, incremented here.        */
int fegnn_adam_step(int64_t n, float* p, const float* g, float* m, float* v, const unsigned char* live /*[n]*/,
                    float* step /*[1] device*/, float lr, double beta1, double beta2, float eps, float weight_decay,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FEGNN_H_ */
