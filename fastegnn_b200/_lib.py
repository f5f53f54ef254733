"""ctypes binding of libfegnn.so (the C ABI declared in include/fegnn.h).

The library is the product: there is no CPU path and no torch fallback.  Importing this
module without the built shared object raises immediately; calling any entry point on a
machine without a CUDA device fails inside the CUDA runtime and is reported as an error.
"""
from __future__ import annotations

import ctypes as C
import os
import warnings

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FEGNN_LIB") or os.path.join(HERE, "_C", "libfegnn.so")     # FEGNN_LIB: an instrumented build (tools/)

H = 64
MAX_C = 16
MAX_FE = 8
MAX_FA = 16

F_ATTENTION, F_NORMALIZE, F_TANH, F_GRAVITY, F_LAST, F_RF, F_COORDS_SUM, F_NODE_SUM, F_PREZEROED = 1, 2, 4, 8, 16, 32, 64, 128, 256
F_RECOMPUTE = 2048          # training stack: two saved blocks, each layer's rebuilt in the backward (DESIGN 3.8)
F_REBUILD_ALL = 4096        # with F_RECOMPUTE: a backward after another one over the same forward rebuilds every layer
F_LIVE_EDGES = 8192         # fegnn_dims.E is a capacity; the live edge count is the device word fegnn_graph.n_edges
# sticky status bits of fegnn_graph_prep_live / fegnn_radius_graph_fill_live
LIVE_BAD_COUNT, LIVE_CAND_OVERFLOW, LIVE_EDGE_OVERFLOW = 1, 2, 4

fp = C.POINTER(C.c_float)
ip = C.POINTER(C.c_int32)
lp = C.POINTER(C.c_int64)


class Dims(C.Structure):
    _fields_ = [("N", C.c_int32), ("Nl", C.c_int32), ("E", C.c_int32), ("B", C.c_int32), ("C", C.c_int32),
                ("Fe", C.c_int32), ("flags", C.c_uint32), ("gravity", C.c_float * 3), ("eps", C.c_float),
                ("Fa", C.c_int32), ("node_attr", C.c_void_p)]


class Graph(C.Structure):
    _fields_ = [("row", C.c_void_p), ("col", C.c_void_p), ("batch", C.c_void_p), ("edge_attr", C.c_void_p),
                ("dinv", C.c_void_p), ("inv_nb", C.c_void_p), ("ready_event", C.c_void_p), ("n_edges", C.c_void_p)]


# member order of fegnn_layer_params / fegnn_layer_grads -> reference state_dict suffix
LAYER_FIELDS = [
    ("edge_w0", "edge_mlp.0.weight"), ("edge_b0", "edge_mlp.0.bias"),
    ("edge_w2", "edge_mlp.2.weight"), ("edge_b2", "edge_mlp.2.bias"),
    ("edgev_w0", "edge_mlp_virtual.0.weight"), ("edgev_b0", "edge_mlp_virtual.0.bias"),
    ("edgev_w2", "edge_mlp_virtual.2.weight"), ("edgev_b2", "edge_mlp_virtual.2.bias"),
    ("cr_w0", "coord_mlp_r.0.weight"), ("cr_b0", "coord_mlp_r.0.bias"), ("cr_w2", "coord_mlp_r.2.weight"),
    ("crv_w0", "coord_mlp_r_virtual.0.weight"), ("crv_b0", "coord_mlp_r_virtual.0.bias"),
    ("crv_w2", "coord_mlp_r_virtual.2.weight"),
    ("cvv_w0", "coord_mlp_v_virtual.0.weight"), ("cvv_b0", "coord_mlp_v_virtual.0.bias"),
    ("cvv_w2", "coord_mlp_v_virtual.2.weight"),
    ("vel_w0", "coord_mlp_vel.0.weight"), ("vel_b0", "coord_mlp_vel.0.bias"),
    ("vel_w2", "coord_mlp_vel.2.weight"), ("vel_b2", "coord_mlp_vel.2.bias"),
    ("grav_w0", "gravity_mlp.0.weight"), ("grav_b0", "gravity_mlp.0.bias"),
    ("grav_w2", "gravity_mlp.2.weight"), ("grav_b2", "gravity_mlp.2.bias"),
    ("node_w0", "node_mlp.0.weight"), ("node_b0", "node_mlp.0.bias"),
    ("node_w2", "node_mlp.2.weight"), ("node_b2", "node_mlp.2.bias"),
    ("nodev_w0", "node_mlp_virtual.0.weight"), ("nodev_b0", "node_mlp_virtual.0.bias"),
    ("nodev_w2", "node_mlp_virtual.2.weight"), ("nodev_b2", "node_mlp_virtual.2.bias"),
    ("att_w", "att_mlp.0.weight"), ("att_b", "att_mlp.0.bias"),
    ("attv_w", "att_mlp_virtual.0.weight"), ("attv_b", "att_mlp_virtual.0.bias"),
]
assert len(LAYER_FIELDS) == 37


class LayerPtrs(C.Structure):
    """fegnn_layer_params and fegnn_layer_grads share this layout (const-ness aside)."""
    _fields_ = [(n, C.c_void_p) for n, _ in LAYER_FIELDS]


class InputGrads(C.Structure):
    """fegnn_input_grads: requested gradients to node_vel [N,3], node_attr [N,Fa], edge_attr [E,Fe] (NULL = not requested)
    and the CSR -> caller edge order map (NULL = CSR order)."""
    _fields_ = [("node_vel", C.c_void_p), ("node_attr", C.c_void_p), ("edge_attr", C.c_void_p), ("perm", C.c_void_p)]


SAVED_FIELDS = ["P", "Q", "Av", "Uh", "sv", "sg", "M", "Zc", "G1", "msum", "tsum", "u", "zh1", "Dsum", "Usum", "scratch", "wimg"]


class Saved(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in SAVED_FIELDS]


P2P_MAX_WORLD, P2P_CHANNELS = 16, 4


class P2P(C.Structure):
    """fegnn_p2p: peers' signal pads / all-reduce slots (symmetric memory) + this rank's local counters."""
    _fields_ = [("sig_peer", C.c_uint64 * P2P_MAX_WORLD), ("ar_peer", C.c_uint64 * P2P_MAX_WORLD),
                ("epoch", C.c_void_p), ("done", C.c_void_p), ("err", C.c_void_p),
                ("rank", C.c_int32), ("world", C.c_int32), ("ar_capacity", C.c_int32)]


class FegnnError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  fastegnn_b200 has no CPU or eager fallback.")
    return C.CDLL(LIB_PATH)


lib = _load()

vp = C.c_void_p
i32 = C.c_int32
_PD, _PG, _PP, _PS = C.POINTER(Dims), C.POINTER(Graph), C.POINTER(LayerPtrs), C.POINTER(Saved)
_PI = C.POINTER(InputGrads)

SIGNATURES = {
    "fegnn_last_error": (C.c_char_p, []),
    "fegnn_version": (C.c_int, []),
    "fegnn_launch_count": (C.c_ulonglong, []),
    "fegnn_set_mode": (C.c_int, [C.c_char_p, C.c_int]),
    "fegnn_get_mode": (C.c_int, [C.c_char_p]),
    "fegnn_graph_prep_workspace_bytes": (C.c_size_t, [i32, i32]),
    "fegnn_graph_prep": (C.c_int, [i32, i32, i32, i32] + [vp] * 12 + [vp, C.c_size_t, vp]),
    "fegnn_graph_prep_live": (C.c_int, [i32, i32, i32, i32] + [vp] * 12 + [vp, C.c_size_t, vp, vp, vp, vp]),
    "fegnn_radius_graph_workspace_bytes": (C.c_size_t, [i32, i32]),
    "fegnn_radius_graph_count": (C.c_int, [i32, i32, vp, vp, C.c_float, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]),
    "fegnn_radius_graph_fill": (C.c_int, [i32, i32, i32, C.c_float, C.c_double, vp, vp, vp, vp, i32, vp, vp, vp, i32,
                                          vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]),
    "fegnn_radius_graph_fill_live": (C.c_int, [i32, i32, i32, C.c_float, C.c_double, vp, vp, vp, vp, i32, vp, vp, vp, i32,
                                               vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]),
    "fegnn_embed_forward": (C.c_int, [i32, i32, vp, vp, vp, vp, vp]),
    "fegnn_embed_backward": (C.c_int, [i32, i32, vp, vp, vp, vp, vp, vp, vp]),
    "fegnn_graph_xsum": (C.c_int, [i32, i32, vp, vp, vp, vp]),
    "fegnn_graph_pre_forward": (C.c_int, [_PD, _PG, _PP, vp, vp, vp, _PS, vp]),
    "fegnn_node_pre_forward": (C.c_int, [_PD, _PP, vp, _PS, vp]),
    "fegnn_edge_forward": (C.c_int, [_PD, _PG, _PP, vp, _PS, vp]),
    "fegnn_virtual_forward": (C.c_int, [_PD, _PG, _PP, vp, vp, vp, _PS, vp, vp, vp]),
    "fegnn_node_h_forward": (C.c_int, [_PD, _PG, _PP, vp, _PS, vp, vp]),
    "fegnn_node_h_weight_images": (C.c_int, [_PD, i32, _PP, C.POINTER(C.c_void_p), vp]),
    "fegnn_graph_post_forward": (C.c_int, [_PD, _PG, _PP, vp, vp, _PS, vp, vp, vp]),
    "fegnn_graph_post_backward": (C.c_int, [_PD, _PG, _PP, _PP, vp, _PS, vp, vp, vp, vp, vp, vp, vp]),
    "fegnn_node_h_backward": (C.c_int, [_PD, _PG, _PP, _PP, _PS, vp, vp, vp, vp, vp]),
    "fegnn_virtual_backward": (C.c_int, [_PD, _PG, _PP, _PP, vp, vp, vp, _PS] + [vp] * 12 + [vp]),
    "fegnn_edge_backward": (C.c_int, [_PD, _PG, _PP, _PP, vp, _PS, vp, vp, vp, vp, vp, vp]),
    "fegnn_graph_pre_backward": (C.c_int, [_PD, _PG, _PP, _PP, vp, _PS, vp, vp, vp, vp, vp]),
    "fegnn_node_pre_backward": (C.c_int, [_PD, _PP, _PP, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "fegnn_virtual_backward_inputs": (C.c_int, [_PD, _PG, _PP, _PP, vp, vp, vp, _PS] + [vp] * 12 + [_PI, vp]),
    "fegnn_edge_backward_inputs": (C.c_int, [_PD, _PG, _PP, _PP, vp, _PS, vp, vp, vp, vp, vp, _PI, vp]),
    "fegnn_node_pre_backward_inputs": (C.c_int, [_PD, _PP, _PP, vp, vp, vp, vp, vp, vp, vp, vp, _PI, vp]),
    "fegnn_edge_length_backward": (C.c_int, [_PD, _PG, vp, vp, vp, vp, vp]),
    "fegnn_halo_push": (C.c_int, [i32, vp, vp, vp, vp, vp, vp]),
    "fegnn_halo_reduce_push": (C.c_int, [i32, i32, vp, vp, vp, vp, vp]),
    "fegnn_halo_push_signal": (C.c_int, [C.POINTER(P2P), i32, i32, vp, i32, vp, vp, vp, vp, vp]),
    "fegnn_halo_reduce_apply": (C.c_int, [i32, vp, vp, vp, vp, vp, vp, vp, vp]),
    "fegnn_p2p_allreduce": (C.c_int, [C.POINTER(P2P), i32, i32, C.POINTER(C.c_void_p), C.POINTER(C.c_int32), vp]),
    "fegnn_rf_vel_forward": (C.c_int, [i32, vp, _PP, vp, vp]),
    "fegnn_rf_vel_backward": (C.c_int, [i32, vp, _PP, _PP, vp, vp]),
    "fegnn_layer_saved_floats": (C.c_size_t, [_PD]),
    "fegnn_layer_saved_accum_floats": (C.c_size_t, [_PD]),
    "fegnn_layer_saved_bind": (C.c_int, [_PD, vp, _PS]),
    "fegnn_model_workspace_floats": (C.c_size_t, [_PD, i32]),
    "fegnn_model_backward_scratch_floats": (C.c_size_t, [_PD]),
    "fegnn_model_forward": (C.c_int, [_PD, i32, i32, _PG, _PP] + [vp] * 9 + [vp, C.c_size_t, vp]),
    "fegnn_model_inference_workspace_floats": (C.c_size_t, [_PD]),
    "fegnn_model_inference_det_workspace_floats": (C.c_size_t, [_PD]),
    "fegnn_model_forward_inference": (C.c_int, [_PD, i32, i32, _PG, _PP] + [vp] * 9 + [vp, C.c_size_t, vp]),
    "fegnn_model_backward": (C.c_int, [_PD, i32, i32, _PG, _PP, _PP] + [vp] * 11 + [vp, vp, C.c_size_t, vp]),
    "fegnn_model_backward_inputs": (C.c_int, [_PD, i32, i32, _PG, _PP, _PP] + [vp] * 11 + [vp, vp, C.c_size_t, _PI, vp]),
    "fegnn_peak_probe": (C.c_int, [i32, i32, vp, C.POINTER(C.c_double), vp]),
    "fegnn_segment_reduce": (C.c_int, [C.c_int64, i32, i32, vp, vp, i32, vp, vp, vp]),
    "fegnn_segment_reduce_backward": (C.c_int, [C.c_int64, i32, i32, vp, vp, vp, vp, vp]),
    "fegnn_adam_step": (C.c_int, [C.c_int64, vp, vp, vp, vp, vp, vp, C.c_float, C.c_double, C.c_double, C.c_float, C.c_float, vp]),
    "fegnn_loss_workspace_floats": (C.c_size_t, [i32, i32]),
    "fegnn_mmd_forward": (C.c_int, [i32, i32, i32, C.c_float, C.c_float, C.c_float, vp, vp, vp, vp, vp, C.c_size_t, vp]),
    "fegnn_mmd_backward": (C.c_int, [i32, i32, i32, i32, C.c_float, C.c_float, C.c_float, vp, vp, vp, vp, vp, vp, vp]),
    "fegnn_mse_mmd_forward": (C.c_int, [i32, i32, i32, i32] + [C.c_float] * 5 + [vp] * 7 + [C.c_size_t, vp]),
    "fegnn_mse_mmd_backward": (C.c_int, [i32, i32, i32, i32] + [C.c_float] * 5 + [vp] * 9),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)      # AttributeError here == the .so does not export what fegnn.h declares
    _fn.restype = _res
    _fn.argtypes = _args


def set_mode(phase: str, mode: int) -> None:
    """0 = fp32 FMA kernels, 1 = tcgen05 TF32, 3 = tcgen05 3xTF32, ... (see fegnn_set_mode in fegnn.h)."""
    check(lib.fegnn_set_mode(phase.encode(), int(mode)), "fegnn_set_mode")


PHASES = ("edge_forward", "edge_backward", "virtual_forward", "virtual_backward", "node_forward", "node_backward")


def set_precision(name: str) -> None:
    """"fp32": every phase on the fp32 FMA kernels (tight parity).  "tf32" (default): the fused edge phase and the
    dense real<->virtual phase run on tcgen05 TF32 tiles, forward and backward (stated tolerance, see DESIGN.md); phi_h of
    the forward runs on tcgen05 3xTF32 tiles (fp32-grade).
    "tf32x3": TF32 backward, fp32-grade forward (3xTF32 edge and phi_h tiles, fp32 FMA virtual and node_pre phases).
    "tf32_all": "tf32" plus the tcgen05 node_pre forward (h rounded to TF32: fastest, but equivariance only to ~3e-4 on
    equivariant_test.py's inputs)."""
    table = {"fp32": (0, 0, 0, 0, 0, 0), "tf32": (1, 6, 1, 1, 3, 2), "tf32x3": (3, 6, 0, 1, 3, 2), "tf32_all": (1, 6, 1, 1, 1, 2)}
    for phase, mode in zip(PHASES, table[name]):
        set_mode(phase, mode)


def get_mode(phase: str) -> int:
    return int(lib.fegnn_get_mode(phase.encode()))


# Why the layer stack has no deterministic form (DESIGN.md section 9): FastEGNN, FastRF, VNEGNN, E_GCL_vel, the partitioned
# runner and the segment helpers all reach kernels that add floats across CTAs in arrival order.
NO_DET_LAYERS = "its edge, virtual and node kernels add sums across CTAs with float atomics"


def deterministic(what: str, missing: str = None) -> bool:
    """Sets the library's "deterministic" mode from torch.are_deterministic_algorithms_enabled() for one call of `what`
    and returns the mode the call runs in.  `missing` says why `what` has no deterministic form (None: it has one).  Such
    a call raises under the flag, as torch's own ops do, or warns and runs as without the flag under warn_only=True."""
    on = torch.are_deterministic_algorithms_enabled()
    if on and missing is not None:
        msg = (f"{what} does not have a deterministic implementation ({missing}), but you set "
               "'torch.use_deterministic_algorithms(True)'.  Use torch.use_deterministic_algorithms(True, warn_only=True) "
               "to run it anyway.")
        if not torch.is_deterministic_algorithms_warn_only_enabled():
            raise RuntimeError(msg)
        warnings.warn(msg, stacklevel=3)
        on = False
    if get_mode("deterministic") != int(on):
        set_mode("deterministic", int(on))
    return on


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib.fegnn_last_error().decode("utf-8", "replace")
        raise FegnnError(f"{what or 'fegnn'} failed with code {rc}: {msg}")


DEFAULT_MODES = {ph: get_mode(ph) for ph in PHASES}      # the library's built-in defaults
if os.environ.get("FEGNN_PRECISION"):
    set_precision(os.environ["FEGNN_PRECISION"])
for _phase in PHASES:
    _env = os.environ.get("FEGNN_MODE_" + _phase.upper())
    if _env is not None:
        set_mode(_phase, int(_env))


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
