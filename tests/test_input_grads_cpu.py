"""Gradients to node_vel, edge_attr and node_attr without a GPU: the hand-written backward (oracle/staged.py plus the terms
below, which is what the kernels compute) against the oracle's fp64 autograd, and the C ABI's entries and refusals."""
import ctypes as C
import dataclasses
import os

import pytest
import torch

from oracle import fastegnn_oracle as orc
from oracle import staged
from tests import node_attr_spec as spec
from tests.gpu_util import make_graph_case
from tests.helpers import MODEL_CASES, case_inputs, case_params, load_case


def edge_gz1(w, g, fl, P, Q, x, ea, gm, gt):
    """dL/dz1 of every (CSR-ordered) edge: staged.edge_bwd up to its gz1."""
    r = staged._edge_recompute(w, g, fl, P, Q, x, ea)
    gte = gt[g.row]
    gs = (r["dn"] * gte).sum(1)
    if fl.tanh:
        gs = gs * (1 - r["s"] ** 2)
    gz3 = gs[:, None] * w.w4 * staged.dsilu(r["z3"])
    gmm = gm[g.row] + gz3 @ w.W3
    if fl.attention:
        gpre = (gmm * r["m0"]).sum(1) * r["gate"] * (1 - r["gate"])
        gmm = gmm * r["gate"][:, None] + gpre[:, None] * w.wa
    return ((gmm * staged.dsilu(r["z2"])) @ w.W2) * staged.dsilu(r["z1"])


class InputGradStaged(staged.StagedModel):
    """The staged backward plus the three input gradients, per layer l (summed):
         node_vel  += sv_l * gxn_l                 (x' = ... + phi_v(h) v; gxn = dL/dx' including the next xbar)
         edge_attr += gz1_l Wa_l, back in caller order through the sort permutation
         node_attr += gUh_l U1att_l                (layers with a Uh block: all but the last)
    With node attributes the forward runs through the folded weights of tests/node_attr_spec.py."""

    def __init__(self, sd, node_attr, H, C_, Fe, L, fl):
        super().__init__(sd if node_attr is None else spec.fold(sd, node_attr), H, C_, Fe, L, fl)
        self.raw, self.node_attr_in = sd, node_attr

    def forward(self, node_feat, x0, v, edge_index, batch, loc_mean, edge_attr):
        self.perm = torch.sort(edge_index[0], stable=True).indices          # the order staged.StagedModel sorts into
        return super().forward(node_feat, x0, v, edge_index, batch, loc_mean, edge_attr)

    def backward(self, gx_out, gZ_out):
        grads, gin = super().backward(gx_out, gZ_out)
        g, fl, N = self.g, self.fl, self.g.N
        gv = gx_out.new_zeros(N, 3)
        gea = self.ea.new_zeros(self.ea.shape)
        ga = None if self.node_attr_in is None else gx_out.new_zeros(self.node_attr_in.shape)
        for l in range(self.L):
            w, sv, b = self.w[l], self.saved[l], self.bsaved[l]
            gv += sv["npre"]["sv"][:, None] * b["gxn"]
            gz1 = edge_gz1(w, g, fl, sv["npre"]["P"], sv["npre"]["Q"], sv["x"], self.ea, b["b"]["gm"], b["c"]["gt"])
            gea += gz1 @ w.Wa                                            # Wa = W1[:, 2H+1:], [H, Fe]
            if ga is not None and l < self.L - 1:
                W0 = self.raw[f"gcl_{l}.node_mlp.0.weight"]
                ga += b["b"]["gzh1"] @ W0[:, W0.size(1) - ga.size(1):]
        out = torch.zeros_like(gea)
        out[self.perm] = gea
        gin = dict(gin, node_vel=gv, edge_attr=out)
        if ga is not None:
            gin["node_attr"] = ga
        return grads, gin


def staged_vs_autograd(cfg, params, inp, node_attr=None):
    p64 = {k: v.double() for k, v in params.items()}
    d = {k: (v.double() if v.is_floating_point() else v) for k, v in inp.items()}
    fl = staged.Flags(cfg.attention, cfg.normalize, cfg.tanh, cfg.gravity)
    na = None if node_attr is None else node_attr.double()
    m = InputGradStaged(p64, na, cfg.hidden_nf, cfg.virtual_channels, cfg.edge_attr_nf, cfg.n_layers, fl)
    m.forward(d["node_feat"], d["node_loc"], d["node_vel"], d["edge_index"], d["data_batch"], d["loc_mean"], d["edge_attr"])
    _, gin = m.backward(d["wx"], d["wz"])
    leaf = {k: d[k].clone().requires_grad_(True) for k in ("node_vel", "edge_attr")}
    if na is not None:
        leaf["node_attr"] = na.clone().requires_grad_(True)
    args = (d["node_feat"], d["node_loc"], leaf["node_vel"], d["edge_index"], d["data_batch"], d["loc_mean"], leaf["edge_attr"])
    x, Z = (spec.oracle_forward(p64, cfg, *args, leaf["node_attr"]) if na is not None else orc.fastegnn_forward(p64, cfg, *args))
    ((x * d["wx"]).sum() + (Z * d["wz"]).sum()).backward()
    for k, t in leaf.items():
        assert torch.allclose(gin[k], t.grad, rtol=1e-9, atol=1e-9 * float(t.grad.abs().max())), k
    return gin


@pytest.mark.parametrize("case", MODEL_CASES)
def test_staged_node_vel_and_edge_attr_gradients_equal_autograd(case):
    meta, arr = load_case(case)
    cfg, params = case_params(meta["case"])
    inp = case_inputs(arr)
    staged_vs_autograd(cfg, params, inp)


@pytest.mark.parametrize("attention,normalize", [(False, False), (True, True)])
def test_staged_gradients_unsorted_edges_with_duplicates_and_self_loops(attention, normalize):
    cfg, params, inp = make_graph_case(7, [30, 22, 41], 6, 3, Fe=3, L=3, attention=attention, normalize=normalize)
    ei = inp["edge_index"]
    loops = torch.arange(0, 90, 9)
    dup = ei[:, :15]
    inp["edge_index"] = torch.cat([ei, torch.stack([loops, loops]), dup], dim=1)
    g = torch.Generator().manual_seed(1)
    inp["edge_attr"] = torch.rand(inp["edge_index"].size(1), 3, generator=g)
    staged_vs_autograd(cfg, params, inp)


@pytest.mark.parametrize("Fa", [1, 5, 16])
def test_staged_node_attr_gradient_equals_spec_autograd(Fa):
    cfg0, params0, inp = make_graph_case(9, [30, 40], 5, 2, Fe=2, L=3)
    cfg = dataclasses.replace(cfg0, node_attr_nf=Fa)
    params = orc.make_params(cfg, 1009)
    na = torch.randn(inp["node_loc"].size(0), Fa, generator=torch.Generator().manual_seed(2))
    staged_vs_autograd(cfg, params, inp, node_attr=na)


# ----------------------------------------------------------------------------- C ABI
NEW_SYMBOLS = ["fegnn_model_backward_inputs", "fegnn_virtual_backward_inputs", "fegnn_edge_backward_inputs",
               "fegnn_node_pre_backward_inputs"]


def test_new_symbols_are_declared_and_exported():
    from fastegnn_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "fegnn.h")).read()
    assert "typedef struct fegnn_input_grads" in header
    for s in NEW_SYMBOLS:
        assert f"int {s}(" in header and s in _lib.SIGNATURES and hasattr(_lib.lib, s), s
    assert C.sizeof(_lib.InputGrads) == 32


ENTRIES = ("model", "virtual", "edge", "node_pre")


def _refusal(entry, dims_kw, ig_kw, edge_mode=None):
    """One of the four _inputs entries with a request it must refuse.  Nothing could touch memory even if the refusal came
    late: every size is 0 (N = E = B = 0: zero-length fills, empty grids), every other pointer is NULL, and the requested
    output is a real one-float device buffer where a device exists (elsewhere no launch can run at all).  The library's
    launch counter must not move."""
    import torch
    from fastegnn_b200 import _lib as L
    from fastegnn_b200.ops import make_dims
    d = make_dims(0, 0, 0, 0, 3, dims_kw.get("Fe", 2), dims_kw.get("flags", 0))
    buf = torch.zeros(1, device="cuda") if torch.cuda.is_available() else None
    out = buf.data_ptr() if buf is not None else 0x100
    ig = L.InputGrads(**{k: out for k in ig_kw})
    pd, pg, pi = C.byref(d), C.byref(L.Graph()), C.byref(ig)
    pp, pgr, ps = C.byref(L.LayerPtrs()), C.byref(L.LayerPtrs()), C.byref(L.Saved())
    old = L.get_mode("edge_backward")
    if edge_mode is not None:
        L.set_mode("edge_backward", edge_mode)
    launches = L.lib.fegnn_launch_count()
    try:
        if entry == "model":
            lp = (L.LayerPtrs * 2)()
            rc = L.lib.fegnn_model_backward_inputs(pd, 2, 2, pg, lp, lp, *[None] * 11, None, None, 0, pi, None)
        elif entry == "virtual":
            rc = L.lib.fegnn_virtual_backward_inputs(pd, pg, pp, pgr, None, None, None, ps, *[None] * 12, pi, None)
        elif entry == "edge":
            rc = L.lib.fegnn_edge_backward_inputs(pd, pg, pp, pgr, None, ps, *[None] * 5, pi, None)
        else:
            rc = L.lib.fegnn_node_pre_backward_inputs(pd, pp, pgr, *[None] * 8, pi, None)
    finally:
        L.set_mode("edge_backward", old)
    assert L.lib.fegnn_launch_count() == launches
    return rc, L.lib.fegnn_last_error().decode()


# (entry, dims, request, edge_backward mode, message); each per-phase entry with the request it consumes
REFUSALS = [
    ("model", dict(Fe=2), ["node_attr"], None, "Fa = 0"),
    ("model", dict(Fe=0), ["edge_attr"], None, "Fe = 0"),
    ("model", dict(Fe=2, flags=32), ["node_vel"], None, "FEGNN_F_RF"),
    ("model", dict(Fe=2), ["edge_attr"], 4, "edge_backward mode 4"),
    ("model", dict(Fe=2), ["edge_attr"], 8, "edge_backward mode 8"),
    ("virtual", dict(Fe=2, flags=32), ["node_vel"], None, "FEGNN_F_RF"),
    ("edge", dict(Fe=0), ["edge_attr"], None, "Fe = 0"),
    ("edge", dict(Fe=2), ["edge_attr"], 1, "edge_backward mode 1"),
    ("edge", dict(Fe=4), ["edge_attr"], 5, "edge_backward mode 5"),
    ("node_pre", dict(Fe=2), ["node_attr"], None, "Fa = 0"),
]


@pytest.mark.parametrize("entry,dims_kw,ig_kw,edge_mode,needle", REFUSALS)
def test_requests_are_refused_before_any_launch(entry, dims_kw, ig_kw, edge_mode, needle):
    rc, msg = _refusal(entry, dims_kw, ig_kw, edge_mode)
    assert rc == -1 and needle in msg, msg
