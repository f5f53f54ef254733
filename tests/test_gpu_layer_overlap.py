"""fegnn_set_mode("layer_overlap", 2) (the overlapped arrangement at every size; the default, auto, takes it at Water-3D
size only): the backward with each layer's virtual backward on a second stream next to its edge
backward (edge tiles claimed dynamically) against the same backward with the two one after the other (static tile split).
Both arrangements run the same kernels on the same inputs; only the order of float atomics differs, so they agree to the
run-to-run level of the default arithmetic mode (DESIGN.md 3.7)."""
import contextlib

import pytest
import torch

from tests.gpu_util import make_graph_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@contextlib.contextmanager
def overlap(mode):
    from fastegnn_b200 import _lib
    old = _lib.get_mode("layer_overlap")
    _lib.set_mode("layer_overlap", mode)
    try:
        yield
    finally:
        _lib.set_mode("layer_overlap", old)


def model(cfg, params, rf=False, Fa=0):
    from fastegnn_b200 import FastEGNN, FastRF
    torch.manual_seed(7)
    m = (FastRF if rf else FastEGNN)(node_feat_nf=cfg.node_feat_nf, node_attr_nf=Fa, edge_attr_nf=cfg.edge_attr_nf,
                                     hidden_nf=64, virtual_channels=cfg.virtual_channels, device=DEV,
                                     n_layers=cfg.n_layers, attention=cfg.attention, normalize=cfg.normalize,
                                     tanh=cfg.tanh, gravity=cfg.gravity)
    if Fa == 0 and not rf:             # FastRF and node attributes: the seeded default initialisation
        m.load_state_dict({k: v.to(DEV) for k, v in params.items()})
    return m


def step(m, inp, want, node_attr=None):
    """loss, parameter gradients and the requested input gradients of one forward + backward."""
    t = {k: (None if v is None else v.to(DEV)) for k, v in inp.items()}
    if node_attr is not None:
        t["node_attr"] = node_attr.to(DEV)
    leaf = {k: t[k].clone().requires_grad_(k in want)
            for k in ("node_feat", "node_loc", "node_vel", "loc_mean", "edge_attr", "node_attr") if t.get(k) is not None}
    m.zero_grad(set_to_none=True)
    x, Z = m(node_feat=leaf["node_feat"], node_loc=leaf["node_loc"], node_vel=leaf["node_vel"],
             edge_index=t["edge_index"], data_batch=t["data_batch"], loc_mean=leaf["loc_mean"],
             edge_attr=leaf.get("edge_attr"), **({"node_attr": leaf["node_attr"]} if "node_attr" in leaf else {}))
    loss = (x * t["wx"]).sum() + (Z * t["wz"]).sum()
    loss.backward()
    torch.cuda.synchronize()
    out = {"loss": loss.detach().reshape(1)}
    out.update({"grad." + k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None})
    out.update({"input." + k: leaf[k].grad.detach().clone() for k in want})
    return out


def compare(m, inp, want, tol, node_attr=None):
    with overlap(0):
        ref = step(m, inp, want, node_attr)
    with overlap(2):
        got = step(m, inp, want, node_attr)
    assert ref.keys() == got.keys()
    for k in ref:
        scale = ref[k].abs().max().item()
        err = (got[k] - ref[k]).abs().max().item() / max(scale, 1e-30)
        print(f"LAYER_OVERLAP {k} {err:.3e}")
        assert err <= tol, (k, err)


# a second run of the same step in the default mode (the layer kernels add floats across CTAs in arrival order); the
# same bound as tests/test_gpu_input_grads.py RUN_TO_RUN["tf32"]
TOL = 1e-3

CASES = {
    # Water-3D size: 8 000 nodes, ~180 k edges (1 400 edge tiles, 188 virtual tiles), C = 3, gravity, 4 layers
    "water3d": dict(seed=3, sizes=[8000], deg=22, C=3, L=4, gravity=[0, -1, 0]),
    # fewer tiles than SMs: one edge tile (120 edges), one virtual tile (40 nodes x 3 channels)
    "one_tile": dict(seed=4, sizes=[40], deg=3, C=3, L=3),
    "one_layer": dict(seed=5, sizes=[300, 200, 250], deg=9, C=3, L=1),
}


@pytest.mark.parametrize("name", list(CASES))
def test_overlap_matches_sequential(name):
    kw = dict(CASES[name])
    cfg, params, inp = make_graph_case(kw.pop("seed"), kw.pop("sizes"), kw.pop("deg"), kw.pop("C"), L=kw.pop("L"), **kw)
    compare(model(cfg, params), inp, ("node_loc", "loc_mean", "node_feat"), TOL)


def test_overlap_matches_sequential_fastrf():
    cfg, params, inp = make_graph_case(6, [400, 350], 10, 3, L=3)
    compare(model(cfg, params, rf=True), inp, ("node_loc", "loc_mean", "node_feat"), TOL)


def test_overlap_matches_sequential_all_input_gradients():
    cfg, params, inp = make_graph_case(8, [900, 700], 12, 3, L=3, gravity=[0, -1, 0])
    g = torch.Generator().manual_seed(9)
    node_attr = torch.randn(inp["node_loc"].size(0), 2, generator=g)
    compare(model(cfg, params, Fa=2), inp, ("node_loc", "loc_mean", "node_feat", "node_vel", "edge_attr", "node_attr"),
            TOL, node_attr)


def test_dynamic_claims_cover_every_edge_tile_once():
    """Water-3D size, layer_overlap 2, repeated: a tile skipped or taken twice changes the edge weights' gradients by
    about 1/1400 of their size; they must match the static split well below that."""
    from fastegnn_b200 import _lib
    cfg, params, inp = make_graph_case(10, [8000], 22, 3, L=2)
    m = model(cfg, params)
    old = _lib.get_mode("edge_backward")
    try:
        _lib.set_mode("edge_backward", 7)
        with overlap(0):
            ref = step(m, inp, ())
        with overlap(2):
            got = [step(m, inp, ()) for _ in range(3)]
    finally:
        _lib.set_mode("edge_backward", old)
    for k in ref:
        if ".edge_mlp." not in k and ".coord_mlp_r." not in k:
            continue
        scale = ref[k].abs().max().item()
        for g in got:
            err = (g[k] - ref[k]).abs().max().item() / max(scale, 1e-30)
            print(f"LAYER_OVERLAP_CLAIMS {k} {err:.3e}")
            assert err <= 1e-4, (k, err)
