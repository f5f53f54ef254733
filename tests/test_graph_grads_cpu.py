"""Differentiable prebuilt graphs on the host: the fp64 torch composition the GPU tests take as their specification
(tests/graph_grads_spec.py) under torch.autograd.gradcheck, and every refusal of fegnn_edge_length_backward and of the
Python API that happens before any device work (so these run without a GPU)."""
import ctypes as C
import os
import re

import pytest
import torch

from fastegnn_b200 import CsrGraph, _lib
from fastegnn_b200.ops import make_dims
from oracle import fastegnn_oracle as orc
from oracle import fastrf_oracle as rfo
from tests import graph_grads_spec as spec

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 0x1000          # a non-NULL device address that nothing on the host dereferences


# ----------------------------------------------------------------------------- the specification
def _case(seed, rf):
    cfg = orc.OracleConfig(node_feat_nf=2, edge_attr_nf=2, hidden_nf=16, virtual_channels=2, n_layers=1)
    params = {k: v.double() for k, v in (rfo if rf else orc).make_params(cfg, seed).items()}
    orc.rescale_coord_heads(params, 100.0)
    g = torch.Generator().manual_seed(seed)
    sizes = [5, 4]
    batch = torch.cat([torch.full((n,), b, dtype=torch.long) for b, n in enumerate(sizes)])
    x = torch.rand(9, 3, generator=g, dtype=torch.float64)
    x[3] = x[2]                                            # a coincident pair: lengths 0, torch's norm subgradient
    # every ordered pair of each graph (the complete graph of from_radius(r = inf)); step 2 drops some edges
    eis = []
    for drop in (0, 3):
        rows, cols, off = [], [], 0
        for n in sizes:
            for i in range(n):
                for j in range(n):
                    if i != j and (drop == 0 or (i + j) % drop):
                        rows.append(off + i)
                        cols.append(off + j)
            off += n
        eis.append(torch.tensor([rows, cols]))
    lm = torch.stack([x[batch == b].mean(0) for b in range(2)]).unsqueeze(-1).repeat(1, 1, 2)
    return cfg, params, dict(x=x, batch=batch, eis=eis, lm=lm, feat=torch.rand(9, 2, generator=g, dtype=torch.float64),
                             v=0.1 * torch.randn(9, 3, generator=g, dtype=torch.float64))


@pytest.mark.parametrize("rf", [False, True], ids=["FastEGNN", "FastRF"])
def test_rollout_composition_passes_gradcheck(rf):
    """Two steps, each on its own edge list with edge_attr = lengths of that step's positions and v = (x' - x) / dt: the
    fp64 autograd gradient with respect to the initial positions and one weight matches finite differences."""
    cfg, params, t = _case(5, rf)
    fwd = rfo.fastrf_forward if rf else orc.fastegnn_forward
    w = params["gcl_0.edge_mlp.0.weight"]

    def loss(x0, w0):
        p = dict(params, **{"gcl_0.edge_mlp.0.weight": w0})
        f = lambda x, v, ei, ea, lm: fwd(p, cfg, t["feat"], x, v, ei, t["batch"], lm, ea)
        xo, Zo = spec.rollout(f, x0, t["v"], t["lm"], t["eis"], cfg.edge_attr_nf, 0.5)
        return (xo * torch.linspace(-1, 1, xo.numel(), dtype=xo.dtype).view_as(xo)).sum() + Zo.sum()

    x0 = t["x"].clone().requires_grad_(True)
    w0 = w.clone().requires_grad_(True)
    assert torch.autograd.gradcheck(loss, (x0, w0), eps=1e-6, atol=1e-5, rtol=1e-4)


def test_zero_length_subgradient_is_zero():
    x = torch.tensor([[0.0, 0.0, 0.0], [0.0, 0.0, 0.0], [1.0, 0.0, 0.0]], dtype=torch.float64, requires_grad=True)
    ei = torch.tensor([[0, 1, 0], [1, 0, 2]])
    spec.lengths(x, ei, 2).sum().backward()
    assert torch.equal(x.grad, torch.tensor([[-2.0, 0, 0], [0, 0, 0], [2.0, 0, 0]], dtype=torch.float64))


# ----------------------------------------------------------------------------- the C entry's refusals
def _graph(n_edges=None):
    return _lib.Graph(FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, None, n_edges)


def _call(dims, graph, rowptr=FAKE, x=FAKE, g_ea=FAKE, g_x=FAKE):
    return _lib.lib.fegnn_edge_length_backward(C.byref(dims), C.byref(graph), rowptr, x, g_ea, g_x, None)


def _expect_einval(rc, pattern):
    assert rc == -1, rc
    assert re.search(pattern, _lib.lib.fegnn_last_error().decode()), _lib.lib.fegnn_last_error().decode()


def test_symbol_in_header_and_binding():
    header = open(os.path.join(ROOT, "include", "fegnn.h")).read()
    assert re.search(r"\bfegnn_edge_length_backward\s*\(", header)
    assert "fegnn_edge_length_backward" in _lib.SIGNATURES


def test_entry_refuses_before_any_launch():
    _expect_einval(_call(make_dims(100, 100, 1000, 2, 1, 0, 0), _graph()), r"Fe = 0")
    _expect_einval(_call(make_dims(100, 100, 1000, 2, 1, 2, _lib.F_LIVE_EDGES), _graph()), r"n_edges is NULL")
    _expect_einval(_call(make_dims(100, 100, 1000, 2, 1, 2, 0), _graph(), x=None), r"requirement failed")
    _expect_einval(_call(make_dims(100, 100, 1000, 2, 1, 2, 0), _graph(), rowptr=None), r"requirement failed")
    _expect_einval(_call(make_dims(100, 100, 1000, 2, 1, 9, 0), _graph()), r"Fe=9")


def test_entry_refuses_the_deterministic_mode():
    _lib.set_mode("deterministic", 1)
    try:
        _expect_einval(_call(make_dims(100, 100, 1000, 2, 1, 2, 0), _graph()), r"no deterministic form")
    finally:
        _lib.set_mode("deterministic", 0)


# ----------------------------------------------------------------------------- the Python API
def test_differentiable_graph_needs_an_edge_attr():
    x = torch.zeros(4, 3)
    batch = torch.zeros(4, dtype=torch.long)
    with pytest.raises(_lib.FegnnError, match="edge_attr_nf > 0"):
        CsrGraph.from_radius(x, batch, 1, 1.0, edge_attr_nf=0, differentiable=True)
    with pytest.raises(_lib.FegnnError, match="needs an edge_attr"):
        CsrGraph(torch.zeros(2, 3, dtype=torch.long), batch, None, 1, differentiable=True)


def test_defaults_are_not_differentiable():
    assert CsrGraph.differentiable is False and CsrGraph.builds == 0


def test_check_build_names_both_builds():
    g = CsrGraph.__new__(CsrGraph)
    g.builds = 3
    g.check_build(3)
    with pytest.raises(_lib.FegnnError, match=r"rebuilt .*build 2, now 3"):
        g.check_build(2)
