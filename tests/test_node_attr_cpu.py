"""Node attributes (node_attr_nf > 0) without a GPU: the specification (tests/node_attr_spec.py), its staged pipeline
against the oracle's autograd, the module API's bounds and argument checks, and the C ABI's refusal of inconsistent dims."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F
from torch import nn

from oracle import fastegnn_oracle as orc
from oracle import staged
from tests import node_attr_spec as spec
from tests.helpers import oracle_run


def _case(Fa, seed=3, sizes=(7, 5, 9), C_=3, gravity=None):
    g = torch.Generator().manual_seed(seed)
    N, B = sum(sizes), len(sizes)
    batch = torch.cat([torch.full((n,), b, dtype=torch.long) for b, n in enumerate(sizes)])
    rows, cols, off = [], [], 0
    for n in sizes:
        rows.append(torch.randint(0, n, (3 * n,), generator=g) + off)
        cols.append(torch.randint(0, n, (3 * n,), generator=g) + off)
        off += n
    ei = torch.stack([torch.cat(rows), torch.cat(cols)])
    x = torch.randn(N, 3, generator=g)
    cfg = orc.OracleConfig(node_feat_nf=2, node_attr_nf=Fa, edge_attr_nf=2, virtual_channels=C_, n_layers=3,
                           gravity=gravity)
    params = {k: v.double() for k, v in orc.make_params(cfg, seed + 100).items()}
    orc.rescale_coord_heads(params, 1000.0)
    inp = dict(node_feat=torch.rand(N, 2, generator=g).double(), node_loc=x.double(),
               node_vel=(0.5 * torch.randn(N, 3, generator=g)).double(),
               loc_mean=torch.randn(B, 3, C_, generator=g).double(),
               edge_attr=torch.rand(ei.size(1), 2, generator=g).double(), edge_index=ei, data_batch=batch,
               wx=torch.randn(N, 3, generator=g).double(), wz=torch.randn(B, 3, C_, generator=g).double(),
               node_attr=torch.randn(N, Fa, generator=g).double())
    return cfg, params, inp


def _oracle_with_attr(cfg, params, inp):
    p = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    leaf = {k: inp[k].clone().requires_grad_(True) for k in ("node_loc", "loc_mean", "node_feat")}
    x, Z = spec.oracle_forward(p, cfg, leaf["node_feat"], leaf["node_loc"], inp["node_vel"], inp["edge_index"],
                               inp["data_batch"], leaf["loc_mean"], inp["edge_attr"], inp["node_attr"])
    ((x * inp["wx"]).sum() + (Z * inp["wz"]).sum()).backward()
    return x.detach(), Z.detach(), {k: t.grad for k, t in leaf.items()}, {k: t.grad for k, t in p.items()}


@pytest.mark.parametrize("Fa", [1, 3])
@pytest.mark.parametrize("gravity", [None, (0.0, 0.0, -1.0)])
def test_staged_attr_term_equals_oracle_autograd_fp64(Fa, gravity):
    cfg, params, inp = _case(Fa, gravity=gravity)
    x_r, Z_r, gin_r, gp_r = _oracle_with_attr(cfg, params, inp)
    fl = staged.Flags(cfg.attention, cfg.normalize, cfg.tanh, cfg.gravity, cfg.eps)
    sm = spec.StagedModel(params, inp["node_attr"], 64, cfg.virtual_channels, cfg.edge_attr_nf, cfg.n_layers, fl)
    x, Z = sm.forward(inp["node_feat"], inp["node_loc"], inp["node_vel"], inp["edge_index"], inp["data_batch"],
                      inp["loc_mean"], inp["edge_attr"])
    assert torch.allclose(x, x_r, rtol=1e-10, atol=1e-11)
    assert torch.allclose(Z, Z_r, rtol=1e-10, atol=1e-11)
    grads, gin = sm.backward(inp["wx"], inp["wz"])
    for k in ("node_loc", "loc_mean", "node_feat"):
        assert torch.allclose(gin[k], gin_r[k], rtol=1e-8, atol=1e-10 * float(gin_r[k].abs().max())), k
    last = f"gcl_{cfg.n_layers - 1}.node_mlp"
    for k, g in gp_r.items():
        if g is None or k.startswith(last):
            assert g is None or float(g.abs().max()) == 0.0 or k not in grads, k
            continue
        s = float(g.abs().max()) + 1e-30
        assert torch.allclose(grads[k], g, rtol=1e-7, atol=1e-9 * s), (k, float((grads[k] - g).abs().max()), s)
    # the attribute columns of node_mlp.0.weight get a gradient in every layer but the last
    W = grads["gcl_0.node_mlp.0.weight"]
    assert W.shape == (64, (2 + cfg.virtual_channels) * 64 + Fa) and float(W[:, -Fa:].abs().max()) > 0


def test_spec_is_the_linear_on_attributes_last():
    """fold() restates node_mlp.0 on [x ; a], attribute columns last, as the attribute-free Linear plus a per-node bias."""
    g = torch.Generator().manual_seed(0)
    x, a = torch.randn(9, 5 * 64, generator=g).double(), torch.randn(9, 3, generator=g).double()
    W, b = torch.randn(64, 5 * 64 + 3, generator=g).double(), torch.randn(64, generator=g).double()
    f = spec.fold({"node_mlp.0.weight": W, "node_mlp.0.bias": b, "node_mlp_virtual.0.weight": W}, a)
    assert f["node_mlp_virtual.0.weight"] is W
    assert torch.allclose(F.linear(x, f["node_mlp.0.weight"], f["node_mlp.0.bias"]), F.linear(torch.cat([x, a], 1), W, b),
                          rtol=1e-13, atol=1e-12)


def test_zero_attributes_give_the_attribute_free_oracle():
    """Zero attributes: the model with attributes is the attribute-free oracle (whose Fa = 0 function the golden cases
    pin) on the leading columns of node_mlp.0.weight."""
    cfg, params, inp = _case(1)
    cfg0 = orc.OracleConfig(**{**cfg.__dict__, "node_attr_nf": 0})
    p0 = {k: (v[:, :-1].contiguous() if k.endswith("node_mlp.0.weight") else v) for k, v in params.items()}
    zero = dict(inp, node_attr=torch.zeros_like(inp["node_attr"]))
    x_a, Z_a, _, _ = _oracle_with_attr(cfg, params, zero)
    r0 = oracle_run(cfg0, p0, inp)
    assert torch.allclose(x_a, r0["x"], rtol=0, atol=1e-12) and torch.allclose(Z_a, r0["Z"], rtol=0, atol=1e-12)


def test_constructor_bounds_and_weight_shape():
    from fastegnn_b200 import FastEGNN, E_GCL_vel
    for Fa in (1, 5, 16):
        m = FastEGNN(node_feat_nf=2, node_attr_nf=Fa, edge_attr_nf=2, hidden_nf=64, virtual_channels=3, n_layers=2)
        assert m.gcl_0.node_mlp[0].weight.shape == (64, 5 * 64 + Fa)
        assert m.gcl_1.node_attr_nf == Fa
    for bad in (17, -1):
        with pytest.raises(NotImplementedError, match="node_attr_nf"):
            FastEGNN(node_feat_nf=2, node_attr_nf=bad, edge_attr_nf=2, hidden_nf=64, virtual_channels=3)
        with pytest.raises(NotImplementedError, match="node_attr_nf"):
            E_GCL_vel(64, 64, bad, 0, 64, 3)
    layer = E_GCL_vel(64, 64, 4, 0, 64, 8)
    assert layer.node_mlp[0].weight.shape == (64, 10 * 64 + 4)


def test_argument_checks_raise_before_device_work():
    """A CPU-resident model and CPU inputs: every node_attr check fires before anything needs a device."""
    from fastegnn_b200 import FastEGNN, E_GCL_vel
    N = 6
    args = dict(node_feat=torch.rand(N, 2), node_loc=torch.randn(N, 3), node_vel=torch.randn(N, 3),
                edge_index=torch.zeros(2, 4, dtype=torch.long), data_batch=torch.zeros(N, dtype=torch.long),
                loc_mean=torch.zeros(1, 3, 3), edge_attr=torch.zeros(4, 2))
    m2 = FastEGNN(node_feat_nf=2, node_attr_nf=2, edge_attr_nf=2, hidden_nf=64, virtual_channels=3, n_layers=1)
    with pytest.raises(TypeError, match="node_attr is required"):
        m2(**args)
    with pytest.raises(RuntimeError, match="node_attr_nf=2"):
        m2(**args, node_attr=torch.zeros(N, 3))
    with pytest.raises(RuntimeError, match="rows"):
        m2(**args, node_attr=torch.zeros(N + 1, 2))
    with pytest.raises(RuntimeError, match="CUDA"):
        m2(**args, node_attr=torch.zeros(N, 2))
    m0 = FastEGNN(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, hidden_nf=64, virtual_channels=3, n_layers=1)
    with pytest.raises(RuntimeError, match="node_attr_nf=0"):
        m0(**args, node_attr=torch.zeros(N, 1))
    layer = E_GCL_vel(64, 64, 2, 2, 64, 3)
    largs = (torch.randn(N, 64), args["edge_index"], args["node_loc"], args["node_vel"], torch.zeros(1, 3, 3),
             torch.zeros(1, 64, 3), args["data_batch"], args["edge_attr"])
    with pytest.raises(TypeError, match="node_attr is required"):
        layer(*largs)
    with pytest.raises(RuntimeError, match="rows"):
        layer(*largs, node_attr=torch.zeros(N - 1, 2))


def test_make_dims_positional_form_and_defaults():
    from fastegnn_b200 import _lib as L
    from fastegnn_b200.ops import make_dims
    d = make_dims(8, 8, 16, 1, 3, 2, 0, None)
    assert (d.N, d.Nl, d.E, d.B, d.C, d.Fe, d.Fa) == (8, 8, 16, 1, 3, 2, 0) and not d.node_attr
    a = torch.zeros(8, 3)
    d = make_dims(8, 8, 16, 1, 3, 2, 0, None, 1e-8, Fa=3, node_attr=a)
    assert d.Fa == 3 and d.node_attr == a.data_ptr()
    assert L.MAX_FA == 16 and L.lib.fegnn_version() == 103
    # the appended members sit where fegnn.h puts them (after eps, pointer-aligned)
    assert L.Dims.Fa.offset == 44 and L.Dims.node_attr.offset == 48 and C.sizeof(L.Dims) == 56


@pytest.mark.parametrize("Fa,with_ptr,flags,msg", [(17, True, 0, b"Fa=17 outside"), (-1, False, 0, b"Fa=-1 outside"),
                                                   (2, False, 0, b"must be non-NULL"), (0, True, 0, b"must be NULL"),
                                                   (1, True, 32, b"FEGNN_F_RF")])
def test_check_dims_rejects_bad_node_attr_through_the_abi(Fa, with_ptr, flags, msg):
    """Refused in check_dims, before any launch: no device is touched (the pointer is never dereferenced)."""
    from fastegnn_b200 import _lib as L
    from fastegnn_b200.ops import make_dims
    d = make_dims(8, 8, 16, 1, 3, 0, flags, None)
    d.Fa, d.node_attr = Fa, (256 if with_ptr else None)
    rc = L.lib.fegnn_node_pre_forward(C.byref(d), None, None, None, None)
    assert rc == -1 and msg in L.lib.fegnn_last_error()
    rc = L.lib.fegnn_model_forward(C.byref(d), 1, 1, None, None, *([None] * 9), None, 0, None)
    assert rc == -1 and msg in L.lib.fegnn_last_error()


def test_siblings_and_partitioned_wrapper_still_refuse():
    from fastegnn_b200 import FastEGNN
    from fastegnn_b200.FastRF import FastRF
    from fastegnn_b200.VNEGNN import VNEGNN
    from fastegnn_b200.partitioned import PartitionedFastEGNN
    with pytest.raises(NotImplementedError, match="node_attr_nf"):
        FastRF(node_feat_nf=2, node_attr_nf=1, edge_attr_nf=2, hidden_nf=64, virtual_channels=3)
    with pytest.raises(NotImplementedError, match="node_attr_nf"):
        VNEGNN(node_feat_nf=2, node_attr_nf=1, edge_attr_nf=2, hidden_nf=64, virtual_channels=3)
    m = FastEGNN(node_feat_nf=2, node_attr_nf=1, edge_attr_nf=2, hidden_nf=64, virtual_channels=3, n_layers=1)
    with pytest.raises(NotImplementedError, match="node attributes"):
        PartitionedFastEGNN(m, plan=None, rank=0, device="cpu")
