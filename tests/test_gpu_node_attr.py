"""Node attributes (node_attr_nf > 0) on the GPU: the model, its phases and the layer-level API against the oracle with
the attribute term (tests/node_attr_spec.py on top of oracle/), in every arithmetic mode."""
import ctypes as C
import dataclasses
import os
import subprocess
import sys

import pytest
import torch

from oracle import fastegnn_oracle as orc
from oracle import staged
from tests import node_attr_spec as spec
from tests.gpu_util import EPS32, TOLERANCES, make_graph_case, precision, rel_err, update_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def attr_case(Fa, C_=3, seed=11, sizes=(50, 37, 61), deg=6, gravity=None, attention=False, L=3):
    """make_graph_case's batch plus node attributes [N, Fa] and parameters drawn with node_attr_nf = Fa."""
    cfg0, _, inp = make_graph_case(seed, list(sizes), deg, C_, L=L, gravity=gravity, attention=attention)
    cfg = dataclasses.replace(cfg0, node_attr_nf=Fa)
    params = orc.make_params(cfg, seed + 1000)
    orc.rescale_coord_heads(params, 1000.0)
    g = torch.Generator().manual_seed(seed + 7)
    inp = dict(inp, node_attr=torch.randn(inp["node_loc"].size(0), Fa, generator=g))
    return cfg, params, inp


def build(cfg, params):
    from fastegnn_b200 import FastEGNN
    m = FastEGNN(node_feat_nf=cfg.node_feat_nf, node_attr_nf=cfg.node_attr_nf, edge_attr_nf=cfg.edge_attr_nf,
                 hidden_nf=64, virtual_channels=cfg.virtual_channels, device=DEV, n_layers=cfg.n_layers,
                 attention=cfg.attention, normalize=cfg.normalize, tanh=cfg.tanh, gravity=cfg.gravity)
    m.load_state_dict({k: v.to(DEV) for k, v in params.items()})
    return m


def oracle(cfg, params, inp, dtype=torch.float64):
    p = {k: v.to(dtype).requires_grad_(True) for k, v in params.items()}
    f = lambda k: inp[k].to(dtype)
    leaf = {k: f(k).requires_grad_(True) for k in ("node_loc", "loc_mean", "node_feat")}
    x, Z = spec.oracle_forward(p, cfg, leaf["node_feat"], leaf["node_loc"], f("node_vel"), inp["edge_index"],
                               inp["data_batch"], leaf["loc_mean"], f("edge_attr"), f("node_attr"))
    ((x * f("wx")).sum() + (Z * f("wz")).sum()).backward()
    return dict(x=x.detach(), Z=Z.detach(), gin={k: t.grad for k, t in leaf.items()},
                gp={k: t.grad for k, t in p.items()})


def gpu(m, inp, want_grads=True, node_attr="given"):
    t = {k: v.to(DEV) for k, v in inp.items()}
    leaf = {k: t[k].clone().requires_grad_(want_grads) for k in ("node_loc", "loc_mean", "node_feat")}
    x, Z = m(node_feat=leaf["node_feat"], node_loc=leaf["node_loc"], node_vel=t["node_vel"], edge_index=t["edge_index"],
             data_batch=t["data_batch"], loc_mean=leaf["loc_mean"], edge_attr=t["edge_attr"],
             node_attr=t["node_attr"] if node_attr == "given" else None)
    res = dict(x=x.detach().cpu(), Z=Z.detach().cpu())
    if want_grads:
        ((x * t["wx"]).sum() + (Z * t["wz"]).sum()).backward()
        res["gin"] = {k: v.grad.cpu() for k, v in leaf.items()}
        res["gp"] = {k: (None if p.grad is None else p.grad.cpu()) for k, p in m.named_parameters()}
    torch.cuda.synchronize()
    return res


def check_against_oracle(res, ref, inp, tol):
    bad = []
    for k, base in (("x", inp["node_loc"]), ("Z", inp["loc_mean"])):
        e = update_err(res[k], ref[k], base)
        if e > tol.out:
            bad.append((k, e))
    for k, g in ref["gin"].items():
        e = rel_err(res["gin"][k], g)
        if e > tol.gin:
            bad.append((k, e))
    for k, g in ref["gp"].items():
        got = res["gp"][k]
        if g is None or float(g.abs().max()) == 0.0:
            if got is not None and float(got.abs().max()) != 0.0:
                bad.append((k, "should have no grad"))
            continue
        e = rel_err(got, g)
        # bias gradients are column sums of signed terms that cancel, like the two virtual-head biases tol.gb covers: on
        # these inputs (coordinate heads at gain 1000) the edge backward's TF32 / fp16 bias sums of coord_mlp_r.0 and
        # edge_mlp.2 reach 2.6e-2 / 2.8e-2 -- kernels node_attr does not touch
        t = tol.gb if k.endswith(".bias") else tol.for_param(k)
        if e > t:
            bad.append((k, e))
    return bad


MODEL_CASES = [dict(Fa=1, C_=3), dict(Fa=3, C_=8, gravity=[0.0, -1.0, 0.0]), dict(Fa=16, C_=3, attention=True),
               dict(Fa=3, C_=3), dict(Fa=16, C_=8)]


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "tf32"])
@pytest.mark.parametrize("case", range(len(MODEL_CASES)))
def test_model_forward_backward_against_oracle(case, prec):
    cfg, params, inp = attr_case(**MODEL_CASES[case])
    ref = oracle(cfg, params, inp)
    with precision(prec) as tol:
        res = gpu(build(cfg, params), inp)
    bad = check_against_oracle(res, ref, inp, tol)
    assert not bad, bad
    # the attribute columns of every layer but the last carry a gradient
    Fa = cfg.node_attr_nf
    assert float(res["gp"]["gcl_0.node_mlp.0.weight"][:, -Fa:].abs().max()) > 0


def _phase_setup(Fa, C_=3, gravity=None, last=False):
    from fastegnn_b200 import _lib as L
    from fastegnn_b200.ops import CsrGraph, SavedBlock, layer_ptrs, make_dims
    cfg, params, inp = attr_case(Fa, C_=C_, gravity=gravity, sizes=(300, 211))
    N = inp["node_loc"].size(0)
    g = torch.Generator().manual_seed(3)
    h = torch.randn(N, 64, generator=g) * 2
    a = inp["node_attr"]
    named = {k[len("gcl_0."):]: v.to(DEV).contiguous() for k, v in params.items() if k.startswith("gcl_0.")}
    graph = CsrGraph(inp["edge_index"].to(DEV), inp["data_batch"].to(DEV), inp["edge_attr"].to(DEV), 2)
    a_dev = a.to(DEV)
    flags = (L.F_GRAVITY if gravity else 0) | (L.F_LAST if last else 0)
    dims = make_dims(N, N, graph.E, 2, C_, graph.Fe, flags, gravity, Fa=Fa, node_attr=a_dev)
    w = spec.layer_weights({f"gcl_0.{k}": v.double().cpu() for k, v in named.items()}, a.double(), "gcl_0", 64, C_, 2,
                           False, gravity is not None)
    fl = staged.Flags(gravity=gravity)
    return L, dims, layer_ptrs(named, ""), SavedBlock(dims, DEV), h, a, a_dev, w, fl, named


@pytest.mark.parametrize("mode", [0, 1, 3])
@pytest.mark.parametrize("Fa", [1, 3, 16])
def test_node_pre_forward_modes_against_staged(Fa, mode):
    L, dims, ptrs, sv, h, a, a_dev, w, fl, _ = _phase_setup(Fa, gravity=[0.0, -1.0, 0.0])
    want = staged.node_pre(w, h.double(), fl)            # Uh carries U1att a through the per-node e1 of the spec
    old = L.get_mode("node_forward")
    try:
        L.set_mode("node_forward", mode)
        hd = h.to(DEV)
        L.check(L.lib.fegnn_node_pre_forward(C.byref(dims), C.byref(ptrs), L.ptr(hd), C.byref(sv.c), None))
        torch.cuda.synchronize()
    finally:
        L.set_mode("node_forward", old)
    tol = 2e-3 if mode == 1 else 2e-6                  # mode 1 rounds h to TF32; the attribute term is fp32 in every mode
    for k in ("P", "Q", "Av", "Uh"):
        e = rel_err(sv.view(k, (h.size(0), 64)).cpu(), want[k])
        assert e <= tol, (k, e)


def _node_pre_backward(Fa, mode):
    L, dims, ptrs, sv, h, a, a_dev, w, fl, named = _phase_setup(Fa, gravity=[0.0, -1.0, 0.0])
    N = h.size(0)
    g = torch.Generator().manual_seed(5)
    G = {k: torch.randn(N, 64, generator=g) for k in ("gP", "gQ", "gAv", "gUh")}
    G.update(gsv=torch.randn(N, generator=g), gsg=torch.randn(N, generator=g))
    want = staged.node_pre_bwd(w, None, fl, h.double(), *[G[k].double() for k in ("gP", "gQ", "gAv", "gUh", "gsv", "gsg")])
    dU1att = G["gUh"].double().T @ a.double()
    from fastegnn_b200.ops import layer_ptrs
    grads = {k: torch.zeros_like(v) for k, v in named.items()}
    gptrs = layer_ptrs(grads, "")
    Gd = {k: v.to(DEV).contiguous() for k, v in G.items()}
    gh = torch.zeros(N, 64, device=DEV)
    old = L.get_mode("node_backward")
    try:
        L.set_mode("node_backward", mode)
        L.check(L.lib.fegnn_node_pre_backward(C.byref(dims), C.byref(ptrs), C.byref(gptrs), L.ptr(h.to(DEV)),
                                              *[L.ptr(Gd[k]) for k in ("gP", "gQ", "gAv", "gUh", "gsv", "gsg")],
                                              L.ptr(gh), None))
        torch.cuda.synchronize()
    finally:
        L.set_mode("node_backward", old)
    tol = 2e-5 if mode == 0 else 4e-3
    assert rel_err(gh.cpu(), want["gh"]) <= tol
    C_ = 3
    W = grads["node_mlp.0.weight"].cpu()
    assert rel_err(W[:, 2 * 64 + 64 * C_:], dU1att) <= 2e-5       # fp32 column walk in every mode
    assert rel_err(W[:, :64], want["wg"]["U1h"]) <= tol
    assert rel_err(grads["node_mlp.0.bias"].cpu(), want["wg"]["e1"]) <= 2e-5


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("Fa", [1, 3, 16])
def test_node_pre_backward_modes_against_staged(Fa, mode):
    _node_pre_backward(Fa, mode)


def test_node_pre_backward_tile_block_kernel():
    """The (tile, block) tensor-core kernel, selectable by environment (read once per process): a fresh process."""
    if os.environ.get("FEGNN_DENSE_ROWS_MAX_TILES_PER_SM") == "0":
        for Fa in (1, 3, 16):
            _node_pre_backward(Fa, 1)
        return
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, FEGNN_DENSE_ROWS_MAX_TILES_PER_SM="0")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider",
                        "tests/test_gpu_node_attr.py::test_node_pre_backward_tile_block_kernel"],
                       cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
def test_zero_attributes_equal_the_attribute_free_model(prec):
    """Outputs and weight gradients to fp32 rounding on the fp32 kernels; on the TF32 tiles two runs differ by atomics
    order (which can move an operand across a 10-bit rounding boundary): outputs within test_gpu_model.py's eval-test bound
    2e-3, weight gradients within the mode's stated tolerance (2.6e-4 observed).  The attribute columns' gradient is 0."""
    cfg, params, inp = attr_case(3, C_=3)
    Fa = cfg.node_attr_nf
    inp = dict(inp, node_attr=torch.zeros_like(inp["node_attr"]))
    cfg0 = dataclasses.replace(cfg, node_attr_nf=0)
    p0 = {k: (v[:, :-Fa].contiguous() if k.endswith("node_mlp.0.weight") else v) for k, v in params.items()}
    with precision(prec) as tol:
        r = gpu(build(cfg, params), inp)
        r0 = gpu(build(cfg0, p0), inp, node_attr=None)
    for k in ("x", "Z"):
        if prec == "fp32":
            assert float((r[k] - r0[k]).abs().max()) <= 8 * EPS32 * float(r0[k].abs().max()), k
        else:
            assert rel_err(r[k], r0[k]) < 2e-3, k
    for k, g in r["gp"].items():
        if g is None:
            assert r0["gp"][k] is None
            continue
        if k.endswith("node_mlp.0.weight"):
            assert float(g[:, -Fa:].abs().max()) == 0.0, k          # exactly 0: sum of gUh * 0
            g = g[:, :-Fa]
        assert rel_err(g, r0["gp"][k]) <= (5e-5 if prec == "fp32" else tol.for_param(k)), k


@pytest.mark.parametrize("prec,bound", [("fp32", 1e-5), ("tf32", 2e-3)])
def test_forward_only_stack_equals_training_forward(prec, bound):
    """Bounds of test_gpu_model.py's eval test: atomics order differs between two launches (fp32 rounding on the fp32
    kernels; on the TF32 tiles that noise can move an operand across a 10-bit rounding boundary)."""
    cfg, params, inp = attr_case(3, C_=8, gravity=[0.0, -1.0, 0.0])
    m = build(cfg, params)
    with precision(prec):
        train = gpu(m, inp, want_grads=False)        # requires_grad=False leaves + grad mode on: the training stack
        m.eval()
        with torch.no_grad():
            ev = gpu(m, inp, want_grads=False)
    for k in ("x", "Z"):
        assert rel_err(ev[k], train[k]) < bound, k


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
def test_layer_level_api_with_node_attr_matches_oracle_layer(prec):
    cfg, params, inp = attr_case(5, C_=3, L=1)
    N, B = inp["node_loc"].size(0), 3
    g = torch.Generator().manual_seed(9)
    h = torch.randn(N, 64, generator=g)
    S = torch.randn(B, 64, 3, generator=g)
    p64 = {k: v.double() for k, v in params.items()}
    ref = spec.layer_forward(p64, "gcl_0", cfg, h.double(), inp["edge_index"], inp["node_loc"].double(),
                             inp["node_vel"].double(), inp["loc_mean"].double(), S.double(), inp["data_batch"],
                             inp["edge_attr"].double(), inp["node_attr"].double())
    m = build(cfg, params)
    with precision(prec) as tol:
        t = {k: v.to(DEV) for k, v in inp.items()}
        out = m.gcl_0(h.to(DEV), t["edge_index"], t["node_loc"], t["node_vel"], t["loc_mean"], S.to(DEV), t["data_batch"],
                      edge_attr=t["edge_attr"], node_attr=t["node_attr"])
        sum(o.sum() for o in out).backward()
        torch.cuda.synchronize()
    hn, xn, Sn, Zn = [o.detach().cpu() for o in out]
    assert rel_err(hn - h, ref[0] - h.double()) <= 4 * tol.out
    assert update_err(xn, ref[1], inp["node_loc"]) <= tol.out
    assert rel_err(Sn - S, ref[2] - S.double()) <= 4 * tol.out
    assert m.gcl_0.node_mlp[0].weight.grad is not None


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "tf32"])
def test_equivariance_with_invariant_attributes(prec):
    """equivariant_test.py's property with node attributes: invariant data, so f(xR + t) = f(x)R + t at atol 1e-4."""
    cfg = orc.OracleConfig(node_feat_nf=1, node_attr_nf=2, edge_attr_nf=1, virtual_channels=3)
    with precision(prec):
        for seed in range(3):
            g = torch.Generator().manual_seed(seed)
            m = build(cfg, orc.make_params(cfg, 60 + seed))
            N, E = 10, 20
            x, v = torch.rand(N, 3, generator=g) * 10, torch.rand(N, 3, generator=g) * 10
            nf, na = torch.rand(N, 1, generator=g) * 10, torch.rand(N, 2, generator=g) * 10
            ei = torch.randint(0, N, (2, E), generator=g)
            ea = torch.rand(E, 1, generator=g) * 10
            R, _ = torch.linalg.qr(torch.randn(3, 3, generator=g, dtype=torch.float64))
            if torch.det(R) < 0:
                R[:, 0] = -R[:, 0]
            R, t = R.float(), torch.randn(3, generator=g) * 5

            def run(xx, vv):
                lm = xx.mean(0).unsqueeze(-1).repeat(1, 3).unsqueeze(0)
                out, _ = m(node_feat=nf.to(DEV), node_loc=xx.to(DEV), node_vel=vv.to(DEV), edge_index=ei.to(DEV),
                           data_batch=torch.zeros(N, dtype=torch.long, device=DEV), loc_mean=lm.to(DEV),
                           edge_attr=ea.to(DEV), node_attr=na.to(DEV))
                return out.detach().cpu()
            a, b = run(x, v) @ R + t, run(x @ R + t, v @ R)
            assert torch.allclose(a, b, atol=1e-4), (seed, float((a - b).abs().max()))


def test_training_step_with_attributes_graph_replay_matches_eager_and_oracle():
    """A training step (MSE + 0.01 MMD, FusedAdam) with node attributes, captured as a CUDA graph and replayed, tracks the
    eager step and the oracle step (fp32 mode).  Not bitwise: the layer kernels add floats across CTAs in arrival order, so
    two runs differ within the run-to-run bound of DESIGN.md 3.2."""
    from fastegnn_b200 import FusedAdam, mmd_loss
    cfg, params, inp = attr_case(3, C_=3, sizes=(60, 60, 60, 60), deg=8, L=4)
    cfg_p = {k: v.clone() for k, v in params.items()}
    g = torch.Generator().manual_seed(5)
    target = inp["node_loc"] + 0.1 * torch.randn(inp["node_loc"].shape, generator=g)
    idx_local = torch.stack([torch.randperm(60, generator=g)[:9] for _ in range(4)])
    idx_global = (idx_local + torch.arange(4).unsqueeze(1) * 60).to(DEV)
    t = {k: v.to(DEV) for k, v in inp.items()}
    tgt = target.to(DEV)
    steps, warm = 3, 2
    with precision("fp32"):
        models = [build(cfg, params) for _ in range(2)]
        opts = [FusedAdam(m.parameters(), lr=5e-4, weight_decay=1e-12) for m in models]

        def step(i):
            opts[i].zero_grad(set_to_none=True)
            x, Z = models[i](node_feat=t["node_feat"], node_loc=t["node_loc"], node_vel=t["node_vel"],
                             edge_index=t["edge_index"], data_batch=t["data_batch"], loc_mean=t["loc_mean"],
                             edge_attr=t["edge_attr"], node_attr=t["node_attr"])
            loss = torch.nn.functional.mse_loss(x, tgt) + 0.01 * mmd_loss(x, Z, idx_global, 1.5)
            loss.backward()
            opts[i].step()
            return loss
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warm):
                step(1)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            gloss = step(1)
        eager, replayed = [], []
        for _ in range(warm):
            step(0)
        for _ in range(steps):
            eager.append(float(step(0)))
            graph.replay()
            replayed.append(float(gloss))
        torch.cuda.synchronize()
    p_ref = {k: v.double().requires_grad_(True) for k, v in cfg_p.items()}
    opt_ref = torch.optim.Adam(list(p_ref.values()), lr=5e-4, weight_decay=1e-12)
    d = lambda k: inp[k].double()
    ref = []
    for _ in range(warm + steps):
        opt_ref.zero_grad()
        xr, Zr = spec.oracle_forward(p_ref, cfg, d("node_feat"), d("node_loc"), d("node_vel"), inp["edge_index"],
                                     inp["data_batch"], d("loc_mean"), d("edge_attr"), d("node_attr"))
        lr = torch.nn.functional.mse_loss(xr, target.double()) + 0.01 * orc.mmd_loss(xr, Zr, inp["data_batch"], 1.5,
                                                                                      list(idx_local))
        lr.backward()
        opt_ref.step()
        ref.append(float(lr))
    for e, r, o in zip(eager, replayed, ref[warm:]):
        assert abs(e - r) <= 1e-6 * abs(o), (eager, replayed)
        assert abs(e - o) <= 1e-5 * max(1.0, abs(o)), (eager, ref)
    sd = [m.state_dict() for m in models]
    for k in sd[0]:
        assert torch.allclose(sd[0][k], sd[1][k], rtol=1e-4, atol=1e-6), k
    w = sd[0]["gcl_0.node_mlp.0.weight"].cpu()
    assert not torch.equal(w[:, -3:], params["gcl_0.node_mlp.0.weight"][:, -3:])   # the attribute columns train
    assert torch.equal(sd[0]["gcl_3.node_mlp.0.weight"].cpu(), params["gcl_3.node_mlp.0.weight"])   # dead in the last layer


def test_full_size_water3d_with_one_attribute():
    """The Water-3D shape of bench.py (8 000 nodes, C = 3, gravity) with Fa = 1, fp32 mode, judged on the update, the input
    gradients and the weight gradients.  Bias gradients are column sums over 8 000 nodes (x C) of signed terms that cancel
    (1.1e-4 observed for coord_mlp_v_virtual.0.bias against the stated 8e-5); test_gpu_fullsize.py judges them at this
    size without attributes."""
    import bench
    data = bench.make_cloud(8000, 25.0, 3, 0, [0, -1, 0])
    C_ = data["C"]
    cfg = orc.OracleConfig(node_feat_nf=2, node_attr_nf=1, edge_attr_nf=2, hidden_nf=64, virtual_channels=C_,
                           n_layers=4, gravity=data["gravity"])
    params = orc.make_params(cfg, 0)
    orc.rescale_coord_heads(params, 100.0)
    N, B = data["loc_0"].size(0), data["n_graphs"]
    g = torch.Generator().manual_seed(17)
    inp = dict(node_feat=data["node_feat"], node_loc=data["loc_0"], node_vel=data["vel_0"], loc_mean=data["loc_mean"],
               edge_attr=data["edge_attr"], edge_index=data["edge_index"], data_batch=data["batch"],
               node_attr=torch.rand(N, 1, generator=g), wx=torch.randn(N, 3, generator=g) / N,
               wz=torch.randn(B, 3, C_, generator=g) / B)
    torch.set_num_threads(os.cpu_count() or 1)
    ref = oracle(cfg, params, inp)
    with precision("fp32") as tol:
        res = gpu(build(cfg, params), inp)
    bad = [b for b in check_against_oracle(res, ref, inp, tol) if not b[0].endswith(".bias")]
    assert not bad, bad
    W, W_ref = res["gp"]["gcl_0.node_mlp.0.weight"], ref["gp"]["gcl_0.node_mlp.0.weight"]
    assert rel_err(W[:, -1:], W_ref[:, -1:]) <= tol.gw
