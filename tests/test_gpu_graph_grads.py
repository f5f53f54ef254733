"""GPU: differentiable prebuilt graphs (CsrGraph.from_radius(..., differentiable=True), CsrGraph(..., differentiable=True)).

The edge-length backward (fegnn_edge_length_backward) against torch's fp64 autograd of norm; FastEGNN and FastRF on a
differentiable graph against the fp64 oracle of the torch composition (tests/graph_grads_spec.py) on the same edge list;
an unrolled rollout whose every step rebuilds its own live graph from the predicted positions; that rollout's training
step captured as one CUDA graph; and the guards (a rebuilt graph, the deterministic flag, the default off)."""
import ctypes as C
import math

import pytest
import torch

from fastegnn_b200 import CsrGraph, FastEGNN, FastRF, FusedAdam, _lib, mse_mmd_loss
from fastegnn_b200.ops import live_flag, make_dims
from oracle import fastegnn_oracle as orc
from oracle import fastrf_oracle as rfo
from tests import graph_grads_spec as spec
from tests.gpu_util import precision, rel_err
from tests.test_gpu_input_grads import PRECS, RUN_TO_RUN

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
R = 0.035
# Relative to the largest entry of the fp64 gradient, about twice the worst value observed on an NVIDIA B200 (1000 W) over
# every case below (DESIGN.md 3.10).  TOL_KERNEL: fegnn_edge_length_backward alone (3.9e-7 observed: fp32 lengths and
# sums).  node_loc / edge_attr: the input gradients of the model, rollout and CsrGraph cases; params: the worst parameter
# gradient of a case, each relative to its own largest entry.  The per-call route on the same inputs measures the same
# (its edge_attr and params errors equal the differentiable graph's to the printed digits); these cases are larger than
# test_gpu_input_grads.py's, whose TOL_IG params bound does not cover them.
TOL_KERNEL = 8e-7
TOL = {
    "fp32":     dict(node_loc=1.6e-6, edge_attr=2e-6, params=8.5e-5),
    "tf32x3":   dict(node_loc=1.2e-4, edge_attr=1.5e-3, params=1.4e-2),
    "tf32":     dict(node_loc=1.5e-4, edge_attr=1.4e-3, params=1.3e-2),
    "tf32_all": dict(node_loc=1.6e-4, edge_attr=1.6e-3, params=1.3e-2),
}


def check(tag, prec, key, err):
    """err (relative to the largest entry of the fp64 gradient) within the bound of this mode and input."""
    print(f"GRAPH_GRAD_ERR {tag} {prec} {key} {err:.3e}")
    assert err <= TOL[prec][key], (tag, prec, key, err)


@pytest.fixture
def modes():
    """Restores every library mode and torch's deterministic flag."""
    names = list(_lib.PHASES) + ["layer_overlap", "grid_sms", "deterministic"]
    old = {n: _lib.get_mode(n) for n in names}
    on, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    yield _lib.set_mode
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    for n, m in old.items():
        _lib.set_mode(n, m)


def cloud(seed, sizes, mean_deg=20.0, jitter=0.0, coincide=False):
    """Uniform clouds (one per graph) sized so that radius R gives about `mean_deg` neighbours; coincide: nodes 5 and 6
    of the first graph share a position (two edges of length 0)."""
    g = torch.Generator().manual_seed(seed)
    xs = []
    for n in sizes:
        side = (n * 4.0 / 3.0 * math.pi * R ** 3 / mean_deg) ** (1.0 / 3.0)
        xs.append(torch.rand(n, 3, generator=g) * side)
    x = torch.cat(xs)
    if jitter:
        x = x + jitter * R * torch.randn(x.shape, generator=g)
    if coincide:
        x[6] = x[5]
    batch = torch.cat([torch.full((n,), b, dtype=torch.long) for b, n in enumerate(sizes)])
    return x.to(DEV), batch.to(DEV)


def scramble_padding(graph, g_ea, seed):
    """Valid but wrong values in the CSR rows (and the g_ea rows) at and past a live graph's count: nothing may read them."""
    gen = torch.Generator().manual_seed(seed)
    E, n = graph.num_edges(), graph.row.size(0)
    if n > E:
        graph.row[E:] = torch.randint(0, graph.N, (n - E,), generator=gen).to(DEV, torch.int32)
        graph.col[E:] = torch.randint(0, graph.N, (n - E,), generator=gen).to(DEV, torch.int32)
        graph.edge_attr[E:] = (5.0 * torch.rand(n - E, graph.Fe, generator=gen)).to(DEV)
        g_ea[E:] = (100.0 * torch.randn(n - E, graph.Fe, generator=gen)).to(DEV)


# ----------------------------------------------------------------------------- 1. the kernel
def length_backward(graph, x, g_ea, g_x):
    dims = make_dims(graph.N, graph.N, graph.E, graph.B, 1, graph.Fe, live_flag(graph))
    _lib.check(_lib.lib.fegnn_edge_length_backward(C.byref(dims), C.byref(graph.c), _lib.ptr(graph.rowptr), _lib.ptr(x),
                                                   _lib.ptr(g_ea), _lib.ptr(g_x), torch.cuda.current_stream().cuda_stream),
               "fegnn_edge_length_backward")


@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("r", [R, math.inf])
@pytest.mark.parametrize("cutoff", [0.0, 0.5])
@pytest.mark.parametrize("kind", ["exact", "live1.0", "live1.5"])
def test_edge_length_backward_against_torch_norm(kind, cutoff, r, B, modes):
    """g_x += d/dx sum(g_ea * lengths(x)) on from_radius graphs: exact and live (scrambled padding), at the device grid and
    at grid caps of 2, 3 and 5 SMs (many rows per CTA); one pair of coincident nodes (zero lengths) in every graph."""
    sizes = ([300, 500, 200] if B == 3 else [600]) if r == R else ([40, 55, 30] if B == 3 else [70])
    x, batch = cloud(7 + B, sizes, coincide=True)
    for Fe in (1, 2, 8):
        ex = CsrGraph.from_radius(x, batch, B, r, cutoff, Fe)
        if kind == "exact":
            graph = ex
        else:
            f = 1.0 if kind == "live1.0" else 1.5
            graph = CsrGraph.from_radius(x, batch, B, r, cutoff, Fe, capacity=math.ceil(f * ex.E),
                                         candidate_capacity=math.ceil(f * ex.n_candidates))
            graph.check()
        E = graph.num_edges()
        assert E == ex.E and E > 0
        gen = torch.Generator().manual_seed(E + Fe)
        g_ea = torch.randn(graph.E, Fe, generator=gen).to(DEV)
        if graph.live:
            scramble_padding(graph, g_ea, seed=E)
        ei = graph.edge_index().cpu()
        zero = (ei[0] == 5) & (ei[1] == 6)
        assert bool(zero.any()), "the coincident pair is an edge"
        x64 = x.detach().cpu().double().requires_grad_(True)
        (spec.lengths(x64, ei, Fe) * g_ea[:E].cpu().double()).sum().backward()
        base = torch.randn(graph.N, 3, generator=gen).to(DEV)
        for cap in (0, 2, 3, 5):
            modes("grid_sms", cap)
            g_x = base.clone()
            length_backward(graph, x, g_ea, g_x)
            torch.cuda.synchronize()
            got = (g_x - base).cpu()
            assert torch.isfinite(got).all()
            err = rel_err(got, x64.grad)
            print(f"GRAPH_GRAD_ERR kernel {kind} cutoff={cutoff} r={r} B={B} Fe={Fe} cap={cap} {err:.3e}")
            assert err <= TOL_KERNEL, (Fe, cap, err)


# ----------------------------------------------------------------------------- 2. the model against the composition
def model_case(seed, rf=False, Fe=2, L=2, C_=3, gain=1000.0):
    cfg = orc.OracleConfig(node_feat_nf=2, edge_attr_nf=Fe, hidden_nf=64, virtual_channels=C_, n_layers=L)
    params = (rfo if rf else orc).make_params(cfg, seed + 1000)
    if gain != 1.0:
        orc.rescale_coord_heads(params, gain)
    return cfg, params


def build(cfg, params, rf=False):
    cls = FastRF if rf else FastEGNN
    m = cls(node_feat_nf=cfg.node_feat_nf, node_attr_nf=0, edge_attr_nf=cfg.edge_attr_nf, hidden_nf=64,
            virtual_channels=cfg.virtual_channels, device=DEV, n_layers=cfg.n_layers)
    m.load_state_dict({k: v.to(DEV) for k, v in params.items()})
    return m


def inputs(seed, sizes, C_, jitter=0.0):
    x, batch = cloud(seed, sizes, jitter=jitter)
    g = torch.Generator().manual_seed(seed + 1)
    N, B = x.size(0), len(sizes)
    lm = torch.stack([x[batch == b].mean(0) for b in range(B)]).unsqueeze(-1).repeat(1, 1, C_).cpu()
    return dict(x=x, batch=batch, B=B, feat=torch.rand(N, 2, generator=g).to(DEV),
                v=(0.002 * torch.randn(N, 3, generator=g)).to(DEV), lm=(lm + 0.003 * torch.randn(B, 3, C_, generator=g)).to(DEV),
                wx=torch.randn(N, 3, generator=g).to(DEV), wz=torch.randn(B, 3, C_, generator=g).to(DEV))


def oracle_grads(cfg, params, t, edge_indices, rf=False, dt=None):
    """fp64 autograd of sum(x_T * wx) + sum(Z_T * wz) through spec.rollout on the given edge lists (one step: dt unused)."""
    p64 = {k: v.double().requires_grad_(True) for k, v in params.items()}
    x64 = t["x"].cpu().double().requires_grad_(True)
    fwd = rfo.fastrf_forward if rf else orc.fastegnn_forward
    f = lambda x, v, ei, ea, lm: fwd(p64, cfg, t["feat"].cpu().double(), x, v, ei, t["batch"].cpu(), lm, ea)
    xo, Zo = spec.rollout(f, x64, t["v"].cpu().double(), t["lm"].cpu().double(), edge_indices, cfg.edge_attr_nf,
                          dt if dt is not None else 1.0)
    ((xo * t["wx"].cpu().double()).sum() + (Zo * t["wz"].cpu().double()).sum()).backward()
    return x64.grad, {k: p.grad for k, p in p64.items()}


def worst_param_err(m, gp64):
    worst = 0.0
    for k, p in m.named_parameters():
        if gp64[k] is not None and float(gp64[k].abs().max()) > 0:
            worst = max(worst, rel_err(p.grad.cpu(), gp64[k]))
    return worst


@pytest.mark.parametrize("rf", [False, True], ids=["FastEGNN", "FastRF"])
@pytest.mark.parametrize("prec", PRECS)
def test_model_on_differentiable_from_radius_matches_composition(prec, rf, modes):
    """x.grad and the parameter gradients on from_radius(x, differentiable=True), and on edge_index=graph.edge_index() with
    edge_attr=lengths(x) (the torch composition), against the fp64 oracle of that composition."""
    cfg, params = model_case(61, rf=rf)
    t = inputs(61, [400, 300], cfg.virtual_channels)
    ref_x, ref_p = None, None
    with precision(prec):
        m = build(cfg, params, rf)
        res = {}
        for arm in ("graph", "composition"):
            m.zero_grad(set_to_none=True)
            x = t["x"].clone().requires_grad_(True)
            if arm == "graph":
                graph = CsrGraph.from_radius(x, t["batch"], t["B"], R, 0.0, cfg.edge_attr_nf, differentiable=True)
                ei = graph.edge_index()
                kw = dict(edge_index=graph)
            else:
                kw = dict(edge_index=ei, edge_attr=spec.lengths(x, ei, cfg.edge_attr_nf))
            xo, Zo = m(node_feat=t["feat"], node_loc=x, node_vel=t["v"], data_batch=t["batch"], loc_mean=t["lm"], **kw)
            ((xo * t["wx"]).sum() + (Zo * t["wz"]).sum()).backward()
            torch.cuda.synchronize()
            if ref_x is None:
                ref_x, ref_p = oracle_grads(cfg, params, t, [ei.cpu()], rf=rf)
            res[arm] = x.grad.cpu()
            check(f"model_{arm}_{'rf' if rf else 'egnn'}", prec, "node_loc", rel_err(x.grad.cpu(), ref_x))
            check(f"model_{arm}_{'rf' if rf else 'egnn'}", prec, "params", worst_param_err(m, ref_p))
    assert rel_err(res["graph"], res["composition"]) <= 2 * TOL[prec]["node_loc"]


@pytest.mark.parametrize("live", [False, True], ids=["exact", "live"])
@pytest.mark.parametrize("prec", PRECS)
def test_differentiable_csr_graph_gives_edge_attr_its_gradient(prec, live, modes):
    """CsrGraph(edge_index, batch, edge_attr, B, differentiable=True) (and its padded live form): the caller's edge_attr gets
    the gradient of the per-call edge_index + edge_attr route, in the caller's edge order."""
    cfg, params = model_case(63)
    t = inputs(63, [400, 300], cfg.virtual_channels)
    ex = CsrGraph.from_radius(t["x"], t["batch"], t["B"], R, 0.0, 2)
    gen = torch.Generator().manual_seed(64)
    E = ex.E
    perm = torch.randperm(E, generator=gen).to(DEV)
    ei = ex.edge_index()[:, perm]                              # unsorted: the graph's perm is exercised
    ea = (ex.edge_attr[:E][perm] * (0.5 + torch.rand(1, 2, generator=gen).to(DEV))).contiguous()
    p64 = {k: v.double() for k, v in params.items()}
    ea64 = ea.cpu().double().requires_grad_(True)
    x64, Z64 = orc.fastegnn_forward(p64, cfg, t["feat"].cpu().double(), t["x"].cpu().double(), t["v"].cpu().double(),
                                    ei.cpu(), t["batch"].cpu(), t["lm"].cpu().double(), ea64)
    ((x64 * t["wx"].cpu().double()).sum() + (Z64 * t["wz"].cpu().double()).sum()).backward()
    with precision(prec):
        m = build(cfg, params)
        res = {}
        for arm in ("graph", "per_call"):
            leaf = ea.clone().requires_grad_(True)
            args = dict(node_feat=t["feat"], node_loc=t["x"], node_vel=t["v"], data_batch=t["batch"], loc_mean=t["lm"])
            if arm == "graph" and live:
                cap = E + 333
                ei_p = torch.cat([ei, torch.randint(0, ex.N, (2, cap - E), generator=gen).to(DEV)], dim=1)
                ea_full = torch.cat([leaf, 3.0 * torch.rand(cap - E, 2, generator=gen).to(DEV)])
                graph = CsrGraph(ei_p, t["batch"], ea_full, t["B"], n_edges=torch.tensor([E], device=DEV),
                                 differentiable=True)
                xo, Zo = m(edge_index=graph, **args)
            elif arm == "graph":
                xo, Zo = m(edge_index=CsrGraph(ei, t["batch"], leaf, t["B"], differentiable=True), **args)
            else:
                xo, Zo = m(edge_index=ei, edge_attr=leaf, **args)
            ((xo * t["wx"]).sum() + (Zo * t["wz"]).sum()).backward()
            torch.cuda.synchronize()
            assert leaf.grad is not None and leaf.grad.shape == ea.shape
            res[arm] = leaf.grad.cpu()
            check(f"csr_graph_{arm}_{'live' if live else 'exact'}", prec, "edge_attr", rel_err(leaf.grad.cpu(), ea64.grad))
    assert rel_err(res["graph"], res["per_call"]) <= 2 * TOL[prec]["edge_attr"]


# ----------------------------------------------------------------------------- 3. unrolled rollout
STEPS, DT = 3, 0.5


def rollout_gpu(m, t, x0, graphs, capacity):
    """STEPS steps, each rebuilding its own live graph from the predicted positions (graphs: a list that is filled on the
    first call and rebuilt in place afterwards)."""
    x, v, Z = x0, t["v"], t["lm"]
    for s in range(STEPS):
        if len(graphs) <= s:
            graphs.append(CsrGraph.from_radius(x, t["batch"], t["B"], R, 0.0, 2, capacity=capacity, differentiable=True))
        else:
            graphs[s].rebuild_(x)
        x_new, Z = m(node_feat=t["feat"], node_loc=x, node_vel=v, edge_index=graphs[s], data_batch=t["batch"], loc_mean=Z)
        x, v = x_new, (x_new - x) / DT
    return x, Z


@pytest.mark.parametrize("prec", PRECS)
def test_unrolled_rollout_on_live_graphs_matches_oracle(prec, modes):
    cfg, params = model_case(71, gain=100.0)
    t = inputs(71, [500, 400], cfg.virtual_channels)
    cap = 3 * CsrGraph.from_radius(t["x"], t["batch"], t["B"], R, 0.0, 2).E
    with precision(prec):
        m = build(cfg, params)
        x0 = t["x"].clone().requires_grad_(True)
        graphs = []
        xo, Zo = rollout_gpu(m, t, x0, graphs, cap)
        ((xo * t["wx"]).sum() + (Zo * t["wz"]).sum()).backward()
        torch.cuda.synchronize()
    for g in graphs:
        g.check()
    eis = [g.edge_index().cpu() for g in graphs]
    print("GRAPH_GRAD rollout edge counts", [e.size(1) for e in eis])
    ref_x, ref_p = oracle_grads(cfg, params, t, eis, dt=DT)
    check("rollout", prec, "node_loc", rel_err(x0.grad.cpu(), ref_x))
    check("rollout", prec, "params", worst_param_err(m, ref_p))


# ----------------------------------------------------------------------------- 4. captured rollout training step
def test_captured_rollout_training_step_matches_eager(modes):
    """One CUDA graph of a 3-step rollout training step (rebuild_ of each step's live graph, forward, mse_mmd_loss,
    backward, FusedAdam), replayed over initial states whose edge counts differ, against the same step run eagerly."""
    base = inputs(80, [600, 500], 3)
    states = [dict(base, x=cloud(80, [600, 500], jitter=0.1 * k)[0]) for k in range(4)]
    Es = [CsrGraph.from_radius(s["x"], s["batch"], 2, R, 0.0, 2).E for s in states]
    assert len(set(Es)) == len(Es), Es
    cap = int(1.5 * max(Es))
    idx = torch.stack([torch.randperm(500, generator=torch.Generator().manual_seed(9))[:9] + b * 600
                       for b in range(2)]).to(torch.int32).to(DEV)

    def fresh():
        torch.manual_seed(5)
        m = FastEGNN(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, hidden_nf=64, virtual_channels=3, device=DEV,
                     n_layers=2)
        return m, FusedAdam(m.parameters(), lr=1e-3)

    def make_step(m, opt, t, graphs):
        def step():
            opt.zero_grad(set_to_none=True)
            xo, Zo = rollout_gpu(m, t, t["x"], graphs, cap)
            loss, _ = mse_mmd_loss(xo, t["target"], Zo, idx, 1.0, 0.01)
            loss.backward()
            opt.step()
            return loss.detach()
        return step

    for s in states:
        s["target"] = s["x"] + 0.01
    with precision("fp32"):
        m, opt = fresh()
        p0 = {k: p.detach().clone() for k, p in m.named_parameters()}
        ref_losses = []
        for s in [states[0], states[0]] + states:            # two warm-up steps, then every state
            ref_losses.append(float(make_step(m, opt, s, [])()))
        ref_losses = ref_losses[2:]
        ref_params = {k: p.detach().clone() for k, p in m.named_parameters()}

        m, opt = fresh()
        static = {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in states[0].items()}
        graphs = []
        step = make_step(m, opt, static, graphs)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg):
            loss = step()
        losses = []
        for s in states:
            for k in ("x", "target"):
                static[k].copy_(s[k])
            cg.replay()
            losses.append(float(loss))
            for g in graphs:
                g.check()
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= RUN_TO_RUN["fp32"] * abs(b), (losses, ref_losses)
    for k, w in ref_params.items():
        moved = float((w - p0[k]).abs().max())
        assert float((m.state_dict()[k] - w).abs().max()) <= 1e-3 * max(moved, 1e-3), k


# ----------------------------------------------------------------------------- 5. guards and defaults
def _forward(m, t, graph, x):
    return m(node_feat=t["feat"], node_loc=x, node_vel=t["v"], edge_index=graph, data_batch=t["batch"], loc_mean=t["lm"])


def test_graph_rebuilt_before_backward_raises(modes):
    cfg, params = model_case(91)
    t = inputs(91, [400, 300], 3)
    m = build(cfg, params)
    x = t["x"].clone().requires_grad_(True)
    cap = 2 * CsrGraph.from_radius(t["x"], t["batch"], 2, R, 0.0, 2).E
    graph = CsrGraph.from_radius(x, t["batch"], 2, R, 0.0, 2, capacity=cap, differentiable=True)
    xo, Zo = _forward(m, t, graph, x)
    graph.rebuild_(t["x"] + 0.01)
    with pytest.raises(_lib.FegnnError, match="rebuilt"):
        ((xo * t["wx"]).sum() + (Zo * t["wz"]).sum()).backward()


def test_deterministic_flag_raises_or_warns(modes):
    cfg, params = model_case(92)
    t = inputs(92, [400, 300], 3)
    m = build(cfg, params)
    for warn_only in (False, True):
        x = t["x"].clone().requires_grad_(True)
        graph = CsrGraph.from_radius(x, t["batch"], 2, R, 0.0, 2, differentiable=True)
        xo, Zo = _forward(m, t, graph, x)
        torch.use_deterministic_algorithms(True, warn_only=warn_only)
        loss = (xo * t["wx"]).sum() + (Zo * t["wz"]).sum()
        if warn_only:
            with pytest.warns(UserWarning, match="CsrGraph edge-length backward"):
                loss.backward()
            torch.cuda.synchronize()
            assert x.grad is not None and torch.isfinite(x.grad).all()
        else:
            with pytest.raises(RuntimeError, match="deterministic"):
                loss.backward()
        torch.use_deterministic_algorithms(False)
        _lib.set_mode("deterministic", 0)


def test_default_graph_is_data_and_launches_what_it_did(modes):
    """differentiable=False: x.grad is the direct path's only (as with a detached edge_attr per call), and the forward +
    backward launches exactly the kernels of a differentiable graph whose positions need no gradient."""
    cfg, params = model_case(93)
    t = inputs(93, [400, 300], 3)
    with precision("fp32"):
        m = build(cfg, params)
        got, counts = {}, {}
        for arm in ("default", "per_call_data", "differentiable_no_grad"):
            m.zero_grad(set_to_none=True)
            x = t["x"].clone().requires_grad_(arm != "differentiable_no_grad")
            graph = CsrGraph.from_radius(t["x"], t["batch"], 2, R, 0.0, 2,
                                         differentiable=arm == "differentiable_no_grad")
            ei = graph.edge_index()
            torch.cuda.synchronize()
            n0 = int(_lib.lib.fegnn_launch_count())
            if arm == "per_call_data":
                xo, Zo = m(node_feat=t["feat"], node_loc=x, node_vel=t["v"], edge_index=ei, data_batch=t["batch"],
                           loc_mean=t["lm"], edge_attr=graph.edge_attr)
            else:
                xo, Zo = _forward(m, t, graph, x)
            ((xo * t["wx"]).sum() + (Zo * t["wz"]).sum()).backward()
            torch.cuda.synchronize()
            counts[arm] = int(_lib.lib.fegnn_launch_count()) - n0
            got[arm] = None if x.grad is None else x.grad.cpu()
    assert rel_err(got["default"], got["per_call_data"]) <= RUN_TO_RUN["fp32"]
    assert counts["default"] == counts["differentiable_no_grad"], counts
