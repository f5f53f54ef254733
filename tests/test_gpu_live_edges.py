"""GPU: graphs whose edge count lives on the device (FEGNN_F_LIVE_EDGES; CsrGraph.from_radius(capacity=...) and
CsrGraph(..., n_edges=)).  A live graph of capacity E must give exactly the CSR arrays of the exact graph over its live
range, the model must compute on it what it computes on the exact graph (to summation order; bitwise in the deterministic
forward-only stack), whatever its padding holds, and a training step or a rollout that rebuilds its graph inside must
capture as ONE CUDA graph and replay over batches of different edge counts."""
import math

import pytest
import torch

from fastegnn_b200 import CsrGraph, FastEGNN, FastRF, FusedAdam, PipelinedStep, _lib, mse_mmd_loss
from tests.gpu_util import TOLERANCES, build_gpu_model, make_graph_case, precision

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
R = 0.035


def _cloud(seed, sizes, mean_deg=20.0, jitter=0.0):
    """Uniform clouds (one per graph) sized so that radius R gives `mean_deg` neighbours; jitter moves every point."""
    g = torch.Generator().manual_seed(seed)
    xs = []
    for n in sizes:
        side = (n * 4.0 / 3.0 * math.pi * R ** 3 / mean_deg) ** (1.0 / 3.0)
        xs.append(torch.rand(n, 3, generator=g) * side)
    x = torch.cat(xs)
    if jitter:
        x = x + jitter * R * torch.randn(x.shape, generator=g)
    batch = torch.cat([torch.full((n,), b, dtype=torch.long) for b, n in enumerate(sizes)])
    return x.to(DEV), batch.to(DEV)


def _same(a, b, what):
    assert a.dtype == b.dtype and a.shape == b.shape, what
    assert torch.equal(a, b), what


def _csr_equal(lv, ex, perm=False):
    E = ex.E
    assert lv.live and lv.num_edges() == E
    _same(lv.row[:E], ex.row[:E], "row")
    _same(lv.col[:E], ex.col[:E], "col")
    if ex.Fe:
        _same(lv.edge_attr[:E], ex.edge_attr[:E], "edge_attr")
    if perm:
        _same(lv.perm[:E], ex.perm[:E], "perm")
    for k in ("rowptr", "dinv", "batch", "gptr", "inv_nb"):
        _same(getattr(lv, k), getattr(ex, k), k)


def _pad(ei, ea, cap, N, seed):
    """edge_index / edge_attr padded to `cap` rows with valid but wrong entries (indices in range)."""
    g = torch.Generator().manual_seed(seed)
    extra = cap - ei.size(1)
    ei_p = torch.cat([ei.cpu(), torch.randint(0, N, (2, extra), generator=g)], dim=1)
    ea_p = torch.cat([ea.cpu(), 3.0 * torch.rand(extra, ea.size(1), generator=g)]) if ea is not None else None
    return ei_p.to(DEV), (None if ea_p is None else ea_p.to(DEV))


def _scramble_padding(lv, seed):
    """Overwrite the CSR padding of a live graph (row / col / edge_attr at and past the live count) with valid but wrong
    values: nothing may read them."""
    g = torch.Generator().manual_seed(seed)
    E, n = lv.num_edges(), lv.row.size(0)
    if n > E:
        lv.row[E:] = torch.randint(0, lv.N, (n - E,), generator=g).to(DEV, torch.int32)
        lv.col[E:] = torch.randint(0, lv.N, (n - E,), generator=g).to(DEV, torch.int32)
        if lv.Fe:
            lv.edge_attr[E:] = (5.0 * torch.rand(n - E, lv.Fe, generator=g)).to(DEV)


# ----------------------------------------------------------------------------- 1. graph construction
@pytest.mark.parametrize("cutoff", [0.0, 0.5])
@pytest.mark.parametrize("factor", [1.0, 1.3, 4.0])
def test_from_radius_with_capacity_is_the_exact_graph(cutoff, factor):
    """Capacities of factor x the larger of two graphs (factor 1: exactly its edge and candidate counts, which must not
    raise); the live graph is built on one and rebuilt in place on the other, in both orders."""
    x1, batch = _cloud(1, [700, 900, 500])
    x2, _ = _cloud(2, [700, 900, 500], jitter=0.05)
    ex1, ex2 = (CsrGraph.from_radius(x, batch, 3, R, cutoff, 2) for x in (x1, x2))
    assert ex1.E != ex2.E
    cap = math.ceil(factor * max(ex1.E, ex2.E))
    ccap = math.ceil(factor * max(ex1.n_candidates, ex2.n_candidates))
    for (xa, exa), (xb, exb) in (((x1, ex1), (x2, ex2)), ((x2, ex2), (x1, ex1))):
        lv = CsrGraph.from_radius(xa, batch, 3, R, cutoff, 2, capacity=cap, candidate_capacity=ccap)
        assert lv.E == cap
        lv.check()
        _csr_equal(lv, exa)
        assert torch.equal(lv.edge_index(), exa.edge_index())
        row_ptr = lv.row.data_ptr()
        lv.rebuild_(xb)                                  # the same buffers now hold the other graph
        assert lv.row.data_ptr() == row_ptr
        lv.check()
        _csr_equal(lv, exb)


def test_from_radius_undersized_capacities_raise_naming_the_size():
    x, batch = _cloud(3, [800, 600])
    ex = CsrGraph.from_radius(x, batch, 2, R, 0.5, 2)
    few_edges = CsrGraph.from_radius(x, batch, 2, R, 0.5, 2, capacity=ex.E - 1, candidate_capacity=ex.n_candidates)
    with pytest.raises(_lib.FegnnError, match=f"capacity >= {ex.E} is needed"):
        few_edges.check()
    few_cand = CsrGraph.from_radius(x, batch, 2, R, 0.5, 2, capacity=ex.E, candidate_capacity=ex.n_candidates - 1)
    with pytest.raises(_lib.FegnnError, match=f"candidate_capacity >= {ex.n_candidates} is needed"):
        few_cand.check()
    CsrGraph.from_radius(x, batch, 2, R, 0.5, 2, capacity=ex.E, candidate_capacity=ex.n_candidates).check()


@pytest.mark.parametrize("shape", ["fused", "general"])
@pytest.mark.parametrize("extra", [0, 77, -1])
def test_prep_live_over_padded_edges_is_exact(shape, extra):
    """fegnn_graph_prep_live on the short sort chain (Water-3D size) and on the general one (more than 262 144 edges, more
    than 12 160 nodes: the general counts chain too); extra = -1: capacity 3 E."""
    sizes, deg = ([300, 500, 200], 9) if shape == "fused" else ([21000], 14)
    cfg, _, inp = make_graph_case(seed=5, sizes=sizes, deg=deg, C=3)
    ei, ea, db = inp["edge_index"].to(DEV), inp["edge_attr"].to(DEV), inp["data_batch"].to(DEV)
    N, B, E = db.numel(), len(sizes), ei.size(1)
    ex = CsrGraph(ei, db, ea, B)
    cap = 3 * E if extra < 0 else E + extra
    ei_p, ea_p = _pad(ei, ea, cap, N, seed=6)
    for n_dtype in (torch.int32, torch.int64):
        lv = CsrGraph(ei_p, db, ea_p, B, n_edges=torch.tensor([E], dtype=n_dtype, device=DEV))
        lv.check()
        _csr_equal(lv, ex, perm=True)


def test_prep_live_bad_counts_raise():
    cfg, _, inp = make_graph_case(seed=7, sizes=[300, 200], deg=6, C=3)
    ei, ea, db = inp["edge_index"].to(DEV), inp["edge_attr"].to(DEV), inp["data_batch"].to(DEV)
    N, E = db.numel(), ei.size(1)
    ei_p, ea_p = _pad(ei, ea, E + 40, N, seed=8)
    over = CsrGraph(ei_p, db, ea_p, 2, n_edges=torch.tensor([E + 45], device=DEV))
    assert over.num_edges() == E + 40                    # clamped to the capacity
    with pytest.raises(_lib.FegnnError, match=f"a capacity of at least {E + 45} edges is needed"):
        over.check()
    neg = CsrGraph(ei_p, db, ea_p, 2, n_edges=torch.tensor([-3], device=DEV))
    assert neg.num_edges() == 0
    with pytest.raises(_lib.FegnnError, match="outside"):
        neg.check()


# ----------------------------------------------------------------------------- 2. / 4. model results on a live graph
CASES = {
    "base": dict(seed=21, sizes=[600, 900, 400], deg=10, C=3),
    "gravity": dict(seed=22, sizes=[700, 500], deg=10, C=3, gravity=[0.0, -1.0, 0.0]),
    "attention": dict(seed=23, sizes=[700, 500], deg=10, C=3, attention=True),     # fp32 edge kernels
    "wide_fe": dict(seed=24, sizes=[700, 500], deg=10, C=3, Fe=6),                 # Fe above the tensor-core limit
}


def _model(cls, cfg, params, seed):
    if cls is FastEGNN:
        return build_gpu_model(cfg, params, DEV)
    torch.manual_seed(seed)
    return FastRF(node_feat_nf=cfg.node_feat_nf, node_attr_nf=0, edge_attr_nf=cfg.edge_attr_nf, hidden_nf=64,
                  virtual_channels=cfg.virtual_channels, device=DEV, n_layers=cfg.n_layers, attention=cfg.attention,
                  normalize=cfg.normalize, tanh=cfg.tanh, gravity=cfg.gravity)


def _run(model, g, graph):
    leaf = {k: g[k].clone().requires_grad_(True) for k in ("node_loc", "loc_mean", "node_feat")}
    x, Z = model(node_feat=leaf["node_feat"], node_loc=leaf["node_loc"], node_vel=g["node_vel"], edge_index=graph,
                 data_batch=g["data_batch"], loc_mean=leaf["loc_mean"])
    model.zero_grad(set_to_none=True)
    ((x * g["wx"]).sum() + (Z * g["wz"]).sum()).backward()
    torch.cuda.synchronize()
    return dict(x=x.detach(), Z=Z.detach(), gin={k: t.grad for k, t in leaf.items()},
                gp={k: p.grad for k, p in model.named_parameters()})


def _rel(a, b):
    return float((a.double() - b.double()).abs().max() / (b.double().abs().max() + 1e-30))


def _compare(got, want, g, tol):
    """Live against exact, two runs that differ only in the order their float atomics add: each lies within the stated
    tolerance of the fp64 reference (gpu_util.TOLERANCES), so their distance is judged at twice that."""
    bad = []
    for k, base in (("x", g["node_loc"]), ("Z", g["loc_mean"])):
        upd = float((want[k] - base).abs().max())
        if float((got[k] - want[k]).abs().max()) > 2 * tol.out * upd + 8 * 2.0 ** -23 * float(want[k].abs().max()):
            bad.append(k)
    for k in want["gin"]:
        if _rel(got["gin"][k], want["gin"][k]) > 2 * tol.gin:
            bad.append("gin." + k)
    for k, w in want["gp"].items():
        if (w is None) != (got["gp"][k] is None):
            bad.append(k + " (grad presence)")
        elif w is not None:
            # a one-element gradient (coord_mlp_vel.2.bias: a sum over every node of signed terms that nearly cancel, like
            # the .gb tensors of gpu_util) is judged against the largest gradient entry of its module
            mod = k.rsplit(".", 2)[0] + "."
            scale = max(float(v.abs().max()) for n, v in want["gp"].items() if v is not None and n.startswith(mod)) \
                if w.numel() == 1 else float(w.abs().max())
            if float((got["gp"][k].double() - w.double()).abs().max()) > 2 * tol.for_param(k) * (scale + 1e-30):
                bad.append(k)
    return bad


def _graphs(inp, cap_extra=300, aligned=False):
    """(exact graph, live graph with scrambled padding) of one case's inputs."""
    ei, ea, db = inp["edge_index"].to(DEV), inp["edge_attr"].to(DEV), inp["data_batch"].to(DEV)
    if aligned:                                          # a live count that ends on an edge-tile boundary
        E = ei.size(1) - ei.size(1) % 128
        ei, ea = ei[:, :E].contiguous(), ea[:E].contiguous()
    N, B, E = db.numel(), int(inp["loc_mean"].size(0)), ei.size(1)
    if ea.size(1) == 0:
        ea = None
    ex = CsrGraph(ei, db, ea, B)
    ei_p, ea_p = _pad(ei, ea if ea is not None else torch.empty(E, 0, device=DEV), E + cap_extra, N, seed=E)
    lv = CsrGraph(ei_p, db, ea_p if ea is not None else None, B, n_edges=torch.tensor([E], device=DEV))
    _scramble_padding(lv, seed=E + 1)
    return ex, lv


@pytest.fixture
def modes():
    """Restores every mode this file's tests set."""
    names = list(_lib.PHASES) + ["layer_overlap", "grid_sms"]
    old = {n: _lib.get_mode(n) for n in names}
    yield _lib.set_mode
    for n, m in old.items():
        _lib.set_mode(n, m)


def _check_model(name, prec, cls=FastEGNN, recompute=False, aligned=False):
    cfg, params, inp = make_graph_case(**CASES[name])
    g = {k: v.to(DEV) for k, v in inp.items()}
    ex, lv = _graphs(inp, aligned=aligned)
    with precision(prec) as tol:
        model = _model(cls, cfg, params, CASES[name]["seed"])
        model.recompute = recompute
        want = _run(model, g, ex)
        got = _run(model, g, lv)
    bad = _compare(got, want, g, tol)
    assert not bad, f"{name} {prec} {cls.__name__}: live graph differs from the exact one in {bad}"


@pytest.mark.parametrize("cls", [FastEGNN, FastRF])
@pytest.mark.parametrize("prec", ["fp32", "tf32", "tf32x3", "tf32_all"])
def test_model_on_live_graph_matches_exact(prec, cls, modes):
    _check_model("base", prec, cls)


@pytest.mark.parametrize("name", ["gravity", "attention", "wide_fe"])
def test_layer_options_on_live_graph(name, modes):
    _check_model(name, "tf32")


@pytest.mark.parametrize("cls", [FastEGNN, FastRF])
def test_recompute_on_live_graph(cls, modes):
    _check_model("base", "tf32", cls, recompute=True)


@pytest.mark.parametrize("overlap", [0, 2])
@pytest.mark.parametrize("mode", [7, 8])
def test_edge_backward_modes_and_layer_overlap(mode, overlap, modes):
    modes("layer_overlap", overlap)
    with precision("tf32"):
        modes("edge_backward", mode)
        cfg, params, inp = make_graph_case(**CASES["base"])
        g = {k: v.to(DEV) for k, v in inp.items()}
        ex, lv = _graphs(inp)
        model = _model(FastEGNN, cfg, params, 0)
        want, got = _run(model, g, ex), _run(model, g, lv)
    assert not _compare(got, want, g, TOLERANCES["tf32"])


@pytest.mark.parametrize("aligned", [False, True])
@pytest.mark.parametrize("cap", [2, 3, 5])
def test_grid_caps_with_ragged_and_aligned_live_count(cap, aligned, modes):
    """Several tiles per CTA, CTAs past the live tiles, and a live count on an edge-tile boundary (the dynamic claim runs
    under layer_overlap 2)."""
    for ov in (0, 2):
        modes("grid_sms", cap)
        modes("layer_overlap", ov)
        _check_model("base", "tf32", aligned=aligned)


# ----------------------------------------------------------------------------- 3. deterministic forward-only stack
@pytest.fixture
def det():
    on, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    _lib.set_mode("deterministic", 0)


@pytest.mark.parametrize("cls", [FastEGNN, FastRF])
@pytest.mark.parametrize("prec", ["fp32", "tf32", "tf32x3"])
def test_deterministic_inference_is_bitwise_on_live_graph(prec, cls, det, modes):
    """The deterministic forms sum by tile and by chunk, never by CTA: the grid sized from the capacity changes no bit,
    and neither does the scrambled padding."""
    cfg, params, inp = make_graph_case(**CASES["base"])
    g = {k: v.to(DEV) for k, v in inp.items()}
    ex, lv = _graphs(inp)
    with precision(prec), torch.no_grad():
        model = _model(cls, cfg, params, 3).eval()
        args = dict(node_feat=g["node_feat"], node_loc=g["node_loc"], node_vel=g["node_vel"], data_batch=g["data_batch"],
                    loc_mean=g["loc_mean"])
        xe, Ze = model(edge_index=ex, **args)
        xl, Zl = model(edge_index=lv, **args)
    assert torch.equal(xe, xl) and torch.equal(Ze, Zl)


# ----------------------------------------------------------------------------- 5. / 6.
def test_zero_live_edges_matches_the_empty_graph(modes):
    cfg, params, inp = make_graph_case(seed=31, sizes=[300, 200], deg=4, C=3)
    g = {k: v.to(DEV) for k, v in inp.items()}
    r = 1e-6                                             # below every distance of the cloud
    ex = CsrGraph.from_radius(g["node_loc"], g["data_batch"], 2, r, 0.0, 2)
    lv = CsrGraph.from_radius(g["node_loc"], g["data_batch"], 2, r, 0.0, 2, capacity=256)
    assert ex.E == 0 and lv.num_edges() == 0
    lv.check()
    with precision("tf32") as tol:
        model = _model(FastEGNN, cfg, params, 0)
        want, got = _run(model, g, ex), _run(model, g, lv)
    assert not _compare(got, want, g, tol)


@pytest.mark.parametrize("mode", [1, 2, 4, 5])
def test_legacy_edge_backward_modes_refuse_a_live_graph(mode, modes):
    cfg, params, inp = make_graph_case(**CASES["base"])
    g = {k: v.to(DEV) for k, v in inp.items()}
    _, lv = _graphs(inp)
    model = _model(FastEGNN, cfg, params, 0)
    modes("edge_backward", mode)
    with pytest.raises(RuntimeError, match=f"edge_backward mode {mode}"):
        _run(model, g, lv)


# ----------------------------------------------------------------------------- 7. captured training
N_TRAIN, B_TRAIN, STEPS, WARM, LR = 1500, 2, 6, 2, 1e-3


def _batches():
    """STEPS + 1 batches of the same node count whose radius graphs differ (jittered positions)."""
    out = []
    for k in range(STEPS + 1):
        x, batch = _cloud(40 + k, [N_TRAIN // 2] * B_TRAIN, jitter=0.1 * k)
        gen = torch.Generator().manual_seed(k)
        v = (0.01 * torch.randn(N_TRAIN, 3, generator=gen)).to(DEV)
        out.append(dict(loc=x, vel=v, loc_t=x + v, batch=batch, feat=v.norm(dim=1, keepdim=True).repeat(1, 2),
                        loc_mean=torch.stack([x[batch == b].mean(0) for b in range(B_TRAIN)]).unsqueeze(-1).repeat(1, 1, 3)))
    idx = torch.stack([torch.randperm(N_TRAIN // 2, generator=torch.Generator().manual_seed(9))[:9] + b * (N_TRAIN // 2)
                       for b in range(B_TRAIN)]).to(torch.int32).to(DEV)
    return out, idx


def _fresh_model():
    torch.manual_seed(5)
    m = FastEGNN(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, hidden_nf=64, virtual_channels=3, device=DEV, n_layers=4,
                 gravity=[0.0, -1.0, 0.0])
    return m, FusedAdam(m.parameters(), lr=LR)


def _step(model, opt, t, graph, idx):
    opt.zero_grad(set_to_none=True)
    x, Z = model(node_feat=t["feat"], node_loc=t["loc"], node_vel=t["vel"], edge_index=graph, data_batch=t["batch"],
                 loc_mean=t["loc_mean"])
    loss, _ = mse_mmd_loss(x, t["loc_t"], Z, idx, 1.0, 0.01)
    loss.backward()
    opt.step()
    return loss.detach()


def _eager_reference(batches, idx):
    """WARM steps on batch 0, then every batch, each on its exact radius graph."""
    model, opt = _fresh_model()
    p0 = {k: p.detach().clone() for k, p in model.named_parameters()}
    losses = []
    for k, t in enumerate([batches[0]] * WARM + batches[:STEPS]):
        g = CsrGraph.from_radius(t["loc"], t["batch"], B_TRAIN, R, 0.0, 2)
        losses.append(float(_step(model, opt, t, g, idx)))
    return losses[WARM:], {k: p.detach() for k, p in model.named_parameters()}, p0


def _assert_training_matches(losses, params, ref_losses, ref_params, p0):
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= 1e-5 * abs(b), (losses, ref_losses)
    for k, w in ref_params.items():
        moved = float((w - p0[k]).abs().max())
        assert float((params[k] - w).abs().max()) <= 1e-3 * max(moved, LR), k


def test_captured_training_step_over_changing_edge_counts(modes):
    """One CUDA graph (radius graph built inside, forward, mse_mmd_loss, backward, FusedAdam) replayed over batches whose
    live E differs, against the same sequence run eagerly on exact graphs (fp32 kernels: summation order only)."""
    with precision("fp32"):
        batches, idx = _batches()
        Es = [CsrGraph.from_radius(t["loc"], t["batch"], B_TRAIN, R, 0.0, 2).E for t in batches[:STEPS]]
        assert len(set(Es)) >= 5, Es
        ref_losses, ref_params, p0 = _eager_reference(batches, idx)
        cap = int(1.5 * max(Es))
        model, opt = _fresh_model()
        static = {k: v.clone() for k, v in batches[0].items()}
        graphs = []

        def step():
            g = CsrGraph.from_radius(static["loc"], static["batch"], B_TRAIN, R, 0.0, 2, capacity=cap)
            graphs.append(g)
            return _step(model, opt, static, g, idx)

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(WARM):
                step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg):
            loss = step()
        losses = []
        for t in batches[:STEPS]:
            for k in static:
                static[k].copy_(t[k])
            cg.replay()
            losses.append(float(loss))
            graphs[-1].check()
        _assert_training_matches(losses, {k: p.detach() for k, p in model.named_parameters()}, ref_losses, ref_params, p0)


def test_pipelined_step_with_padded_host_edges(modes):
    """The same sequence through PipelinedStep: host edge lists padded to one capacity at collate time, with n_edges."""
    with precision("fp32"):
        batches, idx = _batches()
        ref_losses, ref_params, p0 = _eager_reference(batches, idx)
        graphs = [CsrGraph.from_radius(t["loc"], t["batch"], B_TRAIN, R, 0.0, 2) for t in batches[:STEPS]]
        cap = max(g.E for g in graphs) + 500
        host = []
        for t, g in zip(batches, graphs):
            E = g.E
            ei, ea = _pad(g.edge_index(), g.edge_attr[:E], cap, N_TRAIN, seed=E)
            h = {k: v.cpu().pin_memory() for k, v in t.items()}
            h.update(edge_index=ei.cpu().pin_memory(), edge_attr=ea.cpu().pin_memory(),
                     n_edges=torch.tensor([E], dtype=torch.int64).pin_memory())
            host.append(h)
        model, opt = _fresh_model()

        def step_fn(t):
            g = CsrGraph(t["edge_index"], t["batch"], t["edge_attr"], B_TRAIN, n_edges=t["n_edges"])
            return _step(model, opt, t, g, idx)

        pipe = PipelinedStep(step_fn, host[0], DEV, warmup=WARM)
        assert pipe.why is None and pipe.graphs[0] is not None, pipe.why
        losses = [pipe.run_and_read(host[k + 1] if k + 1 < STEPS else None) for k in range(STEPS)]
        _assert_training_matches(losses, {k: p.detach() for k, p in model.named_parameters()}, ref_losses, ref_params, p0)


# ----------------------------------------------------------------------------- 8. captured rollout
@pytest.mark.parametrize("deterministic", [False, True])
def test_captured_rollout_rebuilds_its_graph_every_step(deterministic, modes):
    steps = 10
    on, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(deterministic)
    try:
        with precision("tf32") as tol, torch.no_grad():
            batches, _ = _batches()
            t = batches[0]
            model, _ = _fresh_model()
            model.eval()
            args = dict(node_feat=t["feat"], node_vel=t["vel"], data_batch=t["batch"], loc_mean=t["loc_mean"])
            x = t["loc"]
            for _ in range(steps):                           # eager: the exact graph of every step's positions
                g = CsrGraph.from_radius(x, t["batch"], B_TRAIN, R, 0.0, 2)
                x, _ = model(node_loc=x, edge_index=g, **args)
            want = x.clone()
            cap = 2 * g.E
            x_in = t["loc"].clone()
            live = CsrGraph.from_radius(x_in, t["batch"], B_TRAIN, R, 0.0, 2, capacity=cap)

            def rollout():
                y = x_in
                for _ in range(steps):
                    live.rebuild_(y)
                    y, _ = model(node_loc=y, edge_index=live, **args)
                return y

            rollout()                                        # warm-up (eager)
            torch.cuda.synchronize()
            cg = torch.cuda.CUDAGraph()
            with torch.cuda.graph(cg):
                out = rollout()
            cg.replay()
            torch.cuda.synchronize()
            live.check()
        if deterministic:
            assert torch.equal(out, want)
        else:
            upd = float((want - t["loc"]).abs().max())
            assert float((out - want).abs().max()) <= 2 * tol.out * upd + 8 * 2.0 ** -23 * float(want.abs().max())
    finally:
        torch.use_deterministic_algorithms(on, warn_only=warn_only)
        _lib.set_mode("deterministic", 0)


# ----------------------------------------------------------------------------- Water-3D size, captured
def test_captured_water3d_step_on_live_graphs_at_several_capacities(modes):
    """bench.py's Water-3D step (8 000 particles, ~2e5 edges, default arithmetic, graph prep inside) captured four times in
    one process -- on its exact graph and on live graphs padded to 1.0x, 1.1x and 1.5x its edge count (short and general
    sort chains; grids with many CTAs past the live tiles) -- each graph with its own model, replayed back to back.  The
    live arms follow the exact one's loss."""
    import bench
    data, hp = bench.make_workload("water3d", seed=0, nodes=0)
    C, B = data["C"], data["n_graphs"]
    t = {k: data[k].to(DEV) for k in ("node_feat", "loc_0", "vel_0", "loc_t", "loc_mean", "batch", "edge_index",
                                         "edge_attr")}
    idx = bench.sample_indices(data["sizes"], 9, torch.Generator().manual_seed(0)).to(DEV)
    E = int(t["edge_index"].size(1))
    n_live = torch.tensor([E], dtype=torch.int32, device=DEV)
    arms = {}
    for f in (None, 1.0, 1.1, 1.5):
        torch.manual_seed(0)
        model = FastEGNN(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, hidden_nf=64, virtual_channels=C, device=DEV,
                         n_layers=4, gravity=data["gravity"])
        opt = FusedAdam(model.parameters(), lr=5e-4, weight_decay=1e-12)
        if f is not None:
            cap = int(round(f * E))
            ei = torch.cat([t["edge_index"], torch.zeros(2, cap - E, dtype=torch.int64, device=DEV)], dim=1)
            ea = torch.cat([t["edge_attr"], torch.zeros(cap - E, 2, device=DEV)])
        graphs = []

        def step(model=model, opt=opt, f=f, ei=(ei if f else None), ea=(ea if f else None), graphs=graphs):
            g = CsrGraph(t["edge_index"], t["batch"], t["edge_attr"], B) if f is None else \
                CsrGraph(ei, t["batch"], ea, B, n_edges=n_live)
            graphs.append(g)
            x, Z = model(node_feat=t["node_feat"], node_loc=t["loc_0"], node_vel=t["vel_0"], edge_index=g,
                         data_batch=t["batch"], loc_mean=t["loc_mean"])
            opt.zero_grad(set_to_none=True)
            loss, _ = mse_mmd_loss(x, t["loc_t"], Z, idx, hp["sigma"], hp["weight"])
            loss.backward()
            opt.step()
            return loss.detach()

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg):
            loss = step()
        arms[f] = (cg, loss, model, opt, graphs)
    losses = {}
    for f, (cg, loss, _, _, graphs) in arms.items():
        for _ in range(50):
            cg.replay()
        torch.cuda.synchronize()
        graphs[-1].check()
        losses[f] = float(loss)
    for f in (1.0, 1.1, 1.5):
        assert abs(losses[f] - losses[None]) <= 1e-4 * abs(losses[None]), losses


def test_layer_call_on_live_graph(modes):
    """The per-layer driver (layer_fn.layer_call, the phase entries) on a live graph: it passes FEGNN_F_LIVE_EDGES, so the
    phases read the live count and never the padding."""
    from fastegnn_b200.layer_fn import layer_call
    cfg, params, inp = make_graph_case(**CASES["base"])
    g = {k: v.to(DEV) for k, v in inp.items()}
    ex, lv = _graphs(inp)
    gen = torch.Generator().manual_seed(3)
    N, B, Cc = ex.N, ex.B, cfg.virtual_channels
    h = torch.randn(N, 64, generator=gen).to(DEV)
    S = torch.randn(B, Cc, 64, generator=gen).to(DEV)
    with precision("tf32") as tol:
        model = _model(FastEGNN, cfg, params, 0)
        named = {n: p.detach() for n, p in model.gcl_0.named_parameters()}
        outs = [layer_call(named, model._flag_word, model._gravity, Cc, graph, h, g["node_loc"], g["node_vel"],
                           g["loc_mean"], S) for graph in (ex, lv)]
        torch.cuda.synchronize()
    for name, a, b in zip(("h", "x", "S", "Z"), outs[0], outs[1]):
        assert _rel(b, a) <= 2 * tol.out + 1e-6, name
