"""FastEGNN.recompute / FastRF.recompute (FEGNN_F_RECOMPUTE, DESIGN.md 3.8): the training stack keeps the layer states and
two saved blocks, and its backward rebuilds each layer's block from the layer's input state.  The recomputed blocks are
the forward's up to the order of float sums.  So a step with recompute matches the fp64 oracle within the stated bounds
of every arithmetic mode (tests/gpu_util.TOLERANCES); only the 5-layer case in the tensor-core modes, where the default
stack's own error already exceeds them, is held to 1.25 times the default's error, with that error itself capped near its
recorded value (DEFAULT_ERR_L5).  A second backward over the same forward (retain_graph) gives the first one's gradients.  On the fp32 kernels it also matches the default stack within 1e-5 of each tensor's largest entry, or
within four times the default's run-to-run spread for a tensor whose sums cancel."""
import contextlib
import dataclasses

import pytest
import torch

from oracle import fastegnn_oracle as orc
from tests import node_attr_spec as spec
from tests.gpu_util import TOLERANCES, make_graph_case, precision, rel_err, update_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
INPUTS = ("node_loc", "node_vel", "loc_mean", "node_feat", "edge_attr", "node_attr")
VS_DEFAULT_FP32 = 1e-5          # recompute vs the default stack on the fp32 kernels, relative to each tensor's max
RUN_TO_RUN = 1e-3               # a second run of a step in the tensor-core modes (tests/test_gpu_input_grads.py)
# The default stack's own error against the fp64 oracle in the 5-layer case (deeper than the cases the TOLERANCES were set on,
# L <= 4): its largest value over every output and gradient, NVIDIA B200.  Input gradients exceed TOLERANCES.gin there
# (tf32: node_loc 1.20e-2, node_vel 8.9e-3, node_feat 1.68e-2; tf32x3: 7.5e-3 / 7.0e-3 / 1.26e-2, and the x update 5.6e-6;
# tf32_all: 1.36e-2 / 1.03e-2 / 1.89e-2).  Recompute measured within 0.94-1.05 times the default's error on every tensor.
DEFAULT_ERR_L5 = {"tf32": 1.7e-2, "tf32x3": 1.3e-2, "tf32_all": 1.9e-2}
DEFAULT_ERR_FACTOR = 1.25       # recompute vs the default's error where the fallback applies

# name -> (make_graph_case arguments, extra: rf / Fa)
CASES = {
    # Water-3D size: 8 000 nodes, ~180 k edges, C = 3, gravity, 4 layers
    "water3d": (dict(seed=3, sizes=[8000], deg=22, C=3, L=4, gravity=[0, -1, 0]), {}),
    # a batch of 20 graphs (water3d_b20-like sizes)
    "batch20": (dict(seed=11, sizes=[400 + 13 * i for i in range(20)], deg=14, C=3, L=4), {}),
    # one large graph at C = 8 (config-5 channel count)
    "n100k_c8": (dict(seed=12, sizes=[100_000], deg=8, C=8, L=3), {}),
    # rows with thousands of edges (span several edge tiles)
    "hub_rows": (dict(seed=13, sizes=[900, 600], deg=6, C=3, L=3, heavy_row=3000), {}),
    "attention": (dict(seed=14, sizes=[300, 250, 410], deg=9, C=3, L=3, attention=True), {}),
    "normalize_tanh": (dict(seed=15, sizes=[500, 350], deg=9, C=4, L=3, normalize=True, tanh=True, gravity=[0, 0, -1]), {}),
    "fe0": (dict(seed=16, sizes=[600, 420], deg=8, C=3, L=3, Fe=0), {}),
    "node_attr3": (dict(seed=17, sizes=[520, 380], deg=8, C=3, L=3), dict(Fa=3)),
    "fastrf": (dict(seed=18, sizes=[500, 450], deg=9, C=3, L=4), dict(rf=True)),
    "L1": (dict(seed=19, sizes=[300, 200, 250], deg=9, C=3, L=1), {}),
    "L2": (dict(seed=20, sizes=[700, 300], deg=9, C=3, L=2), {}),
    "L5": (dict(seed=21, sizes=[800, 650, 300], deg=10, C=3, L=5, gravity=[0, -1, 0]), {}),
}
PRECS = {name: ["fp32", "tf32"] for name in CASES}
PRECS["water3d"] += ["tf32x3", "tf32_all"]
PRECS["L5"] += ["tf32x3", "tf32_all"]


@contextlib.contextmanager
def overlap(mode):
    from fastegnn_b200 import _lib
    old = _lib.get_mode("layer_overlap")
    _lib.set_mode("layer_overlap", mode)
    try:
        yield
    finally:
        _lib.set_mode("layer_overlap", old)


_cases = {}


def case(name):
    """(cfg, params, inp, rf) of a case, with its fp64 oracle gradients (cached: the oracle runs once per case)."""
    if name not in _cases:
        kw, extra = dict(CASES[name][0]), CASES[name][1]
        cfg, params, inp = make_graph_case(kw.pop("seed"), kw.pop("sizes"), kw.pop("deg"), kw.pop("C"), **kw)
        rf, Fa = extra.get("rf", False), extra.get("Fa", 0)
        seed = CASES[name][0]["seed"]
        if rf:
            from oracle import fastrf_oracle as rfo
            params = rfo.make_params(cfg, seed + 1000)
            orc.rescale_coord_heads(params, 1000.0)
        if Fa:
            cfg = dataclasses.replace(cfg, node_attr_nf=Fa)
            params = orc.make_params(cfg, seed + 1000)
            orc.rescale_coord_heads(params, 1000.0)
            g = torch.Generator().manual_seed(seed + 7)
            inp = dict(inp, node_attr=torch.randn(inp["node_loc"].size(0), Fa, generator=g))
        if inp["edge_attr"].size(1) > 1:        # make_graph_case repeats the edge length: tell the columns apart
            g = torch.Generator().manual_seed(seed + 5)
            inp = dict(inp, edge_attr=inp["edge_attr"] * (0.5 + torch.rand(1, inp["edge_attr"].size(1), generator=g)))
        _cases[name] = (cfg, params, inp, rf, oracle(cfg, params, inp, rf))
    return _cases[name]


def wanted(inp, rf):
    """The inputs that receive a gradient: FastRF's velocity enters through |v| and has none."""
    return tuple(k for k in INPUTS if inp.get(k) is not None and inp[k].numel() > 0 and not (rf and k == "node_vel"))


def oracle(cfg, params, inp, rf):
    """fp64 outputs and autograd of sum(x * wx) + sum(Z * wz) with respect to every float input and parameter."""
    p = {k: v.double().requires_grad_(True) for k, v in params.items()}
    leaf = {k: inp[k].double().requires_grad_(True) for k in wanted(inp, rf)}
    d = lambda k: leaf[k] if k in leaf else inp[k].double()
    args = (d("node_feat"), d("node_loc"), d("node_vel"), inp["edge_index"], inp["data_batch"], d("loc_mean"),
            d("edge_attr"))
    if rf:
        from oracle import fastrf_oracle as rfo
        x, Z = rfo.fastrf_forward(p, cfg, *args)
    elif "node_attr" in inp:
        x, Z = spec.oracle_forward(p, cfg, *args, d("node_attr"))
    else:
        x, Z = orc.fastegnn_forward(p, cfg, *args)
    ((x * inp["wx"].double()).sum() + (Z * inp["wz"].double()).sum()).backward()
    out = {"x": x.detach(), "Z": Z.detach()}
    out.update({"input." + k: t.grad for k, t in leaf.items()})
    out.update({"grad." + k: t.grad for k, t in p.items()})
    return out


def build(cfg, params, rf, recompute):
    from fastegnn_b200 import FastEGNN, FastRF
    m = (FastRF if rf else FastEGNN)(node_feat_nf=cfg.node_feat_nf, node_attr_nf=getattr(cfg, "node_attr_nf", 0),
                                     edge_attr_nf=cfg.edge_attr_nf, hidden_nf=64, virtual_channels=cfg.virtual_channels,
                                     device=DEV, n_layers=cfg.n_layers, attention=cfg.attention,
                                     normalize=cfg.normalize, tanh=cfg.tanh, gravity=cfg.gravity)
    m.load_state_dict({k: v.to(DEV) for k, v in params.items()})
    m.recompute = recompute
    return m


def step(m, inp, rf):
    """Outputs, parameter gradients and input gradients of one forward + backward of sum(x * wx) + sum(Z * wz)."""
    t = {k: (None if v is None else v.to(DEV)) for k, v in inp.items()}
    want = wanted(inp, rf)
    leaf = {k: t[k].clone().requires_grad_(k in want) for k in INPUTS if t.get(k) is not None}
    m.zero_grad(set_to_none=True)
    kw = {"node_attr": leaf["node_attr"]} if "node_attr" in leaf else {}
    x, Z = m(node_feat=leaf["node_feat"], node_loc=leaf["node_loc"], node_vel=leaf["node_vel"],
             edge_index=t["edge_index"], data_batch=t["data_batch"], loc_mean=leaf["loc_mean"],
             edge_attr=leaf.get("edge_attr") if inp["edge_attr"].size(1) else None, **kw)
    ((x * t["wx"]).sum() + (Z * t["wz"]).sum()).backward()
    torch.cuda.synchronize()
    out = {"x": x.detach().cpu(), "Z": Z.detach().cpu()}
    out.update({"input." + k: leaf[k].grad.cpu() for k in want})
    out.update({"grad." + k: p.grad.cpu() for k, p in m.named_parameters() if p.grad is not None})
    return out


def check_oracle(tag, got, ref, inp, tol, dflt=None, cap=None):
    """got vs the fp64 oracle within the stated bounds.  dflt / cap (the 5-layer case in the tensor-core modes only): where
    the default stack's error of the same step exceeds a stated bound, recompute is held to DEFAULT_ERR_FACTOR times that
    error instead -- and the default's error must stay within 1.5 cap, so that a growing error of both cannot pass."""
    def fallback(e0):
        if dflt is None:
            return 0.0
        assert e0 <= 1.5 * cap, (tag, "default stack's own error", e0, cap)
        return DEFAULT_ERR_FACTOR * e0
    assert set(k for k in got if k.startswith("input.")) == set(k for k in ref if k.startswith("input.")), tag
    bad = []
    for k, base in (("x", inp["node_loc"]), ("Z", inp["loc_mean"])):
        e = update_err(got[k], ref[k], base)
        e0 = update_err(dflt[k], ref[k], base) if dflt is not None else 0.0
        print(f"RECOMPUTE_ORACLE {tag} {k} {e:.3e} default {e0:.3e}")
        if e > max(tol.out, fallback(e0)):
            bad.append((k, e, e0))
    for k, r in ref.items():
        if k in ("x", "Z"):
            continue
        if r is None or not bool(r.abs().max() > 0):          # no gradient in the reference (the last layer's phi_h)
            assert k not in got or not bool(got[k].abs().max() > 0), k
            continue
        e = rel_err(got[k], r)
        e0 = rel_err(dflt[k], r) if dflt is not None else 0.0
        # edge_attr's gradient is a sum over the edge backward's gz1 like a weight gradient's (fp16 gz1 in the tensor-core
        # modes): it is held to the weight-gradient bound
        bound = tol.for_param(k[5:]) if k.startswith("grad.") else (tol.gw if k == "input.edge_attr" else tol.gin)
        print(f"RECOMPUTE_ORACLE {tag} {k} {e:.3e} default {e0:.3e}")
        if e > max(bound, fallback(e0)):
            bad.append((k, e, e0))
    assert not bad, (tag, bad)


def check_same(tag, got, ref, bound, ref2=None):
    """got vs ref within `bound` of each tensor's max.  With a second run of the reference (ref2), a tensor whose two
    reference runs already differ by more than bound / 4 (float sums in arrival order that cancel, e.g. the first layer's
    att_mlp.0.weight gradient: 3.4e-5 on the B200) is held to four times that spread instead."""
    assert got.keys() == ref.keys(), tag
    bad = []
    for k in ref:
        e = rel_err(got[k], ref[k])
        spread = rel_err(ref2[k], ref[k]) if ref2 is not None else 0.0
        if e > max(bound, 4 * spread):
            bad.append((k, e, spread))
    worst = max((rel_err(got[k], ref[k]), k) for k in ref)
    print(f"RECOMPUTE_VS_DEFAULT {tag} {worst[1]} {worst[0]:.3e}")
    assert not bad, (tag, bad)


@pytest.mark.parametrize("name,prec", [(n, p) for n in CASES for p in PRECS[n]])
def test_recompute_matches_oracle_and_default(name, prec):
    cfg, params, inp, rf, ref = case(name)
    with precision(prec) as tol:
        got = step(build(cfg, params, rf, True), inp, rf)
        m = build(cfg, params, rf, False)
        dflt = step(m, inp, rf)
        deep = name == "L5" and prec != "fp32"
        check_oracle(f"{name} {prec}", got, ref, inp, tol, dflt if deep else None, DEFAULT_ERR_L5.get(prec))
        if prec == "fp32":
            check_same(f"{name} {prec}", got, dflt, VS_DEFAULT_FP32, step(m, inp, rf))


@pytest.mark.parametrize("mode", [0, 2])
def test_recompute_in_both_backward_arrangements(mode):
    """layer_overlap 0 (virtual backward after the edge backward) and 2 (next to it, on a second stream): the recompute of
    layer l - 1 is issued between those of layer l's backward."""
    cfg, params, inp, rf, ref = case("water3d")
    with precision("tf32") as tol, overlap(mode):
        got = step(build(cfg, params, rf, True), inp, rf)
        check_oracle(f"water3d overlap{mode}", got, ref, inp, tol)
        check_same(f"water3d overlap{mode}", got, step(build(cfg, params, rf, False), inp, rf), RUN_TO_RUN)


@pytest.mark.parametrize("name", ["L5", "fastrf", "L2"])
def test_repeated_backward_over_one_forward(name):
    """loss.backward(retain_graph=True) twice and torch.autograd.grad after them, over ONE recompute forward: the first
    backward rebuilds the lower layers into the blocks the forward left holding the top two, so the later ones rebuild
    every layer (FEGNN_F_REBUILD_ALL).  Each gives the first one's gradients, within the default stack's run-to-run spread."""
    cfg, params, inp, rf, ref = case(name)
    with precision("fp32") as tol:
        m = build(cfg, params, rf, True)
        t = {k: v.to(DEV) for k, v in inp.items()}
        x0 = t["node_loc"].clone().requires_grad_(True)
        x, Z = m(node_feat=t["node_feat"], node_loc=x0, node_vel=t["node_vel"], edge_index=t["edge_index"],
                 data_batch=t["data_batch"], loc_mean=t["loc_mean"], edge_attr=t["edge_attr"])
        loss = (x * t["wx"]).sum() + (Z * t["wz"]).sum()
        params_ = [p for _, p in m.named_parameters()]
        runs = []
        for _ in range(2):
            m.zero_grad(set_to_none=True)
            x0.grad = None
            loss.backward(retain_graph=True)
            torch.cuda.synchronize()
            runs.append([x0.grad.cpu()] + [None if p.grad is None else p.grad.cpu() for p in params_])
        gs = torch.autograd.grad(loss, [x0] + params_, allow_unused=True)
        runs.append([None if g is None else g.cpu() for g in gs])
        # the default stack, twice, for the spread of its float sums
        md = build(cfg, params, rf, False)
        spread = []
        for _ in range(2):
            xd, Zd = md(node_feat=t["node_feat"], node_loc=x0, node_vel=t["node_vel"], edge_index=t["edge_index"],
                        data_batch=t["data_batch"], loc_mean=t["loc_mean"], edge_attr=t["edge_attr"])
            spread.append([g.cpu() if g is not None else None for g in torch.autograd.grad(
                (xd * t["wx"]).sum() + (Zd * t["wz"]).sum(), [x0] + [p for _, p in md.named_parameters()], allow_unused=True)])
    names = ["input.node_loc"] + ["grad." + k for k, _ in m.named_parameters()]
    for i, k in enumerate(names):
        first = runs[0][i]
        if first is None:
            assert all(r[i] is None for r in runs), k
            continue
        sp = rel_err(spread[1][i], spread[0][i])
        for j, r in enumerate(runs[1:], 1):
            e = rel_err(r[i], first)
            assert e <= max(VS_DEFAULT_FP32, 4 * sp), (name, j, k, e, sp)
        r64 = ref.get(k)
        if r64 is not None and bool(r64.abs().max() > 0):     # and the repeat is still the oracle's gradient
            bound = tol.gin if k.startswith("input.") else tol.for_param(k[5:])
            assert rel_err(runs[-1][i], r64) <= bound, (name, k)


def test_backward_follows_the_forward_setting():
    """The attribute flipped between forward and backward: the backward runs in the forward's mode (a mismatch would read
    a workspace of the other layout)."""
    cfg, params, inp, rf, ref = case("L5")
    with precision("fp32") as tol:
        for first in (True, False):
            m = build(cfg, params, rf, first)
            t = {k: v.to(DEV) for k, v in inp.items()}
            x, Z = m(node_feat=t["node_feat"], node_loc=t["node_loc"], node_vel=t["node_vel"], edge_index=t["edge_index"],
                     data_batch=t["data_batch"], loc_mean=t["loc_mean"], edge_attr=t["edge_attr"])
            m.recompute = not first
            ((x * t["wx"]).sum() + (Z * t["wz"]).sum()).backward()
            torch.cuda.synchronize()
            for k, p in m.named_parameters():
                r = ref["grad." + k]
                if r is not None and bool(r.abs().max() > 0):
                    assert rel_err(p.grad.cpu(), r) <= tol.for_param(k), (first, k)


def test_graph_captured_training_step_matches_eager():
    """forward, mse_mmd_loss, backward and FusedAdam with recompute, captured as one CUDA graph: a replay from the same
    state gives the eager step's loss, gradients and updated parameters."""
    from fastegnn_b200 import FusedAdam, mse_mmd_loss
    cfg, params, inp, rf, _ = case("L5")
    t = {k: v.to(DEV) for k, v in inp.items()}
    gen = torch.Generator().manual_seed(5)
    target = t["node_loc"] + 0.1 * torch.randn(inp["node_loc"].shape, generator=gen).to(DEV)
    counts = torch.bincount(inp["data_batch"]).tolist()
    offs = [0]
    for c in counts[:-1]:
        offs.append(offs[-1] + c)
    idx = torch.stack([torch.randperm(n, generator=gen)[:16] + o for n, o in zip(counts, offs)]).to(torch.int32).to(DEV)
    with precision("tf32"):
        m = build(cfg, params, rf, True)
        opt = FusedAdam(m.parameters(), lr=1e-3)

        def train_step():
            opt.zero_grad(set_to_none=False)
            x, Z = m(node_feat=t["node_feat"], node_loc=t["node_loc"], node_vel=t["node_vel"], edge_index=t["edge_index"],
                     data_batch=t["data_batch"], loc_mean=t["loc_mean"], edge_attr=t["edge_attr"])
            total, _ = mse_mmd_loss(x, target, Z, idx, 1.5, 0.01)
            total.backward()
            opt.step()
            return total

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                train_step()
        torch.cuda.current_stream().wait_stream(side)
        state = [p.detach().clone() for p in m.parameters()]
        opt_state = {p: {k: v.clone() for k, v in st.items()} for p, st in opt.state.items()}

        def restore():
            with torch.no_grad():
                for p, s in zip(m.parameters(), state):
                    p.copy_(s)
                for p, st in opt_state.items():
                    for k, v in st.items():
                        opt.state[p][k].copy_(v)

        loss_e = train_step().detach().clone()
        grads_e = [None if p.grad is None else p.grad.detach().clone() for p in m.parameters()]
        params_e = [p.detach().clone() for p in m.parameters()]
        restore()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loss_g = train_step()
        restore()
        graph.replay()
        torch.cuda.synchronize()
        assert rel_err(loss_g.cpu(), loss_e.cpu()) <= RUN_TO_RUN
        for (n, p), ge, pe in zip(m.named_parameters(), grads_e, params_e):
            if ge is not None and bool(ge.abs().max() > 0):
                assert rel_err(p.grad.cpu(), ge.cpu()) <= RUN_TO_RUN, n
            assert rel_err(p.detach().cpu(), pe.cpu()) <= 1e-5, n      # one Adam step of lr 1e-3 from the same state


def test_peak_memory_falls_by_three_blocks():
    """Batch shape, L = 5: the default step holds five saved blocks, recompute two."""
    import ctypes as C
    from fastegnn_b200 import _lib
    from fastegnn_b200.ops import make_dims
    cfg, params, inp = make_graph_case(22, [400 + 13 * i for i in range(20)], 14, 3, L=5)
    N, B = inp["node_loc"].size(0), 20
    dims = make_dims(N, N, inp["edge_index"].size(1), B, 3, 2, 0, None)
    block_bytes = 4 * _lib.lib.fegnn_layer_saved_floats(C.byref(dims))
    peak = {}
    with precision("tf32"):
        for rc in (False, True, False, True):
            m = build(cfg, params, False, rc)
            step(m, inp, False)                     # warm: the CSR graph cache, allocator blocks
            del m
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            m = build(cfg, params, False, rc)
            step(m, inp, False)
            peak[rc] = torch.cuda.max_memory_allocated() - base
            del m
    saved = peak[False] - peak[True]
    print(f"RECOMPUTE_PEAK default {peak[False] / 2**20:.1f} MiB recompute {peak[True] / 2**20:.1f} MiB "
          f"block {block_bytes / 2**20:.1f} MiB")
    assert saved >= 0.95 * 3 * block_bytes, (saved, block_bytes)
