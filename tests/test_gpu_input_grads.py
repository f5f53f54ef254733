"""Gradients to node_vel, edge_attr and node_attr (fegnn_model_backward_inputs and the per-phase _inputs entries) on the
GPU, in every arithmetic mode, against the fp64 autograd of the oracle (oracle/fastegnn_oracle.py; tests/node_attr_spec.py
for the attribute term) and the golden vectors of the unmodified reference."""
import dataclasses

import pytest
import torch

from oracle import fastegnn_oracle as orc
from tests import node_attr_spec as spec
from tests.gpu_util import make_graph_case, precision, rel_err
from tests.helpers import H64_CASES, case_inputs, case_params, load_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PRECS = ["fp32", "tf32x3", "tf32", "tf32_all"]
# Relative to the largest entry of the fp64 gradient, per mode and input: about twice the worst value observed on an
# NVIDIA B200 (1000 W) over every case below (DESIGN.md 3.6).  node_loc: dL/dx0 through edge lengths and rollouts; params:
# the rollout's parameter gradients.  The tensor-core modes share the packed-fp16 edge backward, whose fp16 gz1 sets
# g_edge_attr (worst at Fe = 1).
TOL_IG = {
    "fp32":     dict(node_vel=2.5e-6, edge_attr=4e-6, node_attr=1e-6, node_loc=1e-6, params=2e-6),
    "tf32x3":   dict(node_vel=1e-3, edge_attr=2e-2, node_attr=5e-3, node_loc=1e-3, params=5e-3),
    "tf32":     dict(node_vel=1.2e-3, edge_attr=1.3e-2, node_attr=6e-3, node_loc=1.5e-3, params=5e-3),
    "tf32_all": dict(node_vel=5e-3, edge_attr=1.2e-2, node_attr=4e-3, node_loc=1.4e-3, params=6e-3),
}
# a second run of the same step: the layer kernels add floats across CTAs in arrival order (DESIGN.md 3.2)
RUN_TO_RUN = {"fp32": 1e-5, "tf32x3": 1e-3, "tf32": 1e-3, "tf32_all": 1e-3}
INPUTS = ("node_loc", "node_vel", "loc_mean", "node_feat", "edge_attr", "node_attr")


def check(tag, prec, key, err):
    """err (relative to the largest entry of the fp64 gradient) within the bound of this mode and input."""
    print(f"INPUT_GRAD_ERR {tag} {prec} {key} {err:.3e}")
    assert err <= TOL_IG[prec][key], (tag, prec, key, err)


def build(cfg, params, rf=False):
    from fastegnn_b200 import FastEGNN, FastRF
    cls = FastRF if rf else FastEGNN
    m = cls(node_feat_nf=cfg.node_feat_nf, node_attr_nf=cfg.node_attr_nf, edge_attr_nf=cfg.edge_attr_nf, hidden_nf=64,
            virtual_channels=cfg.virtual_channels, device=DEV, n_layers=cfg.n_layers, attention=cfg.attention,
            normalize=cfg.normalize, tanh=cfg.tanh, gravity=cfg.gravity)
    m.load_state_dict({k: v.to(DEV) for k, v in params.items()})
    return m


def oracle(cfg, params, inp, dtype=torch.float64):
    """fp64 autograd of sum(x * wx) + sum(Z * wz) with respect to every float input and parameter."""
    p = {k: v.to(dtype).requires_grad_(True) for k, v in params.items()}
    leaf = {k: inp[k].to(dtype).requires_grad_(True) for k in INPUTS if inp.get(k) is not None}
    args = (leaf["node_feat"], leaf["node_loc"], leaf["node_vel"], inp["edge_index"], inp["data_batch"], leaf["loc_mean"],
            leaf["edge_attr"])
    x, Z = (spec.oracle_forward(p, cfg, *args, leaf["node_attr"]) if "node_attr" in leaf else
            orc.fastegnn_forward(p, cfg, *args))
    ((x * inp["wx"].to(dtype)).sum() + (Z * inp["wz"].to(dtype)).sum()).backward()
    return {k: t.grad for k, t in leaf.items()}, {k: t.grad for k, t in p.items()}


def gpu(m, inp, want=("node_vel", "edge_attr", "node_attr")):
    t = {k: (None if v is None else v.to(DEV)) for k, v in inp.items()}
    leaf = {k: t[k].clone().requires_grad_(k in want or k in ("node_loc", "loc_mean", "node_feat"))
            for k in INPUTS if t.get(k) is not None}
    x, Z = m(node_feat=leaf["node_feat"], node_loc=leaf["node_loc"], node_vel=leaf["node_vel"], edge_index=t["edge_index"],
             data_batch=t["data_batch"], loc_mean=leaf["loc_mean"], edge_attr=leaf.get("edge_attr"),
             node_attr=leaf.get("node_attr"))
    ((x * t["wx"]).sum() + (Z * t["wz"]).sum()).backward()
    torch.cuda.synchronize()
    gin = {k: (None if v.grad is None else v.grad.cpu()) for k, v in leaf.items()}
    return gin, {k: (None if p.grad is None else p.grad.cpu()) for k, p in m.named_parameters()}


def spread_columns(inp, seed):
    """make_graph_case repeats the edge length in every column: scale each column differently so they are told apart."""
    g = torch.Generator().manual_seed(seed)
    ea = inp["edge_attr"]
    return dict(inp, edge_attr=ea * (0.5 + torch.rand(1, ea.size(1), generator=g)) + 0.1 * torch.randn(ea.shape, generator=g))


# ----------------------------------------------------------------------------- node_vel on the golden cases
# (h16_full_grads has hidden_nf = 16, which the kernels do not take; its node_vel gradient is checked on the CPU)
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("case", H64_CASES)
def test_node_vel_gradient_on_golden_cases(case, prec):
    meta, arr = load_case(case)
    cfg, params = case_params(meta["case"])
    inp = case_inputs(arr)
    ref, _ = oracle(cfg, params, inp)
    golden = torch.from_numpy(arr["gin_node_vel"]).double()
    with precision(prec):
        gin, _ = gpu(build(cfg, params), inp, want=("node_vel",))
    tol = TOL_IG[prec]["node_vel"]
    check(case, prec, "node_vel", rel_err(gin["node_vel"], ref["node_vel"]))
    golden_dist = rel_err(golden, ref["node_vel"])
    assert rel_err(gin["node_vel"], golden) <= tol + 1.1 * golden_dist


# ----------------------------------------------------------------------------- edge_attr
EDGE_VARIANTS = {
    "Fe1": dict(Fe=1), "Fe2": dict(Fe=2), "Fe4": dict(Fe=4),                  # packed-fp16 kernel (mode 7)
    "Fe8": dict(Fe=8), "attention": dict(Fe=2, attention=True),             # fp32 kernel
    "normalize_selfloops": dict(Fe=2, normalize=True),
}


def edge_case(variant, seed=21):
    kw = dict(EDGE_VARIANTS[variant])
    cfg, params, inp = make_graph_case(seed, [70, 45, 90], 7, 3, Fe=kw.pop("Fe"), L=3, **kw)
    inp = spread_columns(inp, seed)
    if variant == "normalize_selfloops":              # self-loops: q = 0, 1 / (|d| + eps) large; their gradient is still exact
        ei = inp["edge_index"]
        loops = torch.arange(0, 200, 7)
        inp["edge_index"] = torch.cat([ei, torch.stack([loops, loops])], dim=1)
        inp["edge_attr"] = torch.cat([inp["edge_attr"], torch.rand(loops.numel(), inp["edge_attr"].size(1))])
    return cfg, params, inp


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("variant", list(EDGE_VARIANTS))
def test_edge_attr_gradient_against_oracle(variant, prec):
    cfg, params, inp = edge_case(variant)
    assert not bool((inp["edge_index"][0][1:] >= inp["edge_index"][0][:-1]).all())      # unsorted: perm is exercised
    ref, refp = oracle(cfg, params, inp)
    with precision(prec):
        gin, gp = gpu(build(cfg, params), inp)
    assert gin["edge_attr"].shape == inp["edge_attr"].shape
    check(variant, prec, "edge_attr", rel_err(gin["edge_attr"], ref["edge_attr"]))
    check(variant, prec, "node_vel", rel_err(gin["node_vel"], ref["node_vel"]))


# ----------------------------------------------------------------------------- node_attr
def attr_case(Fa, seed=31, L=3):
    cfg0, _, inp = make_graph_case(seed, [50, 37, 61], 6, 3, L=L)
    cfg = dataclasses.replace(cfg0, node_attr_nf=Fa)
    params = orc.make_params(cfg, seed + 1000)
    orc.rescale_coord_heads(params, 1000.0)
    g = torch.Generator().manual_seed(seed + 7)
    return cfg, params, dict(inp, node_attr=torch.randn(inp["node_loc"].size(0), Fa, generator=g))


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("Fa", [1, 5, 16])
def test_node_attr_gradient_against_spec(Fa, prec):
    cfg, params, inp = attr_case(Fa)
    ref, _ = oracle(cfg, params, inp)
    with precision(prec):
        gin, _ = gpu(build(cfg, params), inp)
    for k in ("node_attr", "edge_attr", "node_vel"):
        check(f"Fa{Fa}", prec, k, rel_err(gin[k], ref[k]))


@pytest.mark.parametrize("prec", ["fp32", "tf32"])
@pytest.mark.parametrize("graph", ["edge_index", "csr_graph", "from_radius"])
def test_embedding_table_trains_through_node_attr(graph, prec):
    """nn.Embedding(type) -> node_attr: the table's gradient matches the oracle's, with the edge list given per call, as a
    CsrGraph reused across calls, and as a CsrGraph.from_radius built on the device (its edge_attr is data)."""
    from fastegnn_b200 import CsrGraph
    cfg, params, inp = attr_case(4)
    N, B = inp["node_loc"].size(0), inp["loc_mean"].size(0)
    types = torch.randint(0, 6, (N,), generator=torch.Generator().manual_seed(3))
    table = torch.randn(6, 4, generator=torch.Generator().manual_seed(4))
    t = {k: v.to(DEV) for k, v in inp.items()}
    g = t["edge_index"]
    if graph == "csr_graph":
        g = CsrGraph(t["edge_index"], t["data_batch"], t["edge_attr"], B)
        g.wait()
    elif graph == "from_radius":
        g = CsrGraph.from_radius(t["node_loc"], t["data_batch"], B, r=1.5, edge_attr_nf=cfg.edge_attr_nf)
        inp = dict(inp, edge_index=g.edge_index().cpu(), edge_attr=g.edge_attr.cpu())
        assert g.E > 100
    emb64 = torch.nn.Embedding.from_pretrained(table.double(), freeze=False)
    p64 = {k: v.double() for k, v in params.items()}
    d = lambda k: inp[k].double()
    x, Z = spec.oracle_forward(p64, cfg, d("node_feat"), d("node_loc"), d("node_vel"), inp["edge_index"], inp["data_batch"],
                               d("loc_mean"), d("edge_attr"), emb64(types))
    ((x * d("wx")).sum() + (Z * d("wz")).sum()).backward()
    with precision(prec):
        m = build(cfg, params)
        emb = torch.nn.Embedding.from_pretrained(table.to(DEV), freeze=False)
        for _ in range(2 if graph == "csr_graph" else 1):          # the reused graph serves two steps
            emb.weight.grad = None
            x, Z = m(node_feat=t["node_feat"], node_loc=t["node_loc"], node_vel=t["node_vel"], edge_index=g,
                     data_batch=t["data_batch"], loc_mean=t["loc_mean"],
                     edge_attr=t["edge_attr"] if graph == "edge_index" else None, node_attr=emb(types.to(DEV)))
            ((x * t["wx"]).sum() + (Z * t["wz"]).sum()).backward()
        torch.cuda.synchronize()
    check(f"embedding_{graph}", prec, "node_attr", rel_err(emb.weight.grad.cpu(), emb64.weight.grad))


# ----------------------------------------------------------------------------- compositions that fail without the gradients
def lengths(x, ei, Fe):
    return (x[ei[0]] - x[ei[1]]).norm(dim=1, keepdim=True).repeat(1, Fe)


@pytest.mark.parametrize("prec", PRECS)
def test_edge_lengths_from_node_loc_reach_node_loc_grad(prec):
    cfg, params, inp = make_graph_case(41, [60, 80], 8, 3, Fe=2, L=3)
    ei = inp["edge_index"]
    p64 = {k: v.double() for k, v in params.items()}
    x64 = inp["node_loc"].double().requires_grad_(True)
    d = lambda k: inp[k].double()
    xo, Zo = orc.fastegnn_forward(p64, cfg, d("node_feat"), x64, d("node_vel"), ei, inp["data_batch"], d("loc_mean"),
                                  lengths(x64, ei, 2))
    ((xo * d("wx")).sum() + (Zo * d("wz")).sum()).backward()
    with precision(prec):
        m = build(cfg, params)
        t = {k: v.to(DEV) for k, v in inp.items()}
        x = t["node_loc"].clone().requires_grad_(True)
        xg, Zg = m(node_feat=t["node_feat"], node_loc=x, node_vel=t["node_vel"], edge_index=t["edge_index"],
                   data_batch=t["data_batch"], loc_mean=t["loc_mean"], edge_attr=lengths(x, t["edge_index"], 2))
        ((xg * t["wx"]).sum() + (Zg * t["wz"]).sum()).backward()
        torch.cuda.synchronize()
    check("composition", prec, "node_loc", rel_err(x.grad.cpu(), x64.grad))


@pytest.mark.parametrize("prec", PRECS)
def test_two_step_unrolled_rollout(prec):
    """x1 = model(x0, v0); v1 = (x1 - x0) / dt; edge lengths recomputed from x1; loss on x2."""
    cfg, params, inp = make_graph_case(43, [60, 80], 8, 3, Fe=1, L=2)
    ei, dt = inp["edge_index"], 0.5

    def rollout(model_fn, x0, v0, to):
        x1, Z1 = model_fn(x0, v0, lengths(x0, to(ei), 1), to(inp["loc_mean"]))
        x2, Z2 = model_fn(x1, (x1 - x0) / dt, lengths(x1, to(ei), 1), Z1)
        return (x2 * to(inp["wx"])).sum() + (Z2 * to(inp["wz"])).sum()

    p64 = {k: v.double().requires_grad_(True) for k, v in params.items()}
    x64 = inp["node_loc"].double().requires_grad_(True)
    f64 = lambda x, v, ea, lm: orc.fastegnn_forward(p64, cfg, inp["node_feat"].double(), x, v, ei, inp["data_batch"], lm, ea)
    rollout(f64, x64, inp["node_vel"].double(), lambda t: t.double() if t.is_floating_point() else t).backward()
    with precision(prec):
        m = build(cfg, params)
        x0 = inp["node_loc"].to(DEV).requires_grad_(True)
        fg = lambda x, v, ea, lm: m(node_feat=inp["node_feat"].to(DEV), node_loc=x, node_vel=v, edge_index=ei.to(DEV),
                                    data_batch=inp["data_batch"].to(DEV), loc_mean=lm, edge_attr=ea)
        rollout(fg, x0, inp["node_vel"].to(DEV), lambda t: t.to(DEV)).backward()
        torch.cuda.synchronize()
    check("rollout", prec, "node_loc", rel_err(x0.grad.cpu(), x64.grad))
    worst = 0.0
    for k, p in m.named_parameters():
        if p64[k].grad is not None and float(p64[k].grad.abs().max()) > 0:
            worst = max(worst, rel_err(p.grad.cpu(), p64[k].grad))
    check("rollout", prec, "params", worst)


# ----------------------------------------------------------------------------- layer level
@pytest.mark.parametrize("prec", PRECS)
def test_layer_level_input_gradients(prec):
    cfg, params, inp = attr_case(5, L=1)
    inp = spread_columns(inp, 5)
    N, B = inp["node_loc"].size(0), 3
    g = torch.Generator().manual_seed(9)
    h, S = torch.randn(N, 64, generator=g), torch.randn(B, 64, 3, generator=g)
    w = [torch.randn(N, 64, generator=g), torch.randn(N, 3, generator=g), torch.randn(B, 64, 3, generator=g),
         torch.randn(B, 3, 3, generator=g)]
    p64 = {k: v.double() for k, v in params.items()}
    leaf = {k: inp[k].double().requires_grad_(True) for k in ("node_vel", "edge_attr", "node_attr")}
    out = spec.layer_forward(p64, "gcl_0", cfg, h.double(), inp["edge_index"], inp["node_loc"].double(), leaf["node_vel"],
                             inp["loc_mean"].double(), S.double(), inp["data_batch"], leaf["edge_attr"], leaf["node_attr"])
    sum((o * wi.double()).sum() for o, wi in zip(out, w)).backward()
    with precision(prec):
        m = build(cfg, params)
        t = {k: v.to(DEV) for k, v in inp.items()}
        lg = {k: t[k].clone().requires_grad_(True) for k in leaf}
        out = m.gcl_0(h.to(DEV), t["edge_index"], t["node_loc"], lg["node_vel"], t["loc_mean"], S.to(DEV), t["data_batch"],
                      edge_attr=lg["edge_attr"], node_attr=lg["node_attr"])
        sum((o * wi.to(DEV)).sum() for o, wi in zip(out, w)).backward()
        torch.cuda.synchronize()
    for k in leaf:
        check("layer", prec, k, rel_err(lg[k].grad.cpu(), leaf[k].grad))


# ----------------------------------------------------------------------------- not requested / FastRF
@pytest.mark.parametrize("prec", PRECS)
def test_parameter_gradients_do_not_depend_on_the_request(prec):
    cfg, params, inp = attr_case(3)
    with precision(prec):
        m = build(cfg, params)
        gin0, gp0 = gpu(m, inp, want=())
        m.zero_grad(set_to_none=True)
        gin1, gp1 = gpu(m, inp)
    assert gin0["node_vel"] is None and gin0["edge_attr"] is None and gin0["node_attr"] is None
    assert gin1["node_vel"] is not None and gin1["edge_attr"] is not None and gin1["node_attr"] is not None
    for k in gp0:
        if gp0[k] is not None:
            assert rel_err(gp1[k], gp0[k]) <= RUN_TO_RUN[prec], k


@pytest.mark.parametrize("prec", PRECS)
def test_fastrf_edge_attr_gradient_and_no_node_vel_gradient(prec):
    """FastRF shares the stack: edge_attr gets its gradient (against the FastRF oracle); node_vel, which enters FastRF
    through |v|, gets none."""
    from oracle import fastrf_oracle as rfo
    cfg, _, inp = make_graph_case(51, [40, 30], 5, 2, Fe=2, L=2)
    inp = spread_columns(inp, 51)
    params = rfo.make_params(cfg, 1051)
    orc.rescale_coord_heads(params, 1000.0)
    p64 = {k: v.double() for k, v in params.items()}
    d = lambda k: inp[k].double()
    ea64 = d("edge_attr").requires_grad_(True)
    x, Z = rfo.fastrf_forward(p64, cfg, d("node_feat"), d("node_loc"), d("node_vel"), inp["edge_index"], inp["data_batch"],
                              d("loc_mean"), ea64)
    ((x * d("wx")).sum() + (Z * d("wz")).sum()).backward()
    with precision(prec):
        m = build(cfg, params, rf=True)
        t = {k: v.to(DEV) for k, v in inp.items()}
        v, ea = t["node_vel"].clone().requires_grad_(True), t["edge_attr"].clone().requires_grad_(True)
        x, Z = m(node_feat=t["node_feat"], node_loc=t["node_loc"], node_vel=v, edge_index=t["edge_index"],
                 data_batch=t["data_batch"], loc_mean=t["loc_mean"], edge_attr=ea)
        ((x * t["wx"]).sum() + (Z * t["wz"]).sum()).backward()
        torch.cuda.synchronize()
    assert v.grad is None
    check("fastrf", prec, "edge_attr", rel_err(ea.grad.cpu(), ea64.grad))


# ----------------------------------------------------------------------------- CUDA graph capture
def test_training_step_with_input_gradients_graph_replay_matches_eager():
    """One step (forward, backward into node_vel / edge_attr / node_attr, an SGD update of the embedding table) captured as
    a CUDA graph: replays equal the eager step within the run-to-run bound."""
    cfg, params, inp = attr_case(4)
    t = {k: v.to(DEV) for k, v in inp.items()}
    types = torch.randint(0, 5, (t["node_loc"].size(0),), device=DEV)
    with precision("tf32"):
        m = build(cfg, params)
        emb = torch.nn.Embedding(5, 4).to(DEV)
        v = t["node_vel"].clone().requires_grad_(True)
        ea = t["edge_attr"].clone().requires_grad_(True)

        def step():
            x, Z = m(node_feat=t["node_feat"], node_loc=t["node_loc"], node_vel=v, edge_index=t["edge_index"],
                     data_batch=t["data_batch"], loc_mean=t["loc_mean"], edge_attr=ea, node_attr=emb(types))
            loss = (x * t["wx"]).sum() + (Z * t["wz"]).sum()
            for p in (v, ea, emb.weight):
                p.grad = None
            loss.backward()
            return loss, v.grad, ea.grad, emb.weight.grad
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                step()
        torch.cuda.current_stream().wait_stream(side)
        eager = [o.detach().clone() for o in step()]
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = step()
        for _ in range(2):
            graph.replay()
            torch.cuda.synchronize()
            for a, b in zip(out, eager):
                assert rel_err(a.cpu(), b.cpu()) <= RUN_TO_RUN["tf32"]
