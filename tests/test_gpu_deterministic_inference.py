"""The forward-only stack under torch.use_deterministic_algorithms(True): FastEGNN / FastRF in eval() or under
torch.no_grad() give the same bits on every run -- eager, CUDA-graph replay, next to other work on another stream, and over
an autoregressive rollout whose graph is rebuilt from each prediction -- and agree with the default kernels to fp32
summation order and with the oracle on the golden-style seeded cases."""
import functools

import pytest
import torch

from fastegnn_b200 import CsrGraph, FastEGNN, FastRF, _lib
from tests.gpu_util import build_gpu_model, make_graph_case, precision, update_err
from tests.helpers import oracle_run

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")

# name -> (make_graph_case arguments, model options).  One Water-3D-sized cloud, a batch of 20 clouds, one graph of 100 000
# nodes with C = 8 (above the ring's 65 536 nodes: the single-block driver), hub rows whose edges span several edge tiles,
# and the layer options.
CASES = {
    "water3d": (dict(seed=1, sizes=[8000], deg=24, C=3), {}),
    "b20": (dict(seed=2, sizes=[400 + 13 * i for i in range(20)], deg=16, C=3), {}),
    "single_block_c8": (dict(seed=3, sizes=[100_000], deg=8, C=8), {}),
    "hubs": (dict(seed=4, sizes=[3000, 2000], deg=6, C=3, heavy_row=700), {}),
    "attention": (dict(seed=5, sizes=[3000, 2500], deg=12, C=3, attention=True), {}),
    "gravity": (dict(seed=6, sizes=[3000, 2500], deg=12, C=3, gravity=[0.0, 0.0, -9.8]), {}),
    "normalize_tanh": (dict(seed=7, sizes=[3000, 2500], deg=12, C=3, normalize=True, tanh=True), {}),
    "no_edge_attr": (dict(seed=8, sizes=[3000, 2500], deg=12, C=3, Fe=0), {}),
    "node_attr": (dict(seed=9, sizes=[3000, 2500], deg=12, C=3), dict(node_attr_nf=2)),
    "fastrf": (dict(seed=10, sizes=[3000, 2500], deg=12, C=3), dict(cls=FastRF)),
}
PRECISIONS = ["fp32", "tf32", "tf32x3", "tf32_all"]


@pytest.fixture
def det():
    on, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    _lib.set_mode("deterministic", 0)


def _setup(name):
    kw, opts = CASES[name]
    cfg, params, inp = make_graph_case(**kw)
    cls, na = opts.get("cls", FastEGNN), opts.get("node_attr_nf", 0)
    if cls is FastEGNN and na == 0:
        model = build_gpu_model(cfg, params, DEV)
    else:
        torch.manual_seed(kw["seed"])
        model = cls(node_feat_nf=cfg.node_feat_nf, node_attr_nf=na, edge_attr_nf=cfg.edge_attr_nf, hidden_nf=64,
                    virtual_channels=cfg.virtual_channels, device=DEV, n_layers=cfg.n_layers, attention=cfg.attention,
                    normalize=cfg.normalize, tanh=cfg.tanh, gravity=cfg.gravity)
    model.eval()
    g = {k: (None if v is None else v.to(DEV)) for k, v in inp.items()}
    if na:
        g["node_attr"] = torch.randn(g["node_loc"].size(0), na, generator=torch.Generator().manual_seed(11)).to(DEV)
    return cfg, params, inp, model, g


def _call(model, g, edge_index=None):
    kw = dict(node_feat=g["node_feat"], node_loc=g["node_loc"], node_vel=g["node_vel"],
              edge_index=g["edge_index"] if edge_index is None else edge_index, data_batch=g["data_batch"],
              loc_mean=g["loc_mean"], edge_attr=g["edge_attr"] if edge_index is None and g["edge_attr"].size(1) else None)
    if "node_attr" in g:
        kw["node_attr"] = g["node_attr"]
    with torch.no_grad():
        x, Z = model(**kw)
    torch.cuda.synchronize()
    return [x.clone(), Z.clone()]


def _matmul_load():
    s = torch.cuda.Stream()
    a = torch.randn(4096, 4096, device=DEV)
    with torch.cuda.stream(s):
        for _ in range(20):
            a = (a @ a).clamp_(-1, 1)
    return s


def _assert_same_bits(runs, label):
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert torch.equal(a, b), label


def _graph_replays(model, g, n=3):
    """CUDA-graph capture of the forward on a prebuilt CsrGraph; the eager run on the same graph, then n replays."""
    B = g["loc_mean"].size(0)
    graph = CsrGraph(g["edge_index"], g["data_batch"], g["edge_attr"] if g["edge_attr"].size(1) else None, B)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = _call(model, g, graph)
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg, stream=s), torch.no_grad():
            kw = dict(node_feat=g["node_feat"], node_loc=g["node_loc"], node_vel=g["node_vel"], edge_index=graph,
                      data_batch=g["data_batch"], loc_mean=g["loc_mean"])
            if "node_attr" in g:
                kw["node_attr"] = g["node_attr"]
            static = model(**kw)
    torch.cuda.current_stream().wait_stream(s)
    replays = []
    for _ in range(n):
        cg.replay()
        torch.cuda.synchronize()
        replays.append([t.clone() for t in static])
    return eager, replays


def _det_vs_default(model, g, tol, label):
    got = _call(model, g)
    torch.use_deterministic_algorithms(False)
    ref = _call(model, g)
    torch.use_deterministic_algorithms(True)
    for a, b, base in zip(got, ref, (g["node_loc"], g["loc_mean"])):
        assert update_err(a.cpu(), b.cpu(), base.cpu()) <= tol, label


@pytest.mark.parametrize("name", list(CASES))
def test_inference_repeats_bitwise(det, name):
    _, _, _, model, g = _setup(name)
    runs = [_call(model, g) for _ in range(3)]
    busy = _matmul_load()
    runs.append(_call(model, g))
    torch.cuda.synchronize()
    del busy
    _assert_same_bits(runs, name)
    assert _lib.get_mode("deterministic") == 1
    eager, replays = _graph_replays(model, g)
    _assert_same_bits([eager] + replays + runs[:1], name + " graph replay")
    with precision("tf32") as tol:
        _det_vs_default(model, g, tol.out, name)


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("name", ["water3d", "hubs", "attention"])
def test_inference_repeats_bitwise_in_every_precision(det, name, prec):
    _, _, _, model, g = _setup(name)
    with precision(prec) as tol:
        runs = [_call(model, g) for _ in range(3)]
        busy = _matmul_load()
        runs.append(_call(model, g))
        torch.cuda.synchronize()
        del busy
        _assert_same_bits(runs, f"{name} [{prec}]")
        _det_vs_default(model, g, tol.out, f"{name} [{prec}]")


@functools.lru_cache(maxsize=None)
def _oracle64(name):
    cfg, params, inp = make_graph_case(**CASES[name][0])
    return oracle_run(cfg, {k: v.double() for k, v in params.items()},
                      {k: (v.double() if v is not None and v.is_floating_point() else v) for k, v in inp.items()})


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("name", ["b20", "gravity", "attention", "normalize_tanh", "no_edge_attr"])
def test_deterministic_inference_against_oracle(det, name, prec):
    cfg, params, inp, model, g = _setup(name)
    with precision(prec) as tol:
        x, Z = _call(model, g)
    r64 = _oracle64(name)
    assert update_err(x.cpu(), r64["x"], inp["node_loc"]) <= tol.out, (name, prec, "x")
    assert update_err(Z.cpu(), r64["Z"], inp["loc_mean"]) <= tol.out, (name, prec, "Z")


def test_rollout_repeats_bitwise(det):
    """30 autoregressive steps: x, v from the prediction, the radius graph rebuilt from x every step."""
    gen = torch.Generator().manual_seed(21)
    N, B, r = 4000, 2, 0.12
    x0 = torch.rand(N, 3, generator=gen).to(DEV)
    v0 = (0.01 * torch.randn(N, 3, generator=gen)).to(DEV)
    batch = torch.cat([torch.zeros(N // 2, dtype=torch.long), torch.ones(N - N // 2, dtype=torch.long)]).to(DEV)
    feat = torch.ones(N, 1, device=DEV)
    torch.manual_seed(22)
    model = FastEGNN(node_feat_nf=1, node_attr_nf=0, edge_attr_nf=2, hidden_nf=64, virtual_channels=3, device=DEV,
                     n_layers=4).eval()

    def rollout():
        x, v, traj = x0.clone(), v0.clone(), []
        for _ in range(30):
            graph = CsrGraph.from_radius(x, batch, B, r)
            loc_mean = torch.stack([x[batch == b].mean(0) for b in range(B)]).unsqueeze(-1).repeat(1, 1, 3)
            with torch.no_grad():
                xn, _ = model(feat, x, v, graph, batch, loc_mean)
            v, x = xn - x, xn
            traj.append(x.clone())
        torch.cuda.synchronize()
        return traj

    a, b = rollout(), rollout()
    _assert_same_bits([a, b], "rollout")
    assert torch.isfinite(a[-1]).all()
