"""Deterministic mode on the GPU: under torch.use_deterministic_algorithms(True), mmd_loss, mse_mmd_loss and a FusedAdam
step give the same bits on every run (eager, CUDA-graph replay, next to other work on another stream), agree with the
default kernels and the torch composition to fp32 summation order, and the models without a deterministic form raise
(or warn and run under warn_only=True)."""
import warnings

import numpy as np
import pytest
import torch

from fastegnn_b200 import FastEGNN, FusedAdam, VNEGNN, _lib, mmd_loss, mse_mmd_loss
from tests.gpu_util import precision, rel_err

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
SIGMA, WEIGHT = 1.5, 0.01

# (graph sizes, virtual channels, samples per graph): one cloud as in Water-3D, a batch of 20 clouds, a C = 8 cloud of
# 60 000 nodes, and one graph of 1 M nodes (the forward's MSE term crosses many CTAs in the default kernels)
CASES = {"b1": ([8000], 3, 64), "b20": ([400 + 13 * i for i in range(20)], 3, 32), "c8": ([60000], 8, 128),
         "1m": ([1_000_000], 3, 64)}


@pytest.fixture
def det():
    on, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    _lib.set_mode("deterministic", 0)


def _inputs(name, seed=3):
    sizes, Cc, ns = CASES[name]
    gen = torch.Generator().manual_seed(seed)
    N, B = sum(sizes), len(sizes)
    x = (3 * torch.randn(N, 3, generator=gen)).to(DEV)
    tgt = (3 * torch.randn(N, 3, generator=gen)).to(DEV)
    Z = (3 * torch.randn(B, 3, Cc, generator=gen)).to(DEV)
    offs = np.concatenate([[0], np.cumsum(sizes)])[:-1]
    idx = torch.stack([torch.randperm(n, generator=gen)[:ns] + int(o) for n, o in zip(sizes, offs)]).to(torch.int32)
    return x, tgt, Z, idx.to(DEV)


def _train_step(x0, tgt, Z0, idx, busy=None):
    """One step from fresh copies of (x0, Z0): mse_mmd_loss, backward, FusedAdam.  Returns every tensor it produced."""
    x = torch.nn.Parameter(x0.clone())
    Z = torch.nn.Parameter(Z0.clone())
    opt = FusedAdam([x, Z], lr=1e-3, weight_decay=1e-2)
    if busy is not None:
        busy()
    total, mse = mse_mmd_loss(x, tgt, Z, idx, SIGMA, WEIGHT)
    total.backward()
    gx, gZ = x.grad.clone(), Z.grad.clone()
    opt.step()
    torch.cuda.synchronize()
    return [total.detach().clone(), mse.detach().clone(), gx, gZ, x.detach().clone(), Z.detach().clone()]


def _assert_same_bits(runs):
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert torch.equal(a, b)


def _matmul_load():
    """A queue of large matmuls on another stream, running while the step's kernels run."""
    s = torch.cuda.Stream()
    a = torch.randn(4096, 4096, device=DEV)
    with torch.cuda.stream(s):
        for _ in range(20):
            a = (a @ a).clamp_(-1, 1)
    return s


@pytest.mark.parametrize("name", list(CASES))
def test_training_step_repeats_bitwise(det, name):
    x0, tgt, Z0, idx = _inputs(name)
    runs = [_train_step(x0, tgt, Z0, idx) for _ in range(3)]
    streams = []
    runs.append(_train_step(x0, tgt, Z0, idx, busy=lambda: streams.append(_matmul_load())))
    torch.cuda.synchronize()
    _assert_same_bits(runs)
    assert _lib.get_mode("deterministic") == 1


@pytest.mark.parametrize("name", ["b1", "b20"])
def test_graph_replay_matches_eager_bitwise(det, name):
    x0, tgt, Z0, idx = _inputs(name)
    s = torch.cuda.Stream()         # leaves, eager run and capture on one side stream (autograd syncs to a leaf's stream)
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        x = x0.clone().requires_grad_(True)
        Z = Z0.clone().requires_grad_(True)

        def fwd_bwd():
            total, mse = mse_mmd_loss(x, tgt, Z, idx, SIGMA, WEIGHT)
            gx, gZ = torch.autograd.grad(total, [x, Z])
            return [total, mse, gx, gZ]

        eager = [t.clone() for t in fwd_bwd()]
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            static = fwd_bwd()
    torch.cuda.current_stream().wait_stream(s)
    replays = []
    for _ in range(3):
        g.replay()
        torch.cuda.synchronize()
        replays.append([t.clone() for t in static])
    _assert_same_bits([eager] + replays)


def _torch_mmd(x, Z, idx):
    """l_vv - l_rv of utils/train.py:111-165 with torch ops (per graph, Laplacian kernel on the L2 distance)."""
    B = Z.size(0)
    out = 0.0
    for b in range(B):
        z = Z[b].t()
        s = x[idx[b].long()]
        k = lambda p, q: torch.exp(-torch.cdist(p, q, compute_mode="donot_use_mm_for_euclid_dist") / (2 * SIGMA ** 2))
        out = out + k(z, z).mean() - 2 * k(s, z).mean()
    return out / B


@pytest.mark.parametrize("name", ["b1", "b20", "c8"])
def test_deterministic_losses_match_default_and_torch(det, name):
    x0, tgt, Z0, idx = _inputs(name)

    def run(fn):
        x = x0.clone().requires_grad_(True)
        Z = Z0.clone().requires_grad_(True)
        total, mse = fn(x, Z)
        (total + 0.25 * mse).backward()
        return [total.detach(), mse.detach(), x.grad, Z.grad]

    loss_ops = lambda x, Z: mse_mmd_loss(x, tgt, Z, idx, SIGMA, WEIGHT)
    mmd_ops = lambda x, Z: (mmd_loss(x, Z, idx, SIGMA), torch.zeros((), device=DEV))
    got = [run(loss_ops), run(mmd_ops)]
    torch.use_deterministic_algorithms(False)
    default = [run(loss_ops), run(mmd_ops)]
    composed = [run(lambda x, Z: (torch.nn.functional.mse_loss(x, tgt) + WEIGHT * _torch_mmd(x, Z, idx),
                                  torch.nn.functional.mse_loss(x, tgt))),
                run(lambda x, Z: (_torch_mmd(x, Z, idx), torch.zeros((), device=DEV)))]
    for g_, d_, c_ in zip(got, default, composed):
        for a, b, c in zip(g_, d_, c_):
            assert rel_err(a.cpu(), b.cpu()) <= 1e-5, name
            assert rel_err(a.cpu(), c.cpu()) <= 1e-4, name


def _small_graph():
    gen = torch.Generator().manual_seed(1)
    N = 64
    row = torch.arange(N).repeat_interleave(4)
    col = (row + torch.randint(1, N, (4 * N,), generator=gen)) % N
    return dict(node_feat=torch.randn(N, 1, generator=gen).to(DEV), node_loc=torch.randn(N, 3, generator=gen).to(DEV),
                node_vel=torch.randn(N, 3, generator=gen).to(DEV), edge_index=torch.stack([row, col]).to(DEV),
                data_batch=torch.zeros(N, dtype=torch.long, device=DEV), loc_mean=torch.zeros(1, 3, 3, device=DEV))


@pytest.mark.parametrize("attention,prec", [(False, "tf32"), (True, "tf32"), (False, "fp32")])
def test_models_without_a_deterministic_form_raise_or_warn(det, attention, prec):
    with precision(prec):
        _policy_case(attention)


def _policy_case(attention):
    torch.manual_seed(0)
    model = FastEGNN(node_feat_nf=1, node_attr_nf=0, edge_attr_nf=0, hidden_nf=64, virtual_channels=3, device=DEV,
                     n_layers=2, attention=attention)
    inp = _small_graph()
    with pytest.raises(RuntimeError, match="FastEGNN does not have a deterministic implementation"):
        model(**inp)
    vn = VNEGNN(node_feat_nf=1, node_attr_nf=0, edge_attr_nf=0, hidden_nf=64, virtual_channels=3, device=DEV, n_layers=1)
    with pytest.raises(RuntimeError, match="VNEGNN does not have a deterministic implementation"):
        vn(inp["node_feat"], inp["node_loc"], inp["edge_index"], inp["data_batch"], torch.randn(1, 3, 3, device=DEV))
    torch.use_deterministic_algorithms(True, warn_only=True)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        x, Z = model(**inp)
        ((x ** 2).sum() + Z.sum()).backward()
        torch.cuda.synchronize()
    msgs = [str(m.message) for m in w]
    assert any("FastEGNN does not have a deterministic implementation" in m for m in msgs), msgs
    assert any("FastEGNN backward does not have a deterministic implementation" in m for m in msgs), msgs
    assert torch.isfinite(x).all() and _lib.get_mode("deterministic") == 0
    torch.use_deterministic_algorithms(False)
    model(**inp)
    assert _lib.get_mode("deterministic") == 0
