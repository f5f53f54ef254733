"""CPU checks behind tests/test_gpu_tile_shapes.py: the tile-boundary fixtures are what they claim, oracle/staged.py
equals the oracle's fp64 autograd on the odd layouts, and the test-only "grid_sms" mode is host code that accepts and
refuses what fegnn.h says."""
import pytest
import torch

from oracle import staged
from tests.helpers import oracle_run
from tests.tile_cases import TILE_CASES, TM, row_starts, tile_case, tile_rows_marks, tiles_per_cta


def _sizes(name):
    cfg, _, inp = tile_case(name)
    return cfg, inp, inp["data_batch"].numel(), inp["edge_index"].size(1)


@pytest.mark.parametrize("name,n_mod,e_mod,nc_ragged", [("ragged_1", 1, 1, True), ("ragged_127", 127, 127, True),
                                                        ("aligned", 0, 0, False)])
def test_ragged_and_aligned_sizes(name, n_mod, e_mod, nc_ragged):
    cfg, inp, N, E = _sizes(name)
    assert N % TM == n_mod and E % TM == e_mod
    assert ((N * cfg.virtual_channels) % TM != 0) == nc_ragged
    assert inp["edge_attr"].shape == (E, cfg.edge_attr_nf)


def test_tile_rows_layout():
    cfg, inp, N, E = _sizes("tile_rows")
    rp = row_starts(inp["edge_index"], N)
    assert int(rp[-1]) == E
    deg = rp[1:] - rp[:-1]
    starts = {int(s): int(d) for s, d in zip(rp[:-1], deg) if d > 0}
    marks = tile_rows_marks()
    for start, length, label in marks:
        assert starts.get(start) == length, label
    assert sorted({s % TM for s, _, _ in marks if "start@" in _}) == [0, 1, 31, 32, 33, 126, 127]
    for length in (TM, TM + 1, 3 * TM + 1):
        assert any(s % TM == 0 and n == length for s, n in starts.items()), length
    # runs of isolated rows between the marked rows, and rows that belong to one graph
    assert int((deg == 0).sum()) >= 20
    b = inp["data_batch"]
    assert bool((b[inp["edge_index"][0]] == b[inp["edge_index"][1]]).all())


def test_small_fixtures():
    _, inp, N, E = _sizes("one_node")
    assert (N, E, inp["loc_mean"].size(0)) == (1, 1, 1) and inp["edge_index"].tolist() == [[0], [0]]
    _, inp, N, E = _sizes("no_edges")
    assert E == 0 and N > TM
    cfg, inp, N, _ = _sizes("many_graphs")
    b = inp["data_batch"]
    B = inp["loc_mean"].size(0)
    assert B >= 390 and int(torch.bincount(b).max()) <= 3
    # a graph boundary inside every node tile and every (node, channel) tile
    bounds = set(torch.nonzero(b[1:] != b[:-1]).flatten().add(1).tolist())
    for t0 in range(0, N, TM):
        assert any(t0 < x < t0 + TM for x in bounds)
    tn = TM // cfg.virtual_channels
    for t0 in range(0, N, tn):
        assert any(t0 < x < min(t0 + tn, N) for x in bounds) or min(t0 + tn, N) - t0 < 4


def test_grid_cap_gives_several_tiles_per_cta():
    """At a cap of 2 SMs every persistent kernel runs at least 3 tiles (tile pairs for the edge backward) per CTA on the
    fixtures of more than one tile, from the launch rules of the kernels."""
    for name in ("ragged_1", "ragged_127", "aligned", "tile_rows", "many_graphs"):
        cfg, inp, N, E = _sizes(name)
        per = tiles_per_cta(N, E, cfg.virtual_channels, 2)
        assert min(per.values()) >= 3, (name, per)


@pytest.mark.parametrize("name", ["tile_rows", "one_node", "many_graphs", "no_edges"])
def test_staged_equals_oracle_autograd_on_tile_fixtures(name):
    """As tests/test_staged_spec.py: the staged pipeline the GPU phases are checked against equals the oracle's fp64
    autograd on the CSR-built layout, one node, 1-3 node graphs and an empty edge list."""
    cfg, params, inp = tile_case(name)
    params = {k: v.double() for k, v in params.items()}
    inp = {k: (v.double() if v.is_floating_point() else v) for k, v in inp.items()}
    ref = oracle_run(cfg, params, inp)
    fl = staged.Flags(cfg.attention, cfg.normalize, cfg.tanh, cfg.gravity, cfg.eps)
    sm = staged.StagedModel(params, cfg.hidden_nf, cfg.virtual_channels, cfg.edge_attr_nf, cfg.n_layers, fl)
    x, Z = sm.forward(inp["node_feat"], inp["node_loc"], inp["node_vel"], inp["edge_index"], inp["data_batch"],
                      inp["loc_mean"], inp["edge_attr"])
    assert torch.allclose(x, ref["x"], rtol=1e-10, atol=1e-11)
    assert torch.allclose(Z, ref["Z"], rtol=1e-10, atol=1e-11)
    grads, gin = sm.backward(inp["wx"], inp["wz"])
    for k in ("node_loc", "loc_mean", "node_feat"):
        s = ref["gin"][k].abs().max()
        assert torch.allclose(gin[k], ref["gin"][k], rtol=1e-8, atol=1e-10 * float(s)), k
    for k, g in ref["gp"].items():
        if g is None:
            assert k not in grads, k
            continue
        s = float(g.abs().max()) + 1e-30
        assert torch.allclose(grads[k], g, rtol=1e-7, atol=1e-9 * s), (k, float((grads[k] - g).abs().max()), s)


def test_grid_sms_mode():
    """Host code: the library loads without a GPU and set / get of a mode launch nothing."""
    from fastegnn_b200 import _lib as L
    old = L.get_mode("grid_sms")
    assert old == 0 and "grid_sms" not in L.PHASES
    try:
        for v in (0, 2, 3, 148, 1000):
            L.set_mode("grid_sms", v)
            assert L.get_mode("grid_sms") == v
        for v in (1, -1, -148):
            with pytest.raises(L.FegnnError, match="grid_sms"):
                L.set_mode("grid_sms", v)
            assert L.get_mode("grid_sms") == 1000
        L.set_precision("fp32")
        assert L.get_mode("grid_sms") == 1000
    finally:
        L.set_precision("tf32")
        L.set_mode("grid_sms", old)


def test_tile_cases_table_is_complete():
    assert set(TILE_CASES) == {"ragged_1", "ragged_127", "aligned", "tile_rows", "one_node", "many_graphs", "no_edges"}
