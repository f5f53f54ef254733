"""Live edge counts (FEGNN_F_LIVE_EDGES) on the host: the ABI additions, and every refusal that has to happen before any
device work (so these run without a GPU)."""
import ctypes as C
import os
import re

import pytest
import torch

from fastegnn_b200 import CsrGraph, _lib
from fastegnn_b200.ops import make_dims

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 0x1000          # a non-NULL device address that nothing on the host dereferences


def test_flag_and_graph_layout():
    assert _lib.F_LIVE_EDGES == 8192
    assert _lib.Graph.n_edges.offset == 7 * C.sizeof(C.c_void_p)       # after ready_event
    assert C.sizeof(_lib.Graph) == 8 * C.sizeof(C.c_void_p)
    header = open(os.path.join(ROOT, "include", "fegnn.h")).read()
    assert re.search(r"#define FEGNN_F_LIVE_EDGES 8192u", header)
    for name, value in (("BAD_COUNT", 1), ("CAND_OVERFLOW", 2), ("EDGE_OVERFLOW", 4)):
        assert re.search(rf"#define FEGNN_LIVE_{name} {value}u", header)
        assert getattr(_lib, "LIVE_" + name) == value


def test_seven_argument_graph_leaves_n_edges_null():
    g = _lib.Graph(FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, None)
    assert g.n_edges is None


def test_new_symbols_in_header_and_binding():
    header = open(os.path.join(ROOT, "include", "fegnn.h")).read()
    for name in ("fegnn_graph_prep_live", "fegnn_radius_graph_fill_live"):
        assert re.search(rf"\b{name}\s*\(", header)
        assert name in _lib.SIGNATURES
        assert getattr(_lib.lib, name) is not None


def test_version_is_unchanged():
    assert _lib.lib.fegnn_version() == 103


def _dims(flags=_lib.F_LIVE_EDGES, E=1000):
    return make_dims(100, 100, E, 2, 3, 2, flags)


def _graph(n_edges=None):
    return _lib.Graph(FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, None, n_edges)


def _expect_einval(rc, pattern):
    assert rc == -1, rc
    assert re.search(pattern, _lib.lib.fegnn_last_error().decode())


def test_live_flag_without_count_is_refused_before_any_launch():
    d, g, p, sv = _dims(), _graph(), _lib.LayerPtrs(), _lib.Saved()
    _expect_einval(_lib.lib.fegnn_edge_forward(C.byref(d), C.byref(g), C.byref(p), FAKE, C.byref(sv), None),
                   "n_edges is NULL")
    _expect_einval(_lib.lib.fegnn_graph_pre_forward(C.byref(d), C.byref(g), C.byref(p), FAKE, FAKE, FAKE, C.byref(sv), None),
                   "n_edges is NULL")
    table = (_lib.LayerPtrs * 2)()
    ptrs = [FAKE] * 9
    _expect_einval(_lib.lib.fegnn_model_forward_inference(C.byref(d), 2, 2, C.byref(g), table, *ptrs, FAKE, 1 << 40, None),
                   "n_edges is NULL")
    _expect_einval(_lib.lib.fegnn_model_forward(C.byref(d), 2, 2, C.byref(g), table, *ptrs, FAKE, 1 << 40, None),
                   "n_edges is NULL")
    grads = (_lib.LayerPtrs * 2)()
    _expect_einval(_lib.lib.fegnn_model_backward(C.byref(d), 2, 2, C.byref(g), table, grads, *([FAKE] * 11), FAKE, FAKE,
                                                 1 << 40, None), "n_edges is NULL")


@pytest.mark.parametrize("mode", [1, 2, 4, 5])
def test_legacy_edge_backward_modes_refuse_the_flag(mode):
    d, g = _dims(), _graph(FAKE)
    table, grads = (_lib.LayerPtrs * 2)(), (_lib.LayerPtrs * 2)()
    old = _lib.get_mode("edge_backward")
    _lib.set_mode("edge_backward", mode)
    try:
        _expect_einval(_lib.lib.fegnn_model_backward(C.byref(d), 2, 2, C.byref(g), table, grads, *([FAKE] * 11), FAKE, FAKE,
                                                     1 << 40, None), f"edge_backward mode {mode}")
        sv, p = _lib.Saved(), _lib.LayerPtrs()
        _expect_einval(_lib.lib.fegnn_edge_backward(C.byref(d), C.byref(g), C.byref(p), C.byref(p), FAKE, C.byref(sv), FAKE,
                                                    FAKE, FAKE, FAKE, FAKE, None), f"edge_backward mode {mode}")
    finally:
        _lib.set_mode("edge_backward", old)


def test_prep_live_needs_its_count_words():
    rc = _lib.lib.fegnn_graph_prep_live(10, 20, 1, 0, *([FAKE] * 3), *([FAKE] * 9), FAKE, 1 << 30, None, FAKE, FAKE, None)
    _expect_einval(rc, "n_edges_in")
    rc = _lib.lib.fegnn_radius_graph_fill_live(10, 1, 2, 1.0, 1.0, *([FAKE] * 4), 10, FAKE, FAKE, FAKE, 10, *([FAKE] * 6),
                                               None, FAKE, FAKE, 1 << 30, None)
    _expect_einval(rc, "n_live")


def test_python_arguments_are_checked_before_device_work():
    ei = torch.zeros(2, 8, dtype=torch.int64)
    db = torch.zeros(4, dtype=torch.int64)
    with pytest.raises(_lib.FegnnError, match="one-element"):
        CsrGraph(ei, db, None, 1, n_edges=torch.zeros(2, dtype=torch.int32))
    with pytest.raises(_lib.FegnnError, match="one-element"):
        CsrGraph(ei, db, None, 1, n_edges=torch.zeros(1, 1, dtype=torch.int32))
    with pytest.raises(_lib.FegnnError, match="int32 or int64"):
        CsrGraph(ei, db, None, 1, n_edges=torch.zeros(1, dtype=torch.float32))
    x = torch.zeros(4, 3)
    with pytest.raises(_lib.FegnnError, match="must be >= 0"):
        CsrGraph.from_radius(x, db, 1, 1.0, capacity=-1)
    with pytest.raises(_lib.FegnnError, match="must be >= 0"):
        CsrGraph.from_radius(x, db, 1, 1.0, capacity=10, candidate_capacity=-5)
    with pytest.raises(_lib.FegnnError, match="needs a capacity"):
        CsrGraph.from_radius(x, db, 1, 1.0, candidate_capacity=10)
