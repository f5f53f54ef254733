"""FEGNN_F_RECOMPUTE without a GPU: the training stack's workspace query with and without the flag, the workspace check of
fegnn_model_forward, the refusal of the flag by the per-layer entries, and the module attribute's plumbing into the
autograd Function (the backward follows the forward's choice)."""
import contextlib
import ctypes as C
import sys

import pytest
import torch

from fastegnn_b200 import FastEGNN, FastRF, _lib
from fastegnn_b200.ops import make_dims

SHAPES = [(8000, 190_000, 1, 3), (10_470, 170_000, 20, 3), (100_000, 800_000, 1, 8), (1_000_000, 24_000_000, 1, 8)]


def per_state(N, B, nc):
    al4 = lambda n: (n + 3) & ~3
    return al4(N * 64) + al4(N * 3) + al4(B * 3 * nc) + al4(B * nc * 64) + al4(B * 3)


@pytest.mark.parametrize("N,E,B,nc", SHAPES)
@pytest.mark.parametrize("L", [1, 2, 3, 4, 8, 32])
def test_workspace_query(N, E, B, nc, L):
    plain = make_dims(N, N, E, B, nc, 2, 0, None)
    rc = make_dims(N, N, E, B, nc, 2, _lib.F_RECOMPUTE, None)
    block = _lib.lib.fegnn_layer_saved_floats(C.byref(plain))
    assert _lib.lib.fegnn_layer_saved_floats(C.byref(rc)) == block
    assert _lib.lib.fegnn_model_workspace_floats(C.byref(plain), L) == (L + 1) * per_state(N, B, nc) + L * block
    assert _lib.lib.fegnn_model_workspace_floats(C.byref(rc), L) == (L + 1) * per_state(N, B, nc) + min(L, 2) * block


def test_saved_block_sizes_match_the_issue_table():
    """1 M nodes, C = 8: a saved block is about 1 556 + 256 C bytes per node."""
    d = make_dims(1_000_000, 1_000_000, 24_000_000, 1, 8, 2, 0, None)
    per_node = 4 * _lib.lib.fegnn_layer_saved_floats(C.byref(d)) / 1e6
    assert abs(per_node - (1556 + 256 * 8)) < 0.01 * per_node


def _call_forward(dims, L, ws_floats):
    dummy = C.c_void_p(16)              # never dereferenced: the workspace check comes before any launch
    table, g = (_lib.LayerPtrs * L)(), _lib.Graph()
    return _lib.lib.fegnn_model_forward(C.byref(dims), L, 1, C.byref(g), table, *([dummy] * 9), dummy, ws_floats, None)


@pytest.mark.parametrize("L", [1, 4, 8])
def test_short_workspace_refused_before_any_launch(L):
    rc = make_dims(8000, 8000, 190_000, 1, 3, 2, _lib.F_RECOMPUTE, None)
    need = _lib.lib.fegnn_model_workspace_floats(C.byref(rc), L)
    before = _lib.lib.fegnn_launch_count()
    assert _call_forward(rc, L, need - 1) == -3                           # FEGNN_ENOMEM
    assert b"model workspace" in _lib.lib.fegnn_last_error()
    assert _lib.lib.fegnn_launch_count() == before


def _null_args(fn):
    """NULL for every argument after the dims (the flag check comes first; the entries have at most 23 more arguments)."""
    at = getattr(_lib.lib, fn).argtypes
    return [0 if t in (C.c_int32, C.c_int64, C.c_size_t) else None for t in at[1:]] if at else [None] * 23


PHASES = ["fegnn_graph_pre_forward", "fegnn_node_pre_forward", "fegnn_edge_forward", "fegnn_graph_post_forward",
          "fegnn_node_h_weight_images", "fegnn_graph_post_backward", "fegnn_node_h_backward", "fegnn_virtual_backward",
          "fegnn_virtual_backward_inputs", "fegnn_edge_backward", "fegnn_edge_backward_inputs", "fegnn_graph_pre_backward",
          "fegnn_node_pre_backward", "fegnn_node_pre_backward_inputs"]


@pytest.mark.parametrize("flag", ["F_RECOMPUTE", "F_REBUILD_ALL"])
@pytest.mark.parametrize("fn", PHASES)
def test_per_phase_entries_refuse_the_flag(fn, flag):
    rc = make_dims(1000, 1000, 9000, 2, 3, 2, getattr(_lib, flag), None)
    before = _lib.lib.fegnn_launch_count()
    assert getattr(_lib.lib, fn)(C.byref(rc), *_null_args(fn)) == -1     # FEGNN_EINVAL
    assert b"FEGNN_F_RECOMPUTE" in _lib.lib.fegnn_last_error()
    assert _lib.lib.fegnn_launch_count() == before


@pytest.mark.parametrize("fn", ["fegnn_virtual_forward", "fegnn_node_h_forward"])
def test_saved_only_phases_take_the_flag(fn):
    """The two saved-only forms accept the flag: they get past it to the argument checks (null pointers here)."""
    rc = make_dims(1000, 1000, 9000, 2, 3, 2, _lib.F_RECOMPUTE, None)
    assert getattr(_lib.lib, fn)(C.byref(rc), *_null_args(fn)) == -1
    assert b"FEGNN_F_RECOMPUTE" not in _lib.lib.fegnn_last_error()


class _Stop(Exception):
    pass


@pytest.mark.parametrize("cls", [FastEGNN, FastRF])
def test_attribute_reaches_the_forward_and_the_backward_follows_it(monkeypatch, cls):
    """recompute is a class attribute (default False) settable per instance.  _StackFn.forward sizes the workspace with the
    flag of the attribute's value at the forward and keeps that dims block for the backward: flipping the attribute between
    the two changes nothing."""
    F = sys.modules["fastegnn_b200.FastEGNN"]          # the module that holds _StackFn (the package exports the class)
    assert cls.recompute is False
    m = cls(node_feat_nf=1, node_attr_nf=0, edge_attr_nf=0, hidden_nf=64, virtual_channels=3, device="cpu", n_layers=4)
    assert m.recompute is False
    m.recompute = True
    other = cls(node_feat_nf=1, node_attr_nf=0, edge_attr_nf=0, hidden_nf=64, virtual_channels=3, device="cpu", n_layers=4)
    assert other.recompute is False                  # per instance

    seen = {}

    def fake_ws(pd, L):
        seen["ws_flags"] = C.cast(pd, C.POINTER(_lib.Dims)).contents.flags
        raise _Stop

    monkeypatch.setattr(F, "lib", type("L", (), {"fegnn_model_workspace_floats": staticmethod(fake_ws)}))

    class Ctx:
        pass
    graph = type("G", (), dict(N=4, B=1, E=4, Fe=0))()
    monkeypatch.setattr(m, "_param_table", lambda: (None, []))
    with pytest.raises(_Stop):
        F._StackFn.forward(Ctx(), m, graph, None, None, None, torch.ones(4, 1), torch.zeros(4, 3), torch.zeros(4, 3),
                           torch.zeros(1, 3, 3))
    assert seen["ws_flags"] & _lib.F_RECOMPUTE
    assert (seen["ws_flags"] & ~_lib.F_RECOMPUTE) == m._flag_word
    m.recompute = False
    with pytest.raises(_Stop):
        F._StackFn.forward(Ctx(), m, graph, None, None, None, torch.ones(4, 1), torch.zeros(4, 3), torch.zeros(4, 3),
                           torch.zeros(1, 3, 3))
    assert not seen["ws_flags"] & _lib.F_RECOMPUTE


@pytest.mark.parametrize("recompute", [True, False])
def test_backward_reads_the_flag_from_ctx(monkeypatch, recompute):
    """_StackFn.backward passes ctx.dims (the forward's flag word) to fegnn_model_backward_inputs, whatever the attribute
    says by then.  With recompute, a second backward over the same forward (retain_graph) adds FEGNN_F_REBUILD_ALL: the
    first one left the two saved blocks holding other layers.  ctx.dims itself is not changed."""
    F = sys.modules["fastegnn_b200.FastEGNN"]
    m = FastEGNN(node_feat_nf=1, node_attr_nf=0, edge_attr_nf=0, hidden_nf=64, virtual_channels=3, device="cpu", n_layers=4)
    m.recompute = not recompute                      # the attribute flipped after the forward
    seen = []

    def fake_bwd(pd, *a):
        seen.append(C.cast(pd, C.POINTER(_lib.Dims)).contents.flags)
        return 0

    fake = type("L", (), {"fegnn_model_backward_inputs": staticmethod(fake_bwd),
                          "fegnn_model_backward_scratch_floats": staticmethod(lambda pd: 4)})
    monkeypatch.setattr(F, "lib", fake)
    monkeypatch.setattr(m, "_param_table", lambda: (None, []))
    views = {k: torch.zeros(1) for k in ("embedding_in.weight", "embedding_in.bias", "virtual_node_feat")}
    monkeypatch.setattr(m, "_grad_table", lambda dev: (None, views, None))
    monkeypatch.setattr(F, "_on", lambda dev: contextlib.nullcontext())
    monkeypatch.setattr(F, "_stream", lambda dev: None)

    class Ctx:
        pass
    ctx = Ctx()
    ctx.mod, ctx.graph, ctx.Fin, ctx.ws = m, type("G", (), dict(N=4, B=1, E=4, Fe=0, perm=None, c=_lib.Graph()))(), 1, None
    ctx.recompute, ctx.blocks_consumed = recompute, False
    ctx.dims = make_dims(4, 4, 4, 1, 3, 0, m._flag_word | (_lib.F_RECOMPUTE if recompute else 0), None)
    ctx.saved_tensors = (torch.ones(4, 1), torch.zeros(4, 3), None)
    ctx.need_nf, ctx.needs_input_grad = False, (False,) * 9
    ctx.names, ctx.in_dtypes = [], (None, None, torch.float32)
    for _ in range(3):
        F._StackFn.backward(ctx, torch.zeros(4, 3), torch.zeros(1, 3, 3))
    assert [bool(f & _lib.F_RECOMPUTE) for f in seen] == [recompute] * 3
    assert [bool(f & _lib.F_REBUILD_ALL) for f in seen] == [False, recompute, recompute]
    assert not ctx.dims.flags & _lib.F_REBUILD_ALL


def test_rebuild_all_needs_recompute():
    """FEGNN_F_REBUILD_ALL without FEGNN_F_RECOMPUTE: the backward refuses it before any launch."""
    d = make_dims(1000, 1000, 9000, 2, 3, 2, _lib.F_REBUILD_ALL, None)
    dummy = C.c_void_p(16)
    table, g = (_lib.LayerPtrs * 4)(), _lib.Graph()
    before = _lib.lib.fegnn_launch_count()
    rc = _lib.lib.fegnn_model_backward_inputs(C.byref(d), 4, 1, C.byref(g), table, table, *([dummy] * 13), 1 << 30, None,
                                              None)
    assert rc == -1 and b"FEGNN_F_REBUILD_ALL" in _lib.lib.fegnn_last_error()
    assert _lib.lib.fegnn_launch_count() == before


def test_deterministic_training_still_raises():
    m = FastEGNN(node_feat_nf=1, node_attr_nf=0, edge_attr_nf=0, hidden_nf=64, virtual_channels=3, device="cpu", n_layers=2)
    m.recompute = True
    on, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        ei = torch.tensor([[0, 1, 2, 3], [1, 0, 3, 2]])
        with pytest.raises(RuntimeError, match="FastEGNN does not have a deterministic implementation"):
            m(torch.ones(4, 1), torch.randn(4, 3), torch.randn(4, 3), ei, torch.zeros(4, dtype=torch.long),
              torch.zeros(1, 3, 3))
    finally:
        torch.use_deterministic_algorithms(on, warn_only=warn_only)
        _lib.set_mode("deterministic", 0)
