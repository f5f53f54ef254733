"""Deterministic mode, host side: the library mode round-trips, entries without a deterministic form refuse to run under
it before touching the device, and the package turns torch.use_deterministic_algorithms(True) into an error (or a
warning under warn_only=True) for the models that have no deterministic form."""
import warnings

import pytest
import torch

from fastegnn_b200 import FastEGNN, _lib, unsorted_segment_sum
from fastegnn_b200.ops import make_dims


@pytest.fixture
def torch_flag():
    """Restores torch's flag and the library mode after the test."""
    on, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    yield
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    _lib.set_mode("deterministic", 0)


def test_mode_round_trips(torch_flag):
    assert _lib.get_mode("deterministic") == 0
    _lib.set_mode("deterministic", 1)
    assert _lib.get_mode("deterministic") == 1
    with pytest.raises(_lib.FegnnError, match="deterministic mode must be 0 or 1"):
        _lib.set_mode("deterministic", 2)
    assert _lib.get_mode("deterministic") == 1
    _lib.set_mode("deterministic", 0)
    assert _lib.get_mode("deterministic") == 0


def test_uncovered_entries_refuse_under_the_mode(torch_flag):
    _lib.set_mode("deterministic", 1)
    assert _lib.lib.fegnn_graph_xsum(0, 0, None, None, None, None) == -1
    assert b"fegnn_graph_xsum has no deterministic form" in _lib.lib.fegnn_last_error()
    dims = make_dims(8, 8, 16, 1, 3, 0, 0, None)
    import ctypes as C
    rc = _lib.lib.fegnn_model_forward(C.byref(dims), 1, 1, None, None, *([None] * 9), None, 0, None)
    assert rc == -1 and b"fegnn_model_forward has no deterministic form" in _lib.lib.fegnn_last_error()


def test_loss_workspace_only_under_the_mode(torch_flag):
    """The deterministic loss forward keeps one partial per CTA in a caller's workspace: the query answers 0 with the mode
    off, and the forward refuses a missing or short workspace under the mode before touching the device."""
    assert _lib.lib.fegnn_loss_workspace_floats(8000, 20) == 0
    _lib.set_mode("deterministic", 1)
    n = _lib.lib.fegnn_loss_workspace_floats(8000, 20)
    assert n >= 20 + 2 and _lib.lib.fegnn_loss_workspace_floats(0, 20) <= n
    dummy = 256          # never dereferenced: the workspace check comes first
    rc = _lib.lib.fegnn_mse_mmd_forward(8000, 20, 3, 4, 1.5, 0.01, 1.0, 1.0, 1.0, *([dummy] * 6), dummy, n - 1, None)
    assert rc == -3 and b"loss workspace" in _lib.lib.fegnn_last_error()
    rc = _lib.lib.fegnn_mmd_forward(20, 3, 4, 1.5, 1.0, 1.0, *([dummy] * 4), None, 0, None)
    assert rc == -3 and b"loss workspace" in _lib.lib.fegnn_last_error()


def test_model_workspace_queries_do_not_depend_on_the_mode(torch_flag):
    """The model's size queries answer the same in both modes (the model has no deterministic form to size for)."""
    import ctypes as C
    dims = make_dims(1000, 1000, 20000, 2, 3, 2, 0, None)
    queries = lambda: (_lib.lib.fegnn_model_workspace_floats(C.byref(dims), 4),
                       _lib.lib.fegnn_model_backward_scratch_floats(C.byref(dims)),
                       _lib.lib.fegnn_model_inference_workspace_floats(C.byref(dims)),
                       _lib.lib.fegnn_graph_prep_workspace_bytes(1000, 20000))
    off = queries()
    _lib.set_mode("deterministic", 1)
    assert queries() == off


def _cpu_model():
    torch.manual_seed(0)
    return FastEGNN(node_feat_nf=1, node_attr_nf=0, edge_attr_nf=0, hidden_nf=64, virtual_channels=3, device="cpu",
                    n_layers=2)


def _cpu_inputs():
    ei = torch.tensor([[0, 1, 2, 3], [1, 0, 3, 2]])
    return dict(node_feat=torch.ones(4, 1), node_loc=torch.randn(4, 3), node_vel=torch.randn(4, 3), edge_index=ei,
                data_batch=torch.zeros(4, dtype=torch.long), loc_mean=torch.zeros(1, 3, 3))


def test_model_raises_under_torch_flag(torch_flag):
    model = _cpu_model()
    torch.use_deterministic_algorithms(True)
    with pytest.raises(RuntimeError, match="FastEGNN does not have a deterministic implementation"):
        model(**_cpu_inputs())
    with pytest.raises(RuntimeError, match="unsorted_segment_sum does not have a deterministic implementation"):
        unsorted_segment_sum(torch.ones(4, 2), torch.zeros(4, dtype=torch.long), 1)


def test_model_warns_and_runs_as_default_under_warn_only(torch_flag):
    model = _cpu_model()
    _lib.set_mode("deterministic", 1)
    torch.use_deterministic_algorithms(True, warn_only=True)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        with pytest.raises(_lib.FegnnError, match="no CPU fallback"):    # past the policy: the CUDA check refuses
            model(**_cpu_inputs())
    assert any("FastEGNN does not have a deterministic implementation" in str(x.message) for x in w)
    assert _lib.get_mode("deterministic") == 0


def test_flag_off_leaves_the_library_mode_off(torch_flag):
    model = _cpu_model()
    _lib.set_mode("deterministic", 1)
    torch.use_deterministic_algorithms(False)
    with pytest.raises(_lib.FegnnError, match="no CPU fallback"):
        model(**_cpu_inputs())
    assert _lib.get_mode("deterministic") == 0
