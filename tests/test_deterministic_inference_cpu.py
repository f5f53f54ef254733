"""The deterministic forward-only stack without a GPU: its workspace query, the workspace check of
fegnn_model_forward_inference under the mode, and the module policy (eval() / torch.no_grad() pass it, training raises)."""
import ctypes as C
import warnings

import pytest
import torch

from fastegnn_b200 import FastEGNN, FastRF, _lib
from fastegnn_b200.ops import make_dims


@pytest.fixture
def torch_flag():
    on, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    yield
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    _lib.set_mode("deterministic", 0)


@pytest.mark.parametrize("N,E,B,nc", [(8000, 190_000, 1, 3), (10_470, 170_000, 20, 3), (100_000, 800_000, 1, 8),
                                     (1_000_000, 24_000_000, 1, 8)])
def test_det_workspace_query_only_under_the_mode(torch_flag, N, E, B, nc):
    dims = make_dims(N, N, E, B, nc, 2, 0, None)
    base = _lib.lib.fegnn_model_inference_workspace_floats(C.byref(dims))
    assert _lib.lib.fegnn_model_inference_det_workspace_floats(C.byref(dims)) == 0
    _lib.set_mode("deterministic", 1)
    det = _lib.lib.fegnn_model_inference_det_workspace_floats(C.byref(dims))
    # at least the edge tiles' boundary slab (2 slots of 68 floats per 128 edges) and the rows D sX (N C 3)
    assert det >= (E + 127) // 128 * 2 * 68 + N * nc * 3
    assert det < base                                       # a fraction of what the stack already takes
    assert _lib.lib.fegnn_model_inference_workspace_floats(C.byref(dims)) == base


def _call_inference(dims, ws_floats):
    dummy = C.c_void_p(16)              # never dereferenced: the workspace check comes before any launch
    table, g = (_lib.LayerPtrs * 1)(), _lib.Graph()
    return _lib.lib.fegnn_model_forward_inference(C.byref(dims), 1, 1, C.byref(g), table, *([dummy] * 9), dummy, ws_floats,
                                                  None)


def test_short_workspace_refused_before_any_launch(torch_flag):
    dims = make_dims(8000, 8000, 190_000, 1, 3, 2, 0, None)
    base = _lib.lib.fegnn_model_inference_workspace_floats(C.byref(dims))
    _lib.set_mode("deterministic", 1)
    det = _lib.lib.fegnn_model_inference_det_workspace_floats(C.byref(dims))
    for short in (base, base + det - 1):
        assert _call_inference(dims, short) == -3                        # FEGNN_ENOMEM
        assert b"inference workspace" in _lib.lib.fegnn_last_error()
    _lib.set_mode("deterministic", 0)
    assert _call_inference(dims, base - 1) == -3


def _cpu_inputs():
    ei = torch.tensor([[0, 1, 2, 3], [1, 0, 3, 2]])
    return dict(node_feat=torch.ones(4, 1), node_loc=torch.randn(4, 3), node_vel=torch.randn(4, 3), edge_index=ei,
                data_batch=torch.zeros(4, dtype=torch.long), loc_mean=torch.zeros(1, 3, 3))


@pytest.mark.parametrize("cls", [FastEGNN, FastRF])
def test_forward_only_stack_passes_the_policy(torch_flag, cls):
    torch.manual_seed(0)
    model = cls(node_feat_nf=1, node_attr_nf=0, edge_attr_nf=0, hidden_nf=64, virtual_channels=3, device="cpu", n_layers=2)
    torch.use_deterministic_algorithms(True)
    for route in ("eval", "no_grad"):
        model.train(route != "eval")
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            with torch.set_grad_enabled(route != "no_grad"):
                with pytest.raises(_lib.FegnnError, match="no CPU fallback"):      # past the policy: the CUDA check
                    model(**_cpu_inputs())
        assert not any("deterministic" in str(x.message) for x in w), route
        assert _lib.get_mode("deterministic") == 1
    model.train()
    with pytest.raises(RuntimeError, match=f"{cls.__name__} does not have a deterministic implementation"):
        model(**_cpu_inputs())
    model.eval()
    model.eval_keeps_graph = True                  # the training forward in eval mode: still no deterministic form
    with pytest.raises(RuntimeError, match=f"{cls.__name__} does not have a deterministic implementation"):
        model(**_cpu_inputs())
