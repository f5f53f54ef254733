"""The stack entries check every layer's parameters against the flags before their first launch: a layer table whose
layer 1 lacks its gravity tensors is refused with FEGNN_EINVAL naming that layer, and nothing is launched (under stream
capture a late refusal would leave the side stream's fork unjoined).  Every size is 0 and every other pointer a dummy
that is never dereferenced."""
import ctypes as C

import pytest

from fastegnn_b200 import _lib
from fastegnn_b200.ops import make_dims

L = 3
DUMMY = C.c_void_p(16)


def _table():
    table = (_lib.LayerPtrs * L)()
    for l in (0, 2):
        for k in ("grav_w0", "grav_b0", "grav_w2", "grav_b2"):
            setattr(table[l], k, 16)
    return table


def _forward(d):
    ws = _lib.lib.fegnn_model_workspace_floats(C.byref(d), L)
    return _lib.lib.fegnn_model_forward(C.byref(d), L, 1, C.byref(_lib.Graph()), _table(), *([DUMMY] * 9), DUMMY, ws, None)


def _inference(d):
    ws = _lib.lib.fegnn_model_inference_workspace_floats(C.byref(d))
    return _lib.lib.fegnn_model_forward_inference(C.byref(d), L, 1, C.byref(_lib.Graph()), _table(), *([DUMMY] * 9), DUMMY,
                                                  ws, None)


def _backward(d):
    scratch = _lib.lib.fegnn_model_backward_scratch_floats(C.byref(d))
    t = _table()
    return _lib.lib.fegnn_model_backward(C.byref(d), L, 1, C.byref(_lib.Graph()), t, t, *([DUMMY] * 13), scratch, None)


@pytest.mark.parametrize("call", [_forward, _inference, _backward])
def test_missing_layer_params_refused_before_any_launch(call):
    d = make_dims(0, 0, 0, 0, 3, 2, _lib.F_GRAVITY, None)
    before = _lib.lib.fegnn_launch_count()
    assert call(d) == -1                                                   # FEGNN_EINVAL
    msg = _lib.lib.fegnn_last_error()
    assert b"layer 1" in msg and b"gravity" in msg, msg
    assert _lib.lib.fegnn_launch_count() == before
