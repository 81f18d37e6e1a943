"""CPU: host-side behaviour of sscvae_decode_step, the single decode step (no device needed)."""
import ctypes

import pytest

from sscvae import _lib


@pytest.fixture
def handle():
    L = _lib.lib()
    h = ctypes.c_void_p()
    d = _lib.SscvaeDims(2048, 600, 900, 768, 150, 10000, 20, 1, 0, 1, 0, 1, 1.0, 0.5)    # the bench dims
    _lib.check(L.sscvae_create(ctypes.byref(d), ctypes.byref(h)))
    yield L, h
    L.sscvae_destroy(h)


def test_decode_step_is_exported():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in ("sscvae_decode_step", "sscvae_decode_step_workspace_bytes"):
        assert hasattr(lib, name)
        assert name in _lib.SYMBOLS


def test_workspace_bytes_grow_with_rows_and_refuse_ragged_rows(handle):
    L, h = handle
    B, N = 16, 36
    sizes = [L.sscvae_decode_step_workspace_bytes(h, B, R, N) for R in (B, 5 * B, 40 * B)]
    assert 0 < sizes[0] < sizes[1] < sizes[2]
    # at R = 640 the step workspace holds, among others, the head GEMM's softmax partials: R * 79 tiles * 12 bytes
    assert sizes[2] > 640 * 79 * 12
    assert L.sscvae_decode_step_workspace_bytes(h, B, 40 * B + 1, N) == 0
    assert L.sscvae_decode_step_workspace_bytes(h, 0, 16, N) == 0
    assert L.sscvae_decode_step_workspace_bytes(None, B, B, N) == 0


def _call(L, h, B=2, R=4, N=3, null=None, states_in=True, states_out=True):
    """sscvae_decode_step with host buffers standing in for every device pointer: the call must return before it
    touches any of them or the device. `null` names the argument to pass as NULL."""
    buf = ctypes.create_string_buffer(1 << 12)
    p = ctypes.cast(buf, ctypes.c_void_p)
    arr = lambda n: (ctypes.c_void_p * n)(*([p.value] * n))
    args = dict(packed=p, weights=arr(_lib.W_COUNT), feats=p, sentiment=p, prev=p, ws=p, log_probs=p, alpha=p, pm_out=p)
    if null is not None:
        args[null] = None
    sin = arr(6) if states_in is True else states_in
    sout = arr(4) if states_out is True else states_out
    return L.sscvae_decode_step(h, B, R, N, args["packed"], args["weights"], args["feats"], args["sentiment"], None, None,
                                None, args["prev"], sin, None, 0, args["ws"], 1 << 40, args["log_probs"], sout,
                                args["alpha"], args["pm_out"], None)


def test_refuses_ragged_rows_before_any_device_work(handle):
    L, h = handle
    assert _call(L, h, B=2, R=5) == -1                              # SSCVAE_ERR_BAD_ARG
    assert b"multiple of B" in L.sscvae_last_error()
    assert _call(L, h, B=3, R=0) == -1


@pytest.mark.parametrize("null", ["packed", "weights", "feats", "prev", "ws", "log_probs", "alpha", "pm_out", "sentiment"])
def test_refuses_null_pointers_before_any_device_work(handle, null):
    L, h = handle
    assert _call(L, h, null=null) == -1
    msg = L.sscvae_last_error()
    assert b"NULL" in msg or b"sentiment" in msg


def test_refuses_incomplete_state_arrays(handle):
    L, h = handle
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p).value
    no_c1 = (ctypes.c_void_p * 6)(p, None, None, None, p, p)
    assert _call(L, h, states_in=no_c1) == -1
    assert b"states_in" in L.sscvae_last_error()
    assert _call(L, h, states_out=None) == -1
    assert _call(L, h, states_out=(ctypes.c_void_p * 4)(p, p, None, p)) == -1
    assert b"states_out" in L.sscvae_last_error()
