"""CPU: host-side behaviour of the training step's C entry points (sscvae_train_step_*), no device needed."""
import ctypes

import pytest

from sscvae import _lib

NAMES = ("sscvae_train_step_image_state_bytes", "sscvae_train_step_tape_bytes", "sscvae_train_step_workspace_bytes",
         "sscvae_train_step_image_state", "sscvae_train_step_forward", "sscvae_train_step_backward")
SIZES = NAMES[:3]


def _handle(sv=1, tied=1):
    L = _lib.lib()
    h = ctypes.c_void_p()
    E = 600 if tied else 512
    d = _lib.SscvaeDims(2048, E, 900, 768, 150, 10000, 20, sv, 0, tied, 0, 1, 1.0, 0.5)    # the bench dims
    _lib.check(L.sscvae_create(ctypes.byref(d), ctypes.byref(h)))
    return L, h


@pytest.fixture
def handle():
    L, h = _handle()
    yield L, h
    L.sscvae_destroy(h)


def test_train_step_is_exported():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in NAMES:
        assert hasattr(lib, name)
        assert name in _lib.SYMBOLS


def test_sizes_are_positive_grow_with_batch_and_refuse_bad_arguments(handle):
    L, h = handle
    for name in SIZES:
        f = getattr(L, name)
        sizes = [f(h, B, 36) for B in (1, 16, 256)]
        assert 0 < sizes[0] < sizes[1] < sizes[2], name
        assert f(h, 16, 36) < f(h, 16, 72)
        assert f(h, 0, 36) == 0 and f(h, 16, 0) == 0 and f(None, 16, 36) == 0
    # the tape holds at least the three LSTMs' activated gates, (B, 4H) fp32 each
    assert L.sscvae_train_step_tape_bytes(h, 256, 36) > 3 * 256 * 3600 * 4


class Bufs:
    """Host buffers standing in for every device pointer, 256-byte aligned: a call must refuse before it touches them."""

    def __init__(self, L, h, B, N):
        self.sizes = {k: getattr(L, "sscvae_train_step_%s_bytes" % k)(h, B, N) for k in ("image_state", "tape", "workspace")}
        self._raw = ctypes.create_string_buffer(1 << 12)
        self.p = (ctypes.addressof(self._raw) + 255) & ~255

    def arr(self, n, null=()):
        return (ctypes.c_void_p * n)(*[None if i in null else self.p for i in range(n)])


def _forward(L, h, B=2, N=3, null=None, states_in=True, states_out=True, sizes=None, misalign=None):
    b = Bufs(L, h, B, N)
    sz = dict(b.sizes, **(sizes or {}))
    a = {k: b.p for k in ("packed", "state", "sentiment", "prev", "tape", "ws", "logits", "mean", "log_var", "pm", "alpha")}
    if null:
        a[null] = None
    if misalign:
        a[misalign] = b.p + 16
    sin = b.arr(6) if states_in is True else states_in
    sout = b.arr(6) if states_out is True else states_out
    return L.sscvae_train_step_forward(h, B, N, a["packed"], b.arr(_lib.W_COUNT), a["state"], sz["image_state"],
                                       a["sentiment"], a["prev"], sin, None, 0, a["tape"], sz["tape"], a["ws"],
                                       sz["workspace"], a["logits"], sout, a["mean"], a["log_var"], a["pm"], a["alpha"], None)


def _backward(L, h, B=2, N=3, null=None, sizes=None, misalign=None):
    b = Bufs(L, h, B, N)
    sz = dict(b.sizes, **(sizes or {}))
    a = {k: b.p for k in ("packed", "state", "tape", "ws", "d_logits")}
    if null:
        a[null] = None
    if misalign:
        a[misalign] = b.p + 16
    grads = None if null == "grads" else b.arr(_lib.W_COUNT)
    return L.sscvae_train_step_backward(h, B, N, a["packed"], b.arr(_lib.W_COUNT), a["state"], sz["image_state"], a["tape"],
                                        sz["tape"], a["ws"], sz["workspace"], a["d_logits"], None, None, None, None, None,
                                        None, grads, None)


@pytest.mark.parametrize("null", ["packed", "state", "prev", "tape", "ws", "logits", "mean", "log_var", "alpha", "sentiment"])
def test_forward_refuses_null_pointers_before_any_device_work(handle, null):
    L, h = handle
    assert _forward(L, h, null=null) == -1                          # SSCVAE_ERR_BAD_ARG
    msg = L.sscvae_last_error()
    assert b"NULL" in msg or b"sentiment" in msg


def test_forward_refuses_incomplete_state_arrays(handle):
    L, h = handle
    b = Bufs(L, h, 2, 3)
    assert _forward(L, h, states_in=b.arr(6, null=(2,))) == -1
    assert b"states_in" in L.sscvae_last_error()
    assert _forward(L, h, states_out=b.arr(6, null=(3,))) == -1
    assert b"states_out" in L.sscvae_last_error()
    assert _forward(L, h, states_out=None) == -1


@pytest.mark.parametrize("which", ["image_state", "tape", "workspace"])
def test_refuses_small_and_misaligned_buffers(handle, which):
    L, h = handle
    need = Bufs(L, h, 2, 3).sizes[which]
    assert _forward(L, h, sizes={which: need - 1}) == -2              # SSCVAE_ERR_WORKSPACE
    assert _backward(L, h, sizes={which: need - 1}) == -2
    key = {"image_state": "state", "tape": "tape", "workspace": "ws"}[which]
    assert _forward(L, h, misalign=key) == -1
    assert b"aligned" in L.sscvae_last_error()
    assert _backward(L, h, misalign=key) == -1


@pytest.mark.parametrize("null", ["packed", "state", "tape", "ws", "d_logits", "grads"])
def test_backward_refuses_null_pointers_before_any_device_work(handle, null):
    L, h = handle
    assert _backward(L, h, null=null) == -1
    assert b"NULL" in L.sscvae_last_error()


def test_sentiment_vae2_needs_obj_means_and_a_prior_mean_output():
    L, h = _handle(sv=2)
    try:
        assert _forward(L, h, null="pm") == -1
        assert b"prior_mean_out" in L.sscvae_last_error()
        b = Bufs(L, h, 2, 3)
        rc = L.sscvae_train_step_image_state(h, 2, 3, b.p, b.arr(_lib.W_COUNT), b.p, None, b.p, b.sizes["image_state"], None)
        assert rc == -1 and b"obj_means" in L.sscvae_last_error()
    finally:
        L.sscvae_destroy(h)
