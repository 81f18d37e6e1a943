"""CPU: host-side behaviour of sscvae_decode_attention and the decode workspace regions it reads (no device needed)."""
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


def test_decode_attention_is_exported_and_refused_before_any_decode(handle):
    L, h = handle
    assert hasattr(ctypes.CDLL(_lib.LIB_PATH), "sscvae_decode_attention")
    assert "sscvae_decode_attention" in _lib.SYMBOLS
    # host buffers stand in for the device pointers: the call must fail before it touches them or the device
    buf = ctypes.create_string_buffer(256)
    p = ctypes.cast(buf, ctypes.c_void_p)
    # a workspace-size query plans a decode but is not one
    assert L.sscvae_decode_workspace_bytes(h, 4, 36, 8, 5) > 0
    rc = L.sscvae_decode_attention(h, p, 1 << 40, None, p, p, None)
    assert rc == -1                     # SSCVAE_ERR_BAD_ARG
    assert b"no decode call" in L.sscvae_last_error()
    assert L.sscvae_decode_attention(h, None, 1 << 40, None, None, p, None) == -1
    assert L.sscvae_decode_attention(h, p, 1 << 40, None, p, None, None) == -1
    assert b"NULL" in L.sscvae_last_error()


def test_attention_history_regions(handle):
    L, h = handle
    off, nb = ctypes.c_size_t(), ctypes.c_size_t()
    B, N, S, K, steps = 4, 36, 8, 5, 20
    R = B * S * K
    total = L.sscvae_decode_workspace_bytes(h, B, N, S, K)
    for name, size in [("alpha_hist", steps * R * N * 4), ("best_state", B * 4), ("search_steps", B * 4)]:
        _lib.check(L.sscvae_decode_region(h, B, N, S, K, name.encode(), ctypes.byref(off), ctypes.byref(nb)))
        assert nb.value == size, name
        assert off.value + nb.value <= total
    # the single-step region it replaces is gone
    assert L.sscvae_decode_region(h, B, N, S, K, b"alpha", ctypes.byref(off), ctypes.byref(nb)) == -1
    J = 20
    _lib.check(L.sscvae_decode_samples_search_region(h, B, J, N, S, K, 1, b"alpha_hist", ctypes.byref(off), ctypes.byref(nb)))
    assert nb.value == steps * B * J * S * K * N * 4
