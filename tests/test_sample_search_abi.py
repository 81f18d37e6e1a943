"""CPU: host-side queries and argument checks of sscvae_decode_samples_search (no device needed)."""
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


def test_workspace_query_at_bench_dims(handle):
    L, h = handle
    # 16 images x 20 samples x S 8 x K 5 = 12 800 rows: the (rows, V) fp32 logits alone are 512 MB
    shared = L.sscvae_decode_samples_search_workspace_bytes(h, 16, 20, 36, 8, 5, 0)
    own = L.sscvae_decode_samples_search_workspace_bytes(h, 16, 20, 36, 8, 5, 1)
    assert 512e6 < shared < 2e9, shared
    # one packed (S, V) uint32 table per image, or per sample: 19 more tables of 8 x 10 000 words per image
    assert own - shared >= 16 * 19 * 8 * 10000 * 4 and own - shared < 16 * 19 * 8 * 10000 * 4 + 4096
    # the shipped shape: S 1, K 1, 64 images x 20 samples
    s1 = L.sscvae_decode_samples_search_workspace_bytes(h, 64, 20, 36, 1, 1, 0)
    assert 50e6 < s1 < 1e9, s1
    # one sample per image is the batch's own decode workspace, apart from the per-image FSM count it keys on
    assert L.sscvae_decode_samples_search_workspace_bytes(h, 4, 1, 36, 8, 5, 0) == L.sscvae_decode_workspace_bytes(h, 4, 36, 8, 5)
    for bad in [(16, 0, 36, 8, 5, 0), (16, 20, 36, 33, 5, 0), (16, 20, 36, 8, 9, 0), (16, 20, 36, 8, 5, 2), (0, 20, 36, 8, 5, 0)]:
        assert L.sscvae_decode_samples_search_workspace_bytes(h, *bad) == 0, bad


def test_region_lookup(handle):
    L, h = handle
    off, nb = ctypes.c_size_t(), ctypes.c_size_t()
    R = 4 * 20 * 8 * 5
    for name, size in [("tok_hist", 20 * R * 4), ("bp_hist", 20 * R * 4), ("score_hist", 20 * R * 4),
                       ("logits", R * 10000 * 4), ("fsm_bits", 4 * 8 * 10000 * 4)]:
        _lib.check(L.sscvae_decode_samples_search_region(h, 4, 20, 36, 8, 5, 0, name.encode(), ctypes.byref(off),
                                                         ctypes.byref(nb)))
        assert nb.value == size, name
    _lib.check(L.sscvae_decode_samples_search_region(h, 4, 20, 36, 8, 5, 1, b"fsm_bits", ctypes.byref(off), ctypes.byref(nb)))
    assert nb.value == 4 * 20 * 8 * 10000 * 4
    total = L.sscvae_decode_samples_search_workspace_bytes(h, 4, 20, 36, 8, 5, 1)
    assert off.value + nb.value <= total
    rc = L.sscvae_decode_samples_search_region(h, 4, 20, 36, 8, 5, 0, b"nope", ctypes.byref(off), ctypes.byref(nb))
    assert rc == -1                     # SSCVAE_ERR_BAD_ARG
    assert b"nope" in L.sscvae_last_error()


@pytest.mark.parametrize("batch,samples,states,beam,per_node,fsm_per_sample,has_fsm,what", [
    (2, 3, 33, 5, 2, 0, True, "bad decode shape"),          # S <= 32
    (2, 3, 8, 9, 2, 0, True, "bad decode shape"),           # K <= 8
    (2, 3, 8, 5, 6, 0, True, "bad decode shape"),           # P <= K
    (2, 3, 8, 5, 0, 0, True, "bad decode shape"),           # P >= 1
    (2, 0, 8, 5, 2, 0, True, "bad decode shape"),           # J >= 1
    (2, 3, 8, 5, 2, 2, True, "bad decode shape"),           # fsm_per_sample is 0 or 1
    (2, 3, 8, 5, 2, 0, False, "an FSM is required"),        # S > 1 without a machine
])
def test_bad_arguments_are_refused_without_a_device(handle, batch, samples, states, beam, per_node, fsm_per_sample,
                                                    has_fsm, what):
    """The checks run before any CUDA call: host buffers stand in for the device pointers and are never touched."""
    L, h = handle
    buf = ctypes.create_string_buffer(256)
    p = ctypes.cast(buf, ctypes.c_void_p)
    weights = (ctypes.c_void_p * _lib.W_COUNT)(*([p.value] * _lib.W_COUNT))
    rc = L.sscvae_decode_samples_search(h, batch, samples, 36, states, beam, per_node, p, weights, p, p, None,
                                        p if has_fsm else None, fsm_per_sample, None, 2, None, ctypes.c_uint64(1), p, 256,
                                        p, p, p, p, None)
    assert rc == -1                     # SSCVAE_ERR_BAD_ARG
    assert what.encode() in L.sscvae_last_error()
