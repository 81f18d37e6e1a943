"""ctypes binding of libsscvae_b200.so (include/sscvae.h). No pybind / ATen dependency: PyTorch is
only the owner of device memory and streams; tensors cross the boundary as raw pointers.

There is NO fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsscvae_b200.so")

W_NAMES = [
    "_embedding_layer.weight",
    "_updown_cell._attention_lstm_cell.weight_ih",
    "_updown_cell._attention_lstm_cell.weight_hh",
    "_updown_cell._attention_lstm_cell.bias_ih",
    "_updown_cell._attention_lstm_cell.bias_hh",
    "_updown_cell._butd_attention._query_vector_projection_layer.weight",
    "_updown_cell._butd_attention._image_features_projection_layer.weight",
    "_updown_cell._butd_attention._attention_layer.weight",
    "_updown_cell._language_lstm_cell_encoder.weight_ih",
    "_updown_cell._language_lstm_cell_encoder.weight_hh",
    "_updown_cell._language_lstm_cell_encoder.bias_ih",
    "_updown_cell._language_lstm_cell_encoder.bias_hh",
    "_updown_cell._language_lstm_cell_decoder.weight_ih",
    "_updown_cell._language_lstm_cell_decoder.weight_hh",
    "_updown_cell._language_lstm_cell_decoder.bias_ih",
    "_updown_cell._language_lstm_cell_decoder.bias_hh",
    "_updown_cell.fc_mean.weight",
    "_updown_cell.fc_mean.bias",
    "_updown_cell.fc_log_var.weight",
    "_updown_cell.fc_log_var.bias",
    "OUT_PROJ_W",   # tied: _output_projection.0.weight | untied: _output_layer.weight
    "OUT_PROJ_B",   # tied: _output_projection.0.bias   | untied: _output_layer.bias
]
W_COUNT = len(W_NAMES)
GRAD_GROUPS = 5

# every symbol include/sscvae.h declares (tests/test_abi.py checks the library exports each one)
SYMBOLS = [
    "sscvae_abi_version", "sscvae_last_error", "sscvae_launch_count", "sscvae_create", "sscvae_destroy", "sscvae_set_option", "sscvae_train_backward_is_persistent", "sscvae_debug_bptt_tiling",
    "sscvae_packed_bytes", "sscvae_pack_weights", "sscvae_test_gemm_splitk", "sscvae_sgd_step_multi", "sscvae_train_workspace_bytes", "sscvae_train_forward",
    "sscvae_train_backward", "sscvae_train_region", "sscvae_fsm_pack", "sscvae_fsm_build", "sscvae_select_best_beam", "sscvae_search_first_step",
    "sscvae_search_step", "sscvae_search_scratch_bytes", "sscvae_search_finish",
    "sscvae_decode_workspace_bytes", "sscvae_decode", "sscvae_decode_region", "sscvae_decode_samples_workspace_bytes",
    "sscvae_decode_samples", "sscvae_decode_samples_search_workspace_bytes", "sscvae_decode_samples_search",
    "sscvae_decode_samples_search_region", "sscvae_grad_sqnorm", "sscvae_sgd_step", "sscvae_test_gemm",
    "sscvae_profile_enable", "sscvae_profile_report", "sscvae_test_gemm_grouped", "sscvae_test_transpose_bf16",
    "sscvae_sgd_step_packed", "sscvae_debug_sgd_pack_jobs", "sscvae_decode_attention",
    "sscvae_decode_step_workspace_bytes", "sscvae_decode_step",
    "sscvae_train_step_image_state_bytes", "sscvae_train_step_tape_bytes", "sscvae_train_step_workspace_bytes",
    "sscvae_train_step_image_state", "sscvae_train_step_forward", "sscvae_train_step_backward",
]


class SscvaeDims(C.Structure):
    _fields_ = [
        ("image_feature_size", C.c_int32), ("embedding_size", C.c_int32), ("hidden_size", C.c_int32),
        ("attention_projection_size", C.c_int32), ("z_space", C.c_int32), ("vocab_size", C.c_int32),
        ("max_caption_length", C.c_int32), ("sentiment_vae", C.c_int32), ("simple_vae", C.c_int32),
        ("tied_embedding", C.c_int32), ("pad_index", C.c_int32), ("boundary_index", C.c_int32),
        ("prior_std", C.c_float), ("senti_prior_multip", C.c_float), ("latent_embedding", C.c_int32),
    ]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C style-seqcvae_b200/csrc`). There is no CPU / PyTorch fallback for this path.")
    L = C.CDLL(LIB_PATH)
    vp, i32, u64, sz, f32 = C.c_void_p, C.c_int, C.c_uint64, C.c_size_t, C.c_float
    L.sscvae_abi_version.restype = C.c_int
    L.sscvae_last_error.restype = C.c_char_p
    L.sscvae_launch_count.restype = u64
    L.sscvae_create.argtypes = [C.POINTER(SscvaeDims), C.POINTER(vp)]
    L.sscvae_destroy.argtypes = [vp]
    L.sscvae_destroy.restype = None
    L.sscvae_packed_bytes.argtypes = [vp]
    L.sscvae_packed_bytes.restype = sz
    L.sscvae_pack_weights.argtypes = [vp, C.POINTER(vp), vp, sz, C.POINTER(C.c_uint8), vp]
    L.sscvae_train_workspace_bytes.argtypes = [vp, i32, i32]
    L.sscvae_train_workspace_bytes.restype = sz
    L.sscvae_train_forward.argtypes = [vp, i32, i32, vp, C.POINTER(vp), vp, vp, vp, vp, vp, u64, vp, sz, vp, vp, vp]
    L.sscvae_train_backward.argtypes = [vp, i32, i32, vp, C.POINTER(vp), vp, sz, vp, vp, C.POINTER(vp), C.POINTER(vp), vp]
    L.sscvae_train_region.argtypes = [vp, i32, i32, C.c_char_p, C.POINTER(sz), C.POINTER(sz)]
    L.sscvae_fsm_pack.argtypes = [vp, i32, i32, i32, vp, vp]
    L.sscvae_fsm_build.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, vp]
    L.sscvae_select_best_beam.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp, vp]
    L.sscvae_search_first_step.argtypes = [vp, i32, i32, i32, i32, vp, i32, vp, vp, vp]
    L.sscvae_search_scratch_bytes.argtypes = [i32, i32, i32, i32]
    L.sscvae_search_scratch_bytes.restype = sz
    L.sscvae_search_step.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, i32, vp, vp, vp, sz, vp, vp, vp, vp]
    L.sscvae_search_finish.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, vp, vp, vp]
    L.sscvae_decode_workspace_bytes.argtypes = [vp, i32, i32, i32, i32]
    L.sscvae_decode_workspace_bytes.restype = sz
    L.sscvae_decode_region.argtypes = [vp, i32, i32, i32, i32, C.c_char_p, C.POINTER(sz), C.POINTER(sz)]
    L.sscvae_decode.argtypes = [vp, i32, i32, i32, i32, i32, vp, C.POINTER(vp), vp, vp, vp, vp, vp, i32, vp, u64, vp, sz,
                                vp, vp, vp, vp, vp]
    L.sscvae_decode_samples_workspace_bytes.argtypes = [vp, i32, i32, i32]
    L.sscvae_decode_samples_workspace_bytes.restype = sz
    L.sscvae_decode_samples.argtypes = [vp, i32, i32, i32, vp, C.POINTER(vp), vp, vp, vp, vp, u64, vp, sz, vp, vp, vp, vp]
    L.sscvae_decode_samples_search_workspace_bytes.argtypes = [vp, i32, i32, i32, i32, i32, i32]
    L.sscvae_decode_samples_search_workspace_bytes.restype = sz
    L.sscvae_decode_samples_search.argtypes = [vp, i32, i32, i32, i32, i32, i32, vp, C.POINTER(vp), vp, vp, vp, vp, i32, vp, i32,
                                               vp, u64, vp, sz, vp, vp, vp, vp, vp]
    L.sscvae_decode_attention.argtypes = [vp, vp, sz, vp, vp, vp, vp]
    L.sscvae_decode_step_workspace_bytes.argtypes = [vp, i32, i32, i32]
    L.sscvae_decode_step_workspace_bytes.restype = sz
    L.sscvae_decode_step.argtypes = [vp, i32, i32, i32, vp, C.POINTER(vp), vp, vp, vp, vp, vp, vp, C.POINTER(vp), vp, u64,
                                     vp, sz, vp, C.POINTER(vp), vp, vp, vp]
    for name in ("sscvae_train_step_image_state_bytes", "sscvae_train_step_tape_bytes", "sscvae_train_step_workspace_bytes"):
        getattr(L, name).argtypes = [vp, i32, i32]
        getattr(L, name).restype = sz
    L.sscvae_train_step_image_state.argtypes = [vp, i32, i32, vp, C.POINTER(vp), vp, vp, vp, sz, vp]
    L.sscvae_train_step_forward.argtypes = [vp, i32, i32, vp, C.POINTER(vp), vp, sz, vp, vp, C.POINTER(vp), vp, u64, vp, sz,
                                            vp, sz, vp, C.POINTER(vp), vp, vp, vp, vp, vp]
    L.sscvae_train_step_backward.argtypes = [vp, i32, i32, vp, C.POINTER(vp), vp, sz, vp, sz, vp, sz, vp, C.POINTER(vp), vp,
                                             vp, vp, vp, C.POINTER(vp), C.POINTER(vp), vp]
    L.sscvae_decode_samples_search_region.argtypes = [vp, i32, i32, i32, i32, i32, i32, C.c_char_p, C.POINTER(sz), C.POINTER(sz)]
    L.sscvae_test_gemm_splitk.argtypes = [vp, i32, vp, i32, i32, i32, i32, vp, i32, i32, vp, vp]
    L.sscvae_sgd_step_multi.argtypes = [i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(u64), C.POINTER(i32),
                                        C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, vp, sz, vp]
    L.sscvae_sgd_step_packed.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(i32), i32,
                                         C.POINTER(i32), f32, f32, f32, f32, f32, vp, sz, vp, sz, vp]
    L.sscvae_debug_sgd_pack_jobs.argtypes = [vp, C.POINTER(C.c_int64), i32]
    L.sscvae_grad_sqnorm.argtypes = [vp, sz, vp, vp, vp]
    L.sscvae_sgd_step.argtypes = [vp, vp, vp, sz, vp, f32, f32, f32, f32, i32, vp]
    L.sscvae_test_gemm.argtypes = [vp, i32, vp, i32, i32, i32, i32, vp, i32, vp, i32, i32, vp]
    L.sscvae_test_gemm_grouped.argtypes = [i32, C.POINTER(vp), C.POINTER(i32), C.POINTER(vp), C.POINTER(i32),
                                           C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(vp), C.POINTER(i32), vp]
    L.sscvae_test_transpose_bf16.argtypes = [i32, C.POINTER(vp), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32),
                                             C.POINTER(vp), C.POINTER(i32), vp]
    L.sscvae_set_option.argtypes = [vp, C.c_char_p, i32]
    L.sscvae_train_backward_is_persistent.argtypes = [vp, i32, i32]
    L.sscvae_debug_bptt_tiling.argtypes = [vp, i32, i32, i32, C.POINTER(i32)]
    L.sscvae_profile_enable.argtypes = [i32]
    L.sscvae_profile_report.argtypes = [C.c_char_p, sz]
    for name in SYMBOLS:
        fn = getattr(L, name)
        if fn.restype is C.c_int and name not in ("sscvae_abi_version",):
            fn.restype = C.c_int
    if L.sscvae_abi_version() != 6:
        raise ImportError("libsscvae_b200.so ABI version mismatch")
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        msg = lib().sscvae_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libsscvae_b200 error {rc}: {msg}")


def ptr(t):
    """Device (or host) address of a tensor, or NULL."""
    return C.c_void_p(0 if t is None else t.data_ptr())


def ptr_array(tensors):
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = 0 if t is None else t.data_ptr()
    return arr


def profile(on: bool):
    check(lib().sscvae_profile_enable(int(on)))


def profile_report() -> dict:
    import json
    buf = C.create_string_buffer(1 << 16)
    check(lib().sscvae_profile_report(buf, len(buf)))
    return json.loads(buf.value.decode())


def launch_count() -> int:
    return int(lib().sscvae_launch_count())
