"""ctypes binding of the C-ABI library (include/genvox_b200.h).  No torch types cross the boundary:
only raw device pointers, sizes and a cudaStream_t.  There is no fallback: if the library is missing
or a call fails, a RuntimeError is raised."""
import ctypes as C
import os

from . import build as _build

_P = C.c_void_p


class GvxDims(C.Structure):
    _fields_ = [("n_mels", C.c_int32), ("enc_dim", C.c_int32), ("att_rnn_dim", C.c_int32), ("dec_rnn_dim", C.c_int32),
                ("prenet_dim", C.c_int32), ("att_dim", C.c_int32), ("loc_filters", C.c_int32), ("loc_kernel", C.c_int32),
                ("p_att_dropout", C.c_float), ("p_dec_dropout", C.c_float), ("precision", C.c_int32)]


# order == struct gvx_weights / gvx_grads; values are the reference's state_dict keys (SURVEY.md §8b)
PARAM_FIELDS = [
    ("prenet_w0", "prenet.layers.0.linear_layer.weight"),
    ("prenet_w1", "prenet.layers.1.linear_layer.weight"),
    ("att_w_ih", "attention_rnn.weight_ih"),
    ("att_w_hh", "attention_rnn.weight_hh"),
    ("att_b_ih", "attention_rnn.bias_ih"),
    ("att_b_hh", "attention_rnn.bias_hh"),
    ("query_w", "attention_layer.query_layer.linear_layer.weight"),
    ("memory_w", "attention_layer.memory_layer.linear_layer.weight"),
    ("v_w", "attention_layer.v.linear_layer.weight"),
    ("loc_conv_w", "attention_layer.location_layer.location_conv.conv.weight"),
    ("loc_dense_w", "attention_layer.location_layer.location_dense.linear_layer.weight"),
    ("dec_w_ih", "decoder_rnn.weight_ih"),
    ("dec_w_hh", "decoder_rnn.weight_hh"),
    ("dec_b_ih", "decoder_rnn.bias_ih"),
    ("dec_b_hh", "decoder_rnn.bias_hh"),
    ("proj_w", "linear_projection.linear_layer.weight"),
    ("proj_b", "linear_projection.linear_layer.bias"),
    ("gate_w", "gate_layer.linear_layer.weight"),
    ("gate_b", "gate_layer.linear_layer.bias"),
]


class GvxWeights(C.Structure):
    _fields_ = [(f, _P) for f, _ in PARAM_FIELDS]


class GvxGrads(C.Structure):
    _fields_ = [(f, _P) for f, _ in PARAM_FIELDS]


class GvxSession(C.Structure):
    _fields_ = [("N", C.c_int32), ("slots", C.c_int32), ("capacity", C.c_int32), ("max_steps", C.c_int32),
                ("ignore_gate", C.c_int32), ("with_alignments", C.c_int32), ("row_offset", C.c_int32),
                ("gate_threshold", C.c_float), ("seed", C.c_uint64), ("steps_run", C.c_longlong), ("submitted", C.c_longlong),
                ("admitted", C.c_longlong), ("finished", C.c_longlong), ("active", C.c_int32), ("parity", C.c_int32),
                ("ready", C.c_int32)]


_SIGNATURES = {
    "gvx_abi_version": (C.c_int, []),
    "gvx_last_error": (C.c_char_p, []),
    "gvx_device_error": (C.c_int, [C.c_int]),
    "gvx_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "gvx_launch_count": (C.c_ulonglong, []),
    "gvx_profile_enable": (C.c_int, [C.c_int]),
    "gvx_profile_reset": (C.c_int, []),
    "gvx_profile_read": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "gvx_profile_slot_name": (C.c_char_p, [C.c_int]),
    "gvx_graph_stats": (C.c_int, [C.POINTER(C.c_ulonglong)]),
    "gvx_dec_packed_bytes": (C.c_size_t, [C.POINTER(GvxDims)]),
    "gvx_dec_pack_weights": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, _P]),
    "gvx_dec_stash_bytes": (C.c_size_t, [C.POINTER(GvxDims), C.c_int, C.c_int, C.c_int]),
    "gvx_dec_bwd_workspace_bytes": (C.c_size_t, [C.POINTER(GvxDims), C.c_int, C.c_int, C.c_int]),
    "gvx_dec_infer_workspace_bytes": (C.c_size_t, [C.POINTER(GvxDims), C.c_int, C.c_int, C.c_int]),
    "gvx_dec_train_fwd": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, _P, _P, _P, C.c_int, C.c_int, C.c_int,
                                    C.c_uint64, C.c_int, C.c_int, _P, _P, _P, _P, _P]),
    "gvx_dec_train_bwd": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, _P, _P, C.c_int, C.c_int, C.c_int,
                                    C.c_uint64, C.c_int, C.c_int, _P, _P, _P, _P, _P, C.POINTER(GvxGrads), _P, _P]),
    "gvx_dec_infer": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, _P, _P, C.c_int, C.c_int, C.c_int,
                                C.c_float, C.c_int, C.c_uint64, C.c_int, C.c_int, _P, _P, _P, _P, C.POINTER(C.c_int), _P, _P]),
    "gvx_dec_infer_windowed": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, _P, _P, C.c_int, C.c_int, C.c_int,
                                         C.c_float, C.c_int, C.c_uint64, C.c_int, C.c_int, _P, _P, _P, _P, C.POINTER(C.c_int),
                                         C.c_int, C.c_int, _P, _P]),
    "gvx_dec_infer_continuous_workspace_bytes": (C.c_size_t, [C.POINTER(GvxDims), C.c_int, C.c_int, C.c_int]),
    "gvx_dec_infer_continuous": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, _P, _P, C.c_int, C.c_int, C.c_int,
                                           C.c_int, _P, C.c_float, C.c_int, C.c_uint64, C.c_int, _P, _P, _P, _P,
                                           C.POINTER(C.c_longlong), _P, _P]),
    "gvx_dec_infer_continuous_windowed": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, _P, _P, C.c_int, C.c_int,
                                                    C.c_int, C.c_int, _P, C.c_float, C.c_int, C.c_uint64, C.c_int, _P, _P, _P,
                                                    _P, C.POINTER(C.c_longlong), C.c_int, C.c_int, _P, _P]),
    "gvx_dec_session_workspace_bytes": (C.c_size_t, [C.POINTER(GvxDims), C.c_int, C.c_int, C.c_int]),
    "gvx_dec_session_init": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxSession), _P, _P]),
    "gvx_dec_session_submit": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, C.POINTER(GvxSession), _P, _P, _P,
                                         C.c_int, _P, _P]),
    "gvx_dec_session_step": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, C.POINTER(GvxSession), C.c_int,
                                       _P, _P, _P, _P, _P, C.POINTER(C.c_int), _P, _P]),
    "gvx_dec_session_step_windowed": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, C.POINTER(GvxSession), C.c_int,
                                                _P, _P, _P, _P, _P, C.POINTER(C.c_int), C.c_int, C.c_int, _P, _P]),
    "gvx_test_tc_gemm": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "gvx_test_nt_gemm": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "gvx_bench_nt_gemm": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "gvx_test_lstm_chain": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_float, C.c_uint64, C.c_int, _P, _P, _P, _P, _P, _P]),
    "gvx_debug_timeline": (C.c_int, [_P]),
    "gvx_debug_option": (C.c_int, [C.c_char_p, C.c_int]),
    "gvx_prenet_fwd": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, C.c_int, C.c_int, C.c_uint64, C.c_int,
                                 C.c_int, _P, _P, _P]),
    "gvx_lstm_step": (C.c_int, [C.POINTER(GvxDims), _P, C.c_int, _P, _P, _P, C.c_int, C.c_uint64, C.c_int, C.c_int,
                                C.c_int, _P, _P, _P, _P]),
    "gvx_attention_step": (C.c_int, [C.POINTER(GvxDims), C.POINTER(GvxWeights), _P, _P, _P, _P, _P, C.c_int, C.c_int,
                                     _P, _P, _P, _P, _P, _P]),
}

EXPORTS = sorted(_SIGNATURES)
_lib = None


def library_path():
    return _build.LIB_PATH


def library_is_fresh():
    """True when the in-tree library was compiled from exactly the sources in the tree (fingerprint compiled into it)."""
    return _build.is_fresh()


def load():
    """Load (building first if the in-tree .so is absent or stale and nvcc is available).  A library that was NOT built
    from the sources in the tree is refused - kernels of other sources under this Python layer and these struct layouts
    would run silently - unless GVX_ALLOW_STALE_LIB=1 says that is intended."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if not _build.is_fresh():
        try:
            _build.build()
        except Exception as exc:
            if not os.path.isfile(path):
                raise RuntimeError(f"genvox_b200: CUDA library missing and could not be built: {exc}") from exc
            if os.environ.get("GVX_ALLOW_STALE_LIB") != "1":
                raise RuntimeError(f"genvox_b200: {path} was built from other sources and the rebuild failed ({exc}); "
                                   "set GVX_ALLOW_STALE_LIB=1 to load it anyway") from exc
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.gvx_abi_version() != 1:
        raise RuntimeError("genvox_b200: ABI version mismatch")
    _lib = lib
    return lib


def check_device_errors(clear=True):
    """Raise if a kernel of an earlier (asynchronous) call aborted on the device.  Meaningful after the stream has been
    synchronised (e.g. where the loss is read); training entry points also refuse to run once the latch is set."""
    code = load().gvx_device_error(1 if clear else 0)
    if code:
        raise RuntimeError(f"genvox_b200: a device kernel aborted (entry {code // 1000}, wait code {code % 1000}); "
                           "the outputs of that call are invalid")


def check(status, what):
    if status != 0:
        msg = load().gvx_last_error()
        raise RuntimeError(f"genvox_b200.{what} failed: {msg.decode() if msg else 'unknown error'}")
