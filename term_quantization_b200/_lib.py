"""ctypes binding of libtq_b200.so (C ABI declared in include/tq_b200.h).

There is no fallback of any kind: if the shared library is missing or a call fails this
module raises.  PyTorch is used only for device memory and the current stream.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# TQ_B200_LIB: another build of the same C ABI (the instrumented debug build of tools/conv_trace.sh)
LIB_PATH = os.environ.get("TQ_B200_LIB") or os.path.join(_HERE, "libtq_b200.so")

TQ_OK, TQ_ERR_INVALID, TQ_ERR_UNSUPPORTED, TQ_ERR_CUDA = 0, 1, 2, 3
TQ_F32, TQ_F64, TQ_BF16, TQ_F16 = 0, 1, 2, 3
TQ_I8, TQ_I16, TQ_I32, TQ_U8, TQ_F16C = 0, 1, 2, 3, 4
ENC_HESE, ENC_BINARY, ENC_BOOTH = 0, 1, 2
ENCODINGS = {"hese": ENC_HESE, "binary": ENC_BINARY, "booth": ENC_BOOTH}


def encoding_id(encoding):
    """TQ_ENC_* value of a term encoding name; ValueError for anything else."""
    if not isinstance(encoding, str) or encoding not in ENCODINGS:
        raise ValueError(f"unknown term encoding {encoding!r}: expected one of {', '.join(ENCODINGS)}")
    return ENCODINGS[encoding]

FLAG_RELU, FLAG_RECIP_DIV, FLAG_EXACT_DIV = 1, 2, 4

# every symbol include/tq_b200.h declares: (restype, argtypes)
_i64, _i, _f, _p, _u = C.c_int64, C.c_int, C.c_float, C.c_void_p, C.c_uint
SYMBOLS = {
    "tq_version": (_i, []),
    "tq_last_error": (C.c_char_p, []),
    "tq_launch_count": (C.c_uint64, []),
    "tq_tr_encode": (_i, [_p, _p, _i, _i64, _i64, _i64, _f, _i, _i, _i, _i, _u, _p]),
    "tq_tr_encode_codes": (_i, [_p, _p, _i, _i, _i64, _i64, _i64, _f, _i, _i, _i, _i, _u, _p, _p]),
    "tq_hist_accumulate": (_i, [_p, _i, _i64, _p, _p, _i, _f, _f, _p]),
    "tq_mse_profile": (_i, [_p, _p, _i, _p, _i, _i, _i, _p, _p, _p]),
    "tq_mse_profile_enc": (_i, [_p, _p, _i, _p, _i, _i, _i, _i, _p, _p, _p]),
    "tq_hese_term_count": (_i, [_p, _i, _i64, _f, _u, _p, _p]),
    "tq_term_count": (_i, [_p, _i, _i64, _f, _i, _u, _p, _p]),
    "tq_conv2d_codes_f16": (_i, [_p, _p, _p, _p] + [_i] * 9 + [_f, _i, _p]),
    "tq_conv2d_codes_fused": (_i, [_p] * 8 + [_i] * 9 + [_f, _i, _f, _i, _i, _i, _p]),
    "tq_conv2d_codes_fused_enc": (_i, [_p] * 8 + [_i] * 9 + [_f, _i, _f, _i, _i, _i, _i, _p]),
    "tq_conv2d_planes_i8": (_i, [_p, _p, _i, _i] + [_p] * 6 + [_i] * 9 + [_f, _i, _f, _i, _i, _i, _i, _p]),
    "tq_conv2d_planes_i8_enc": (_i, [_p, _p, _i, _i] + [_p] * 6 + [_i] * 9 + [_f, _i, _f, _i, _i, _i, _i, _i, _p]),
    "tq_codes_to_planes": (_i, [_p, _p, _i64, _i, _p, _p]),
    "tq_conv_weight_l1": (_i, [_p, _i, _i, _i, _p, _p, _p]),
    "tq_depthwise3x3_codes": (_i, [_p] * 7 + [_i] * 5 + [_f, _i, _i, _f, _i, _i, _p]),
    "tq_depthwise3x3_codes_enc": (_i, [_p] * 7 + [_i] * 5 + [_f, _i, _i, _f, _i, _i, _i, _p]),
    "tq_bn_act_encode": (_i, [_p] * 6 + [_i64, _i, _i, _f, _i, _i, _p]),
    "tq_bn_act_encode_enc": (_i, [_p] * 6 + [_i64, _i, _i, _f, _i, _i, _i, _p]),
    "tq_maxpool2d_f16": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _i, _p]),
    "tq_first_conv3x3_fused": (_i, [_p] * 7 + [_i, _i, _i, _i, _i, _i, _f, _i, _i, _p]),
    "tq_first_conv3x3_fused_enc": (_i, [_p] * 7 + [_i, _i, _i, _i, _i, _i, _f, _i, _i, _i, _p]),
    "tq_u8_normalize_bf16": (_i, [_p, _p, _i64, _p, _p, _p]),
    "tq_bn_relu_maxpool_encode": (_i, [_p] * 5 + [_i] * 5 + [_f, _i, _i, _p]),
    "tq_bn_relu_maxpool_encode_enc": (_i, [_p] * 5 + [_i] * 5 + [_f, _i, _i, _i, _p]),
    "tq_stem_conv7x7s2": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "tq_stem_conv7x7s2_dt": (_i, [_p, _i, _p, _p, _p, _i, _i, _i, _i, _p]),
    "tq_stem_conv7x7s2_u8": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "tq_stem_conv7x7s2_pool": (_i, [_p, _i, _p, _p, _p, _p, _i, _p, _p, _i, _i, _i, _i, _f, _i, _i, _p]),
    "tq_stem_conv7x7s2_pool_enc": (_i, [_p, _i, _p, _p, _p, _p, _i, _p, _p, _i, _i, _i, _i, _f, _i, _i, _i, _p]),
    "tq_stem_conv7x7s2_rowmax": (_i, [_p, _i, _p, _p, _p, _i, _i, _i, _i, _p]),
    "tq_stem_conv7x7s2_u8_rowmax": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "tq_bn_relu_maxpool_encode_rowmax": (_i, [_p] * 5 + [_i] * 5 + [_f, _i, _i, _p]),
    "tq_bn_relu_maxpool_encode_rowmax_enc": (_i, [_p] * 5 + [_i] * 5 + [_f, _i, _i, _i, _p]),
    "tq_lstm_recurrence": (_i, [_p] * 8 + [_i, _i, _i, _p]),
    "tq_gru_recurrence": (_i, [_p] * 6 + [_i, _i, _i, _p]),
    "tq_rnn_recurrence": (_i, [_p] * 6 + [_i, _i, _i, _i, _p]),
    "tq_recurrence_max_hidden": (_i, [_i]),
    "tq_log_softmax_nll": (_i, [_p, _i64, _i64, _i64, _p, _p, _p]),
    "tq_linear_nll_workspace_bytes": (_i64, [_i64, _i64]),
    "tq_linear_codes_nll": (_i, [_p, _p, _i64, _i, _i, _i, _f, _p, _i, _p, _p, _p, _i64, _p]),
    "tq_linear_planes_i8_nll": (_i, [_p, _p, _i, _i, _i64, _i, _i, _i, _f, _p, _i, _i, _p, _p, _p, _i64, _p]),
    "tq_selftest_division": (_i, [C.c_uint64, C.c_uint32, _p, _p]),
}

_lib = None


class TQError(RuntimeError):
    pass


def build(verbose=False):
    """Compile libtq_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    import subprocess
    subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), "-j4", "--no-print-directory"],
                   check=True, stdout=None if verbose else subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TQError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` or `make -C term_quantization_b200/csrc`. There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)          # AttributeError if the ABI lost a symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != TQ_OK:
        msg = lib().tq_last_error().decode("utf-8", "replace")
        if rc == TQ_ERR_INVALID:
            raise ValueError(f"tq_b200: {msg}")
        if rc == TQ_ERR_UNSUPPORTED:
            raise NotImplementedError(f"tq_b200: {msg}")
        raise TQError(f"tq_b200: {msg}")


def launch_count():
    return int(lib().tq_launch_count())
