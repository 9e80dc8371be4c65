"""Drop-in for the reference extension module ``tr_cuda`` (kernels/tr_cuda.cpp:20-28).

    tr(input, sf, bitwidth, group_size, num_keep_terms) -> Tensor

Same positional signature, same preconditions and messages (CUDA + contiguous,
kernels/tr_cuda.cpp:12-18), same result bit for bit; runs on the current device and the
current stream (the reference uses the legacy default stream, kernels/tr_cuda_kernel.cu:147).
Extra keyword-only arguments are additions: ``encoding`` ('hese' | 'binary' | 'booth'),
``relu`` (fused clamp) and ``out`` (write into an existing tensor, may be ``input``).
``tr_codes`` returns the signed integer codes instead of the dequantised values.
"""
import torch

from . import _lib

_DTYPES = {torch.float32: _lib.TQ_F32, torch.float64: _lib.TQ_F64,
           torch.bfloat16: _lib.TQ_BF16, torch.float16: _lib.TQ_F16}
_CODE_DTYPES = {torch.int8: _lib.TQ_I8, torch.int16: _lib.TQ_I16, torch.int32: _lib.TQ_I32,
                torch.uint8: _lib.TQ_U8, torch.float16: _lib.TQ_F16C}
_ENCODINGS = {**_lib.ENCODINGS, 0: 0, 1: 1, 2: 2}


def _check_input(input):
    # kernels/tr_cuda.cpp:12-18 (AT_ASSERTM -> RuntimeError with these messages)
    if not input.is_cuda:
        raise RuntimeError("input must be a CUDA tensor")
    if not input.is_contiguous():
        raise RuntimeError("input must be contiguous")
    if input.dtype not in _DTYPES:
        raise RuntimeError(f'"tr_cuda" not implemented for \'{input.dtype}\'')


def _dims(input):
    # kernels/tr_cuda_kernel.cu:133-141: B = size(0), C = size(1), W,H = size(2),size(3) if 4-D.
    # (The reference ignores trailing dims of 3-D / 5-D inputs, which leaves most of the output
    # zero; here every trailing dim is part of the per-channel plane.)
    if input.dim() < 2:
        raise RuntimeError("tr expects a tensor with at least 2 dimensions (B, C, ...)")
    B, Cc = input.shape[0], input.shape[1]
    WH = 1
    for d in input.shape[2:]:
        WH *= d
    return B, Cc, WH


def _stream_ptr(device):
    return torch.cuda.current_stream(device).cuda_stream


def tr(input, sf, bitwidth, group_size, num_keep_terms, *, encoding="hese", relu=False, out=None,
       _exact_div=False):
    """Term Revealing (TR) (CUDA)"""
    _check_input(input)
    B, Cc, WH = _dims(input)
    if out is None:
        out = torch.empty_like(input)
    elif out.shape != input.shape or out.dtype != input.dtype or out.device != input.device \
            or not out.is_contiguous():
        raise RuntimeError("out must match input in shape, dtype, device and be contiguous")
    with torch.cuda.device(input.device):
        rc = _lib.lib().tq_tr_encode(input.data_ptr(), out.data_ptr(), _DTYPES[input.dtype],
                                     B, Cc, WH, float(sf), int(bitwidth), int(group_size),
                                     int(num_keep_terms), _ENCODINGS[encoding],
                                     (_lib.FLAG_RELU if relu else 0) |
                                     (_lib.FLAG_EXACT_DIV if _exact_div else 0),
                                     _stream_ptr(input.device))
    _lib.check(rc)
    return out


def tr_codes(input, sf, bitwidth, group_size, num_keep_terms, *, dtype=torch.int16,
             encoding="hese", relu=False, out=None, overflow=None):
    """Signed integer codes sign(x) * sum(kept terms) -- the operands of the integer
    conv/linear.  ``overflow`` (int32 CUDA scalar) is set to 1 if a code did not fit."""
    _check_input(input)
    if input.dtype not in (torch.float32, torch.bfloat16):
        raise NotImplementedError("integer codes are produced from float32 or bfloat16 inputs")
    B, Cc, WH = _dims(input)
    if out is None:
        out = torch.empty(input.shape, dtype=dtype, device=input.device)
    elif out.shape != input.shape or out.dtype not in _CODE_DTYPES or out.device != input.device \
            or not out.is_contiguous():
        raise RuntimeError("out must match input in shape and device, hold a code dtype and be contiguous")
    if overflow is not None and (overflow.dtype != torch.int32 or overflow.device != input.device):
        raise RuntimeError("overflow must be an int32 tensor on the input's device")
    with torch.cuda.device(input.device):
        rc = _lib.lib().tq_tr_encode_codes(
            input.data_ptr(), out.data_ptr(), _DTYPES[input.dtype], _CODE_DTYPES[out.dtype],
            B, Cc, WH, float(sf), int(bitwidth), int(group_size), int(num_keep_terms),
            _ENCODINGS[encoding], _lib.FLAG_RELU if relu else 0,
            overflow.data_ptr() if overflow is not None else None, _stream_ptr(input.device))
    _lib.check(rc)
    return out


_PYBIND = None


def pybind():
    """The compiled torch extension with the reference's exact module surface (`tr(input, sf, bitwidth,
    group_size, num_keep_terms)`, kernels/tr_cuda.cpp:20-28), built ahead of time from csrc/pybind/tr_cuda_pybind.cpp
    by `__graft_entry__.build()`; it calls the same C ABI as this module.  Raises if it has not been built."""
    global _PYBIND
    if _PYBIND is None:
        import importlib.util
        import os
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tr_cuda_pybind.so")
        if not os.path.exists(path):
            raise _lib.TQError(f"{path} is missing: run `python term_quantization_b200/csrc/pybind/build.py`")
        _lib.lib()                                   # libtq_b200.so first (the adapter links against it)
        spec = importlib.util.spec_from_file_location("tr_cuda_pybind", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        _PYBIND = mod
    return _PYBIND
