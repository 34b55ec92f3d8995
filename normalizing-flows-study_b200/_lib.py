"""ctypes binding of libnfb200.so (the C ABI declared in include/nfb200.h).

PyTorch is used for device memory and streams only: every call passes raw
`tensor.data_ptr()` device pointers, sizes and the current CUDA stream handle.
There is no CPU path: if the shared library is missing or a tensor is not on
a CUDA device the call raises.
"""
from __future__ import annotations

import ctypes
import os

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NFB200_LIB") or os.path.join(_PKG, "lib", "libnfb200.so")   # override: debug builds

NF_F32, NF_F64 = 0, 1
NF_ERR_UNSUPPORTED = -2
AR_MAF_INVERSE, AR_IAF_FORWARD, AR_MAF_FORWARD, AR_IAF_INVERSE = 0, 1, 2, 3

_c = ctypes
_P, _I, _L, _D, _U = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_double, _c.c_uint64

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/nfb200.h one to one
_SIGNATURES = {
    "nf_abi_version": [],
    "nf_status_string": [_I],
    "nf_last_cuda_error": [],
    "nf_launch_count": [],
    "nf_set_option": [_I, _I],
    "nf_rqs_unit_forward": [_P, _P, _P, _P, _P, _P, _L, _I, _I, _D, _D, _D, _I, _P],
    "nf_rqs_unit_backward": [_P] * 10 + [_L, _I, _I, _D, _D, _D, _I, _P],
    "nf_spline_transform_forward": [_P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _I, _D, _D, _D, _D, _P, _P, _P, _I, _I, _P],
    "nf_spline_transform_backward": [_P] * 8 + [_L, _I, _I, _I, _I, _D, _D, _D, _D, _P, _P, _P, _I, _I, _P],
    "nf_affine_coupling_forward": [_P] * 6 + [_L, _I, _I, _I, _P],
    "nf_affine_coupling_backward": [_P] * 9 + [_L, _I, _I, _I, _P],
    "nf_affine_ar_forward": [_P] * 4 + [_L, _I, _I, _I, _P],
    "nf_affine_ar_backward": [_P] * 7 + [_L, _I, _I, _I, _P],
    "nf_gemm": [_P, _P, _P, _P, _L, _L, _L, _L, _L, _L, _L, _L, _I, _I, _P, _I, _P],
    "nf_mul_rows": [_P, _P, _P, _L, _L, _L, _I, _P],
    "nf_relu_backward": [_P, _P, _P, _L, _I, _P],
    "nf_relu_backward_colsum": [_P, _P, _P, _P, _L, _L, _I, _P],
    "nf_col_sum": [_P, _P, _L, _L, _I, _P],
    "nf_batchnorm_forward": [_P] * 9 + [_L, _I, _I, _D, _D, _I, _I, _P],
    "nf_batchnorm_backward": [_P] * 10 + [_L, _I, _I, _I, _I, _P, _P],
    "nf_spline_stack_forward": [_P, _P, _L, _P, _P, _P, _L, _I, _P],
    "nf_coupling_stack_forward": [_P, _P, _L, _P, _P, _P, _L, _I, _P],
    "nf_spline_stack_packed_floats": [_I, _I, _I, _I],
    "nf_coupling_stack_packed_floats": [_I, _I, _I],
    "nf_made_affine_forward": [_P] * 9 + [_P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _I, _P],
    "nf_ar_sequential_forward": [_P] * 9 + [_P, _P, _P, _L, _I, _I, _I, _P],
    "nf_feature_affine_forward": [_P] * 5 + [_D, _P, _L, _I, _I, _P],
    "nf_feature_affine_backward": [_P] * 11 + [_L, _I, _I, _P],
    "nf_col_stats": [_P] * 4 + [_L, _I, _I, _P],
    "nf_ar_step_forward": [_P] * 6 + [_L, _I, _I, _I, _I, _P],
    "nf_ar_step_backward": [_P] * 7 + [_L, _I, _I, _I, _I, _P],
    "nf_ar_finish_forward": [_P] * 5 + [_L, _I, _I, _I, _P],
    "nf_ar_finish_backward": [_P] * 7 + [_L, _I, _I, _I, _P],
    "nf_std_normal_log_prob_forward": [_P] * 3 + [_L, _I, _I, _P],
    "nf_std_normal_log_prob_backward": [_P] * 3 + [_L, _I, _I, _P],
    "nf_std_normal_draw": [_U, _U, _P, _L, _I, _I, _P],
    "nf_std_normal_log_q_forward": [_P] * 3 + [_L, _I, _I, _P],
    "nf_std_normal_log_q_backward": [_P] * 4 + [_L, _I, _I, _P],
    "nf_spline_stack_sample": [_P, _P, _L, _U, _U, _P, _P, _L, _P],
    "nf_spline_stack_tc_sample": [_P, _P, _L, _U, _U, _P, _P, _L, _P],
    "nf_coupling_stack_sample": [_P, _P, _L, _U, _U, _P, _P, _L, _P],
    "nf_coupling_stack_tc_sample": [_P, _P, _L, _U, _U, _P, _P, _L, _P],
    "nf_made_stack_tc_sample": [_P, _P, _L, _I, _U, _U, _P, _P, _L, _P],
    "nf_std_normal_draw_state": [_P, _P, _L, _I, _I, _P],
    "nf_spline_stack_sample_state": [_P, _P, _L, _P, _P, _P, _L, _P],
    "nf_spline_stack_tc_sample_state": [_P, _P, _L, _P, _P, _P, _L, _P],
    "nf_coupling_stack_sample_state": [_P, _P, _L, _P, _P, _P, _L, _P],
    "nf_coupling_stack_tc_sample_state": [_P, _P, _L, _P, _P, _P, _L, _P],
    "nf_made_stack_tc_sample_state": [_P, _P, _L, _I, _P, _P, _P, _L, _P],
    "nf_debug_tc_gemm128": [_P, _P, _P, _I, _I, _P, _I, _P],
    "nf_linear_tc": [_P, _P, _P, _P, _P, _L, _L, _L, _L, _L, _L, _I, _P, _P],
    "nf_linear_tc_range": [_P, _P, _P, _P, _P, _L, _L, _L, _L, _L, _L, _I, _P, _P, _P],
    "nf_split_tf32": [_P, _P, _P, _L, _P],
    "nf_linear_wgrad_tc_workspace": [_L, _L, _L],
    "nf_linear_wgrad_tc": [_P, _P, _P, _L, _L, _L, _L, _L, _L, _P, _L, _P],
    "nf_linear_wgrad_tc_masked": [_P, _P, _P, _L, _L, _L, _L, _L, _L, _P, _L, _P, _P],
    "nf_arqs_step_forward": [_P, _P, _P, _L, _P, _P, _P, _L, _I, _I, _I, _I, _D, _D, _D, _I, _P],
    "nf_arqs_step_backward": [_P, _P, _L, _P, _P, _P, _P, _P, _L, _I, _I, _I, _I, _D, _D, _D, _I, _P],
    "nf_ar_blocked_forward": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _I, _I, _I, _P],
    "nf_ar_blocked_workspace_floats": [_L, _I, _I],
    "nf_spline_stack_tc_forward": [_P, _P, _L, _P, _P, _P, _L, _I, _P],
    "nf_spline_stack_tc_block_words": [_I, _I, _I],
    "nf_coupling_stack_tc_forward": [_P, _P, _L, _P, _P, _P, _L, _I, _P],
    "nf_coupling_stack_tc_block_words": [_I],
    "nf_coupling_stack_tc_block_words_hidden": [_I, _I],
    "nf_made_stack_tc_forward": [_P, _P, _L, _P, _P, _P, _L, _I, _I, _P],
    "nf_made_stack_tc_block_words": [_I],
    "nf_spline_stack_ctx_tc_forward": [_P, _P, _L, _P, _P, _L, _L, _P, _P, _L, _I, _P],
    "nf_spline_stack_ctx_tc_sample": [_P, _P, _L, _P, _L, _L, _U, _U, _P, _P, _L, _P],
    "nf_spline_stack_ctx_tc_sample_state": [_P, _P, _L, _P, _L, _L, _P, _P, _P, _L, _P],
    "nf_coupling_stack_ctx_tc_forward": [_P, _P, _L, _P, _P, _L, _L, _P, _P, _L, _I, _P],
    "nf_coupling_stack_ctx_tc_sample": [_P, _P, _L, _P, _L, _L, _U, _U, _P, _P, _L, _P],
    "nf_coupling_stack_ctx_tc_sample_state": [_P, _P, _L, _P, _L, _L, _P, _P, _P, _L, _P],
    "nf_coupling_stack_ctx_tc_block_words_hidden": [_I, _I],
    "nf_made_chain_bf16_forward": [_P] * 9 + [_P, _P, _P, _L, _I, _I, _I, _I, _P],
    "nf_batchnorm_forward_staged": [_P] * 9 + [_L, _I, _D, _D, _I, _I, _L, _I, _P],
    "nf_batchnorm_backward_staged": [_P] * 10 + [_L, _I, _I, _I, _L, _I, _P, _P],
}
_RESTYPES = {
    "nf_status_string": _c.c_char_p,
    "nf_last_cuda_error": _c.c_char_p,
    "nf_launch_count": _L,
    "nf_spline_stack_packed_floats": _L,
    "nf_coupling_stack_packed_floats": _L,
    "nf_spline_stack_tc_block_words": _L,
    "nf_ar_blocked_workspace_floats": _L,
    "nf_coupling_stack_tc_block_words": _L,
    "nf_coupling_stack_tc_block_words_hidden": _L,
    "nf_coupling_stack_ctx_tc_block_words_hidden": _L,
    "nf_made_stack_tc_block_words": _L,
    "nf_linear_wgrad_tc_workspace": _L,
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


class NfError(RuntimeError):
    def __init__(self, fn, status):
        self.status = status
        l = lib()
        msg = l.nf_status_string(status).decode()
        if status == -4:
            msg += ": " + l.nf_last_cuda_error().decode()
        super().__init__(f"{fn} failed: {msg} (status {status})")


def lib():
    """Load the shared library once.  Raises if it has not been built (python __graft_entry__.py / build.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python normalizing-flows-study_b200/build.py` "
                "(there is no CPU or PyTorch fallback for the flow kernels)")
        l = ctypes.CDLL(LIB_PATH)
        for name, args in _SIGNATURES.items():
            fn = getattr(l, name)
            fn.argtypes = args
            fn.restype = _RESTYPES.get(name, _I)
        if l.nf_abi_version() != 1:
            raise RuntimeError("libnfb200.so ABI version mismatch")
        # A/B knob for measurement scripts: NFB200_OPTIONS="key:value,..." -> nf_set_option(key, value) at load time
        for kv in filter(None, os.environ.get("NFB200_OPTIONS", "").split(",")):
            try:
                k, v = (int(t) for t in kv.split(":"))
            except ValueError:
                raise RuntimeError(f"NFB200_OPTIONS: expected 'key:value' integers, got {kv!r}") from None
            if l.nf_set_option(k, v) != 0:
                raise RuntimeError(f"NFB200_OPTIONS: nf_set_option({k}, {v}) was refused")
        _lib = l
    return _lib


def launch_count() -> int:
    return int(lib().nf_launch_count())


def dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return NF_F32
    if t.dtype == torch.float64:
        return NF_F64
    raise TypeError(f"libnfb200 computes in float32/float64, got {t.dtype}")


NO_CPU_PATH = "libnfb200 has no CPU path: tensors (and modules) must live on a CUDA device"


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError(NO_CPU_PATH)
    if not t.is_contiguous():
        raise RuntimeError("internal error: non-contiguous tensor passed to libnfb200")
    return t.data_ptr()


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_get_device = getattr(torch._C, "_cuda_getDevice", None)


def stream():
    """cudaStream_t of torch's current stream on the current device.  torch.cuda.current_stream() builds a Python
    Stream object through several layers (measured: a quarter of the host time of a 510-launch training step); the
    raw-handle accessor is ~30x cheaper."""
    if _raw_stream is not None and _get_device is not None:
        return _raw_stream(_get_device())
    return torch.cuda.current_stream().cuda_stream


def call(name, *args):
    """Invoke a status-returning C-ABI function; raise NfError on failure. Returns the status (0)."""
    rc = getattr(lib(), name)(*args)
    if rc != 0:
        raise NfError(name, rc)
    return rc


def try_call(name, *args):
    """Like call(), but returns False on NF_ERR_UNSUPPORTED (caller picks the layer-wise kernels instead)."""
    rc = getattr(lib(), name)(*args)
    if rc == NF_ERR_UNSUPPORTED:
        return False
    if rc != 0:
        raise NfError(name, rc)
    return True
