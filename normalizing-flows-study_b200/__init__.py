"""B200-native (sm_100a) implementation of the normalizing-flow transform hot path of
itxtx/normalizing-flows-study, behind the reference's own nn.Module API.

The directory name is not a Python identifier; import it through the `nfb200` alias module at the repo root
(or the `src.flows` / `src.models` drop-in shims).
"""
from . import _lib, ops, packing, parallel, graphs  # noqa: F401
from .flows import (Flow, SequentialFlow, CouplingLayer, SplineCouplingLayer, rational_quadratic_spline,  # noqa: F401
                    MaskedLinear, MADE, MaskedAutoregressiveFlow, InverseAutoregressiveFlow, ARQS, DeviceGenerator)
from .models import NormalizingFlowModel, RealNVP, RealNVPSpline  # noqa: F401
from .packing import invalidate_caches  # noqa: F401

__all__ = ["Flow", "SequentialFlow", "CouplingLayer", "SplineCouplingLayer", "rational_quadratic_spline",
           "MaskedLinear", "MADE", "MaskedAutoregressiveFlow", "InverseAutoregressiveFlow", "ARQS",
           "NormalizingFlowModel", "RealNVP", "RealNVPSpline", "set_strict_fp32", "set_gemm_precision",
           "get_gemm_precision", "invalidate_caches", "DeviceGenerator"]


def set_strict_fp32(flag: bool = True) -> None:
    """Route every dense layer through the FP32-pipe GEMM (round-to-nearest FFMA accumulation) instead of the tcgen05
    3xTF32 kernels.  The tensor core truncates its fp32 accumulator on every MMA, so long contractions (hidden_dim
    >= 1024) drift: one RealNVPSpline(784, ., 1024) layer shows a coherent log-det bias of ~4e-4 (DESIGN.md,
    "fp32 parity on the tensor cores").  Strict mode meets the reference's fp32 error everywhere at ~1/5 of the GEMM
    throughput; the fused D <= 8 stacks (K = 64 contractions) are unaffected and stay on the tensor cores."""
    ops.USE_TENSOR_CORE_GEMM = not flag


_GEMM_PASSES = {"fp32": 3, "tf32": 1, "bf16": 1}
GEMM_PRECISIONS = tuple(_GEMM_PASSES)
_gemm_precision = "fp32"


def set_gemm_precision(mode: str = "fp32") -> None:
    """Precision of the tensor-core dense layers (conditioner MLPs, MADE masked linears, their input and weight gradients).

    "fp32" (default): 3xTF32 with short accumulation chains -- the reference's fp32 tolerances hold (DESIGN.md section 3).
    "tf32": one TF32 pass per product, operands rounded to the nearest TF32 (10-bit mantissa, three bits more than
    bf16) with fp32 accumulation -- the reduced-precision conditioner-GEMM mode of BASELINE config C4 (what the reference
    reaches with `MixedPrecisionFlow` autocast, optimization/mixed_precision.py:89-105).  Spline / affine transform
    arithmetic, BatchNorm and log-det reductions stay fp32 in both modes; the fused data_dim <= 8 stacks are unaffected.
    "bf16": the MADE-based flows (MAF.inverse / IAF.forward) run their whole parallel direction as ONE fused launch with
    bf16 operands on the tensor cores (kind::f16 MMAs, fp32 accumulation, activations kept on the SM in bf16:
    csrc/made_chain_bf16.cu); every other dense layer behaves as in "tf32".  Bounds: DESIGN.md, tests/test_gpu_bf16.py.
    Measured bounds of the modes: DESIGN.md "Reduced-precision mode", tests/test_gpu_tensorcore.py."""
    global _gemm_precision
    if mode not in _GEMM_PASSES:
        raise ValueError(f"gemm precision must be one of {sorted(_GEMM_PASSES)}, got {mode!r}")
    _lib.call("nf_set_option", 7, _GEMM_PASSES[mode])
    # "bf16": the remaining dense layers feed x to the tensor core straight from shared memory (SS form): the hardware
    # TRUNCATES the fp32 container to TF32 (error <= 2^-10 |x|, tighter than bf16 round-to-nearest's 2^-9) and the
    # converter warps -- the bound of the one-pass mode -- have no work at all (0.41 -> 0.30 ms at 262144 x 512 x 512)
    _lib.call("nf_set_option", 10, 1 if mode == "bf16" else 0)
    ops.MADE_CHAIN_BF16 = (mode == "bf16")
    _gemm_precision = mode


def get_gemm_precision() -> str:
    return _gemm_precision
