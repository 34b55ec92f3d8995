"""Every fused-stack kernel instantiation against the float64 oracle, across its dispatch envelope.

Eval-mode spline-coupling, affine-coupling and MAF / IAF stacks run as one launch of one of the template instantiations in
csrc/stack_small.cu and csrc/stack_tc.cu, each with a SAMPLE twin (sample_and_log_prob).  STACK_KERNELS lists all of them
and CASES states, per call, which instantiation a model must run.  The expectations are written out by hand -- a Python
copy of the dispatch would share its bugs.  Every case is checked four ways:
  * forward and inverse through the module against O.flow_model in float32 and float64 (tests.test_gpu_parity._within);
  * log_prob (fused LOG_PROB_HEAD | SKIP_Y epilogue) against log N(z) + log_det;
  * sample_and_log_prob (the SAMPLE twin) against the oracle's forward of the same N(0, I) draw;
  * the route: under torch.profiler exactly the expected stack kernel ran (or none), in one library launch.
FALLBACK_CASES sit just outside an envelope: no stack kernel may run, and the result must still match the oracle.
test_library_stack_kernels_match_the_table (no GPU) reads the library's entry symbols, so an instantiation added
without a case fails."""
import os
import re
import shutil
import subprocess
from dataclasses import dataclass, field

import numpy as np
import pytest
import torch

import nfb200 as N
from oracle import flows_oracle as O
from tests.test_gpu_parity import LD_ATOL, LD_RTOL, Z_ATOL, Z_RTOL, _within
from tests.test_gpu_published import _perturbed

DEV = "cuda:0"
STACK_KERNEL_NAMES = ("spline_stack_kernel", "spline_stack_tc2_kernel", "coupling_stack_kernel",
                      "coupling_stack_tc_kernel", "made_stack_tc_kernel")
_KERNEL_RE = re.compile(r"nf::(\w+_kernel)<([^>]*)>")

# ---- the coverage table: one row per instantiation, with the launch condition that selects it --------------------
_SPLINE_SIMT = [   # stack_small.cu, spline_stack_launch: HP 64 (R 2) / 128 (R 1), DM 4 (D <= 3) / 8, KMAX 8 (K <= 8) / 16
    "spline_stack_kernel<64, 2, 4, 8", "spline_stack_kernel<64, 2, 4, 16", "spline_stack_kernel<64, 2, 8, 8",
    "spline_stack_kernel<64, 2, 8, 16", "spline_stack_kernel<128, 1, 4, 8", "spline_stack_kernel<128, 1, 4, 16",
    "spline_stack_kernel<128, 1, 8, 8", "spline_stack_kernel<128, 1, 8, 16"]
_SPLINE_TC = [     # stack_tc.cu, spline_stack_tc_launch: DM 2 (D <= 2) / 4 (D = 3) / 8; (KMAX, KS) (8, 8) K = 8,
    # (10, 10) K = 10, (8, 0) K < 8, (10, 0) K = 9
    f"spline_stack_tc2_kernel<{dm}, {km}, {ks}" for dm in (2, 4, 8) for km, ks in ((8, 8), (10, 10), (8, 0), (10, 0))]
_COUPLING_SIMT = [  # stack_small.cu, coupling_stack_launch (USE_TENSOR_CORES=False): HP 64 / 128, DM 4 (D <= 3) / 8
    "coupling_stack_kernel<64, 2, 4", "coupling_stack_kernel<64, 2, 8", "coupling_stack_kernel<128, 1, 4",
    "coupling_stack_kernel<128, 1, 8"]
_COUPLING_TC = [    # stack_tc.cu, coupling_stack_tc_launch: DM 2 / 4 / 8, HP 64 (H <= 64) / 128
    f"coupling_stack_tc_kernel<{dm}, {hp}" for hp in (64, 128) for dm in (2, 4, 8)]
_MADE_TC = [f"made_stack_tc_kernel<{dm}" for dm in (2, 4, 8)]   # made_stack_tc_launch: DM 2 (D <= 2) / 4 (D = 3) / 8
STACK_KERNELS = [f"{k}, {s}>" for k in _SPLINE_SIMT + _SPLINE_TC + _COUPLING_SIMT + _COUPLING_TC + _MADE_TC
                 for s in ("false", "true")]
assert len(STACK_KERNELS) == 66 and len(set(STACK_KERNELS)) == 66


# ---- cases ---------------------------------------------------------------------------------------------------------
SKIP = "skip"      # log_prob of a MADE stack whose density direction is sequential at D != 2 (not fused)


def _fused(kernel):
    """The four calls of a spline / coupling stack: forward, inverse and log_prob on the kernel, sampling on its twin."""
    return dict(fwd=kernel + ", false>", inv=kernel + ", false>", log_prob=kernel + ", false>", sample=kernel + ", true>")


def _none():
    return dict(fwd=None, inv=None, log_prob=None, sample=None)


def _alt(D):
    even = "".join("1" if d % 2 == 0 else "0" for d in range(D))
    return (even, even.translate(str.maketrans("01", "10")))


def _half(D):
    first = "1" * (D // 2) + "0" * (D - D // 2)
    return (first, first.translate(str.maketrans("01", "10")))


@dataclass(frozen=True)
class Case:
    family: str              # spline | coupling | maf | iaf
    D: int
    H: int
    L: int
    B: int
    routes: dict             # fwd / inv / log_prob / sample -> expected instantiation, None (no stack kernel) or SKIP
    masks: tuple = ()        # coupling layers: per-layer mask strings, cycled over the L layers
    K: int = 0
    tc: bool = True          # flows.USE_TENSOR_CORES
    bn: bool = False         # batch_norm_between_layers
    use_bn: bool = False     # MADE conditioner BatchNorm (eval mode)
    spline: dict = field(default_factory=dict)   # bound, min_bin_width / height, min_derivative, data_min / data_max


MINS = dict(min_bin_width=2e-2, min_bin_height=5e-3, min_derivative=1e-1)
BIG = 262147               # > 148 SMs x CTAs per SM x rows per tile: the persistent grid loops over tiles

CASES = {
    # FP32-pipe spline stack: hidden_dim > 64, num_bins > 10 or > 2 transformed dims (the tcgen05 kernel refuses), or
    # USE_TENSOR_CORES=False
    "spl_simt_D1_H33_K7": Case("spline", 1, 33, 1, 129, _fused(_SPLINE_SIMT[0]), ("0",), K=7, tc=False),
    "spl_simt_D2_H8_K10": Case("spline", 2, 8, 3, 1, _fused(_SPLINE_SIMT[1]), _half(2), K=10, tc=False),
    "spl_simt_D3_K11_mins_bound2": Case("spline", 3, 64, 3, 511, _fused(_SPLINE_SIMT[1]), _half(3), K=11,
                                        spline=dict(bound=2.0, **MINS)),
    "spl_simt_D5_alt_H63_K8_bn": Case("spline", 5, 63, 3, 513, _fused(_SPLINE_SIMT[2]), _alt(5), K=8, bn=True),
    "spl_simt_D4_K9_bn": Case("spline", 4, 64, 3, 127, _fused(_SPLINE_SIMT[3]), _half(4), K=9, tc=False, bn=True),
    # D = 8, 4 transformed dims, hidden 64: K = 14 is the largest num_bins whose layer block + parameter columns fit in
    # 227 KB of shared memory (225 KB); K = 15 falls back (FALLBACK_CASES)
    "spl_simt_D8_alt_K14": Case("spline", 8, 64, 2, 4099, _fused(_SPLINE_SIMT[3]), _alt(8), K=14),
    "spl_simt_D2_H127_K5_rescale": Case("spline", 2, 127, 4, 4099, _fused(_SPLINE_SIMT[4]), _half(2), K=5,
                                        spline=dict(data_min=-3.0, data_max=4.0)),
    "spl_simt_D2_H128_K8_grid": Case("spline", 2, 128, 2, 65539, _fused(_SPLINE_SIMT[4]), _half(2), K=8, tc=False),
    "spl_simt_D3_H128_K16_bn": Case("spline", 3, 128, 3, 513, _fused(_SPLINE_SIMT[5]), _half(3), K=16, bn=True),
    "spl_simt_D7_alt_H65_K2": Case("spline", 7, 65, 3, 127, _fused(_SPLINE_SIMT[6]), _alt(7), K=2),
    "spl_simt_D8_twozero_H128_K11": Case("spline", 8, 128, 2, 511, _fused(_SPLINE_SIMT[7]), ("10111011", "01101111"),
                                         K=11, spline=dict(bound=2.0, **MINS)),
    # hidden 128, 4 transformed dims: K = 13 is the largest num_bins that fits (223 KB)
    "spl_simt_D8_alt_H100_K13": Case("spline", 8, 100, 2, 129, _fused(_SPLINE_SIMT[7]), _alt(8), K=13),
    # tcgen05 spline stack: hidden <= 64, num_bins <= 10, 1..2 transformed dims per layer (NO3 = 32 or 64)
    "spl_tc_D2_K8_L16_bn": Case("spline", 2, 64, 16, 4099, _fused(_SPLINE_TC[0]), _half(2), K=8, bn=True),
    "spl_tc_D2_K8_grid": Case("spline", 2, 64, 3, BIG, _fused(_SPLINE_TC[0]), _half(2), K=8),
    "spl_tc_D2_H33_K10_rescale": Case("spline", 2, 33, 3, 513, _fused(_SPLINE_TC[1]), _half(2), K=10,
                                      spline=dict(data_min=-3.0, data_max=4.0)),
    "spl_tc_D1_K2": Case("spline", 1, 64, 1, 127, _fused(_SPLINE_TC[2]), ("0",), K=2),
    "spl_tc_D2_H8_K3_L15_bn": Case("spline", 2, 8, 15, 511, _fused(_SPLINE_TC[2]), _half(2), K=3, bn=True),
    "spl_tc_D2_K9_mins_bound2": Case("spline", 2, 64, 3, 4099, _fused(_SPLINE_TC[3]), _half(2), K=9,
                                     spline=dict(bound=2.0, **MINS)),
    "spl_tc_D3_K8_bn_bound2": Case("spline", 3, 64, 3, 511, _fused(_SPLINE_TC[4]), _half(3), K=8, bn=True,
                                   spline=dict(bound=2.0)),
    "spl_tc_D3_H63_K10_L1": Case("spline", 3, 63, 1, 1, _fused(_SPLINE_TC[5]), _half(3), K=10),
    "spl_tc_D3_H33_K7_identity": Case("spline", 3, 33, 4, 129, _fused(_SPLINE_TC[6]), ("100", "011", "111", "010"), K=7),
    "spl_tc_D3_K9_rescale_mins": Case("spline", 3, 64, 3, 513, _fused(_SPLINE_TC[7]), _half(3), K=9,
                                      spline=dict(bound=3.0, data_min=-2.0, data_max=6.0, **MINS)),
    "spl_tc_D8_onezero_K8": Case("spline", 8, 64, 3, 4099, _fused(_SPLINE_TC[8]), ("11101111", "01111111", "11111110"), K=8),
    "spl_tc_D8_twozero_H48_K10_bn": Case("spline", 8, 48, 3, 513, _fused(_SPLINE_TC[9]),
                                         ("01111101", "10111110", "11011011"), K=10, bn=True),
    "spl_tc_D4_K7_bn": Case("spline", 4, 64, 3, 127, _fused(_SPLINE_TC[10]), _alt(4), K=7, bn=True),
    "spl_tc_D5_K9_rescale": Case("spline", 5, 64, 1, 511, _fused(_SPLINE_TC[11]), ("10110",), K=9,
                                 spline=dict(data_min=-1.0, data_max=2.5)),
    # FP32-pipe affine coupling stack (USE_TENSOR_CORES=False)
    "cpl_simt_D1_H8": Case("coupling", 1, 8, 1, 129, _fused(_COUPLING_SIMT[0]), ("0",), tc=False),
    "cpl_simt_D2_grid": Case("coupling", 2, 64, 2, BIG, _fused(_COUPLING_SIMT[0]), _half(2), tc=False),
    "cpl_simt_D7_alt_bn": Case("coupling", 7, 64, 3, 4099, _fused(_COUPLING_SIMT[1]), _alt(7), tc=False, bn=True),
    "cpl_simt_D3_H128_bn": Case("coupling", 3, 128, 4, 513, _fused(_COUPLING_SIMT[2]), _half(3), tc=False, bn=True),
    "cpl_simt_D8_alt_H65": Case("coupling", 8, 65, 2, 511, _fused(_COUPLING_SIMT[3]), _alt(8), tc=False),
    # tcgen05 affine coupling stack: hidden <= 128
    "cpl_tc_D2_H33_L13": Case("coupling", 2, 33, 13, 4099, _fused(_COUPLING_TC[0]), _half(2)),
    "cpl_tc_D2_grid_bn": Case("coupling", 2, 64, 2, BIG, _fused(_COUPLING_TC[0]), _half(2), bn=True),
    "cpl_tc_D3_H63_bn": Case("coupling", 3, 63, 3, 127, _fused(_COUPLING_TC[1]), _half(3), bn=True),
    "cpl_tc_D5_alt_H8_L1": Case("coupling", 5, 8, 1, 1, _fused(_COUPLING_TC[2]), _alt(5)),
    "cpl_tc_D4_identity": Case("coupling", 4, 64, 3, 513, _fused(_COUPLING_TC[2]), ("1100", "1111", "0011")),
    "cpl_tc_D2_H128_grid": Case("coupling", 2, 128, 3, 100003, _fused(_COUPLING_TC[3]), _half(2)),
    "cpl_tc_D3_H100_L1": Case("coupling", 3, 100, 1, 129, _fused(_COUPLING_TC[4]), _half(3)),
    # at L = 3 this seed grows |z| to ~850 and the float32 reference is itself 1e-3 off; the 48-MMA truncating TMEM chains
    # of the 128-wide kernel then put ~0.4 % of the elements up to 5e-2 off (a CPU emulation of round-toward-zero
    # accumulation reproduces it): outside what this bound can check, so L = 2 keeps the model conditioned (|z| <= 17)
    "cpl_tc_D8_H127_bn": Case("coupling", 8, 127, 2, 511, _fused(_COUPLING_TC[5]), _alt(8), bn=True),
    # MAF / IAF stack: hidden <= 64, D <= 8; the parallel direction (MAF density, IAF sampling) at every D, the sequential
    # one only at D = 2.  The SAMPLE twins of DM 4 and 8 are reached only through IAF stacks.
    "maf_D2_bn": Case("maf", 2, 64, 6, 4099, dict(fwd="made_stack_tc_kernel<2, false>", inv="made_stack_tc_kernel<2, false>",
                                                   log_prob="made_stack_tc_kernel<2, false>",
                                                   sample="made_stack_tc_kernel<2, true>"), bn=True),
    "iaf_D2_grid": Case("iaf", 2, 64, 2, BIG, dict(fwd="made_stack_tc_kernel<2, false>", inv="made_stack_tc_kernel<2, false>",
                                                    log_prob="made_stack_tc_kernel<2, false>",
                                                    sample="made_stack_tc_kernel<2, true>")),
    "iaf_D1_H8": Case("iaf", 1, 8, 1, 129, dict(fwd="made_stack_tc_kernel<2, false>", inv=None, log_prob=SKIP,
                                                sample="made_stack_tc_kernel<2, true>")),
    "maf_D3_H33_usebn": Case("maf", 3, 33, 3, 513, dict(fwd=None, inv="made_stack_tc_kernel<4, false>",
                                                        log_prob="made_stack_tc_kernel<4, false>", sample=None), use_bn=True),
    "iaf_D3_H63_L1": Case("iaf", 3, 63, 1, 127, dict(fwd="made_stack_tc_kernel<4, false>", inv=None, log_prob=SKIP,
                                                     sample="made_stack_tc_kernel<4, true>")),
    "maf_D4_bn": Case("maf", 4, 64, 3, 511, dict(fwd=None, inv="made_stack_tc_kernel<8, false>",
                                                 log_prob="made_stack_tc_kernel<8, false>", sample=None), bn=True),
    "iaf_D6_H48_bn": Case("iaf", 6, 48, 3, 4099, dict(fwd="made_stack_tc_kernel<8, false>", inv=None, log_prob=SKIP,
                                                      sample="made_stack_tc_kernel<8, true>"), bn=True),
    "iaf_D7_usebn": Case("iaf", 7, 64, 2, 513, dict(fwd="made_stack_tc_kernel<8, false>", inv=None, log_prob=SKIP,
                                                    sample="made_stack_tc_kernel<8, true>"), use_bn=True),
    "maf_D8_H8_L12": Case("maf", 8, 8, 12, 129, dict(fwd=None, inv="made_stack_tc_kernel<8, false>",
                                                     log_prob="made_stack_tc_kernel<8, false>", sample=None)),
    "iaf_D8_L1": Case("iaf", 8, 64, 1, 1, dict(fwd="made_stack_tc_kernel<8, false>", inv=None, log_prob=SKIP,
                                               sample="made_stack_tc_kernel<8, true>")),
}

FALLBACK_CASES = {
    # FP32-pipe spline kernel out of shared memory: layer block + [NO][256] parameter columns = 261 KB at K = 16 and
    # 240 KB at K = 15 (> 227 KB); the tcgen05 kernel refuses K > 10 and 4 transformed dims
    "spl_D8_alt_K16": Case("spline", 8, 64, 2, 513, _none(), _alt(8), K=16),
    "spl_D8_alt_K15": Case("spline", 8, 64, 2, 513, _none(), _alt(8), K=15),
    "maf_H65": Case("maf", 4, 65, 2, 513, dict(_none(), log_prob=None)),
    "maf_D3_sequential": Case("maf", 3, 32, 2, 511, dict(fwd=None, inv="made_stack_tc_kernel<4, false>",
                                                         log_prob="made_stack_tc_kernel<4, false>", sample=None)),
}


def _claims():
    rows = {k: [] for k in STACK_KERNELS}
    for name, c in list(CASES.items()) + list(FALLBACK_CASES.items()):
        for call, k in c.routes.items():
            if k not in (None, SKIP):
                assert k in rows, f"case {name} ({call}) expects {k}, which is not a row of STACK_KERNELS"
                rows[k].append(name)
    return rows


KERNEL_TABLE = _claims()          # instantiation -> cases that must land on it
_UNCLAIMED = [k for k, cs in KERNEL_TABLE.items() if not cs]
assert not _UNCLAIMED, f"stack kernels without a case: {_UNCLAIMED}"
for _n, _c in list(CASES.items()) + list(FALLBACK_CASES.items()):
    assert set(_c.routes) == {"fwd", "inv", "log_prob", "sample"}, _n
    assert all(len(m) == _c.D for m in _c.masks), _n
    assert _c.H <= 64 or _c.B < N.flows.WIDE_OVER_STACK_MIN_ROWS or not _c.tc or _c.family != "spline", _n


# ---- model, oracle and inputs --------------------------------------------------------------------------------------
def _masks(c):
    return [torch.tensor([float(ch) for ch in c.masks[i % len(c.masks)]]) for i in range(c.L)]


def _model(c, seed):
    torch.manual_seed(seed)
    if c.family == "spline":
        layers = [N.SplineCouplingLayer(c.D, c.H, m, num_bins=c.K, **c.spline) for m in _masks(c)]
    elif c.family == "coupling":
        layers = [N.CouplingLayer(c.D, c.H, m) for m in _masks(c)]
    else:
        cls = N.MaskedAutoregressiveFlow if c.family == "maf" else N.InverseAutoregressiveFlow
        layers = [cls(c.D, c.H, use_batch_norm=c.use_bn) for _ in range(c.L)]
    model = _perturbed(N.NormalizingFlowModel(layers, batch_norm_between_layers=c.bn), seed)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    spec = dict(kind=c.family)
    if c.family == "spline":
        spec.update(num_bins=c.K, **c.spline)
    return model.to(DEV), sd, [spec] * c.L


def _edges(c):
    """Data-space values that land exactly on the spline's interval ends (±bound, or data_min / data_max)."""
    bound = c.spline.get("bound", 5.0)
    if "data_min" in c.spline:
        return c.spline["data_min"], c.spline["data_max"]
    return -bound, bound


def _inputs(c, seed):
    """randn scaled so a few percent of the values land in the identity tails, and in the last rows (when there is
    room) the edge values: the interval ends exactly and one float32 ulp inside / outside, ±bound, ±0, a subnormal; then
    the stress rows NaN, ±Inf and 1e8."""
    lo, hi = _edges(c)
    mid, half = 0.5 * (lo + hi), 0.5 * (hi - lo)
    x = mid + 0.5 * half * torch.randn(c.B, c.D, generator=torch.Generator().manual_seed(seed))
    f = np.float32
    bound = c.spline.get("bound", 5.0)
    special = [lo, hi, np.nextafter(f(lo), f(0)), np.nextafter(f(lo), f(-np.inf)), np.nextafter(f(hi), f(0)),
               np.nextafter(f(hi), f(np.inf)), -bound, bound, 0.0, -0.0, 1e-40,
               float("nan"), float("inf"), -float("inf"), 1e8]
    if c.B >= 2 * len(special):
        for i, v in enumerate(special):
            x[c.B - len(special) + i, :] = float(v)
        x[c.B - 2 * len(special), 0] = float("nan")          # one NaN dim only: the other dims follow the reference
    return x


def _wild(x):
    """Stress rows: compared only for their NaN / finiteness pattern (as test_gpu_parity._loose)."""
    return (x.abs() > 50).any(dim=1) | ~torch.isfinite(x).all(dim=1)


def _f64(sd):
    return {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}


def _profiled(fn):
    """fn() once to build the packed weights, then again under torch.profiler: (output, stack kernels that ran,
    library launches of the profiled call).  Every call launches at least one library kernel, so a trace without any
    nf:: kernel is a trace whose device activity was not delivered (seen in long test sessions): the call is traced
    again, at most twice more, rather than read as "no stack kernel ran"."""
    fn()
    torch.cuda.synchronize()
    for _ in range(3):
        before = N._lib.launch_count()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        launches = N._lib.launch_count() - before
        names = [e.name for e in prof.events() if "nf::" in e.name]
        if names:
            break
    assert names, "the profiler recorded no library kernel in three traces"
    ran = [f"{m.group(1)}<{m.group(2)}>" for n in names
           for m in [_KERNEL_RE.search(n)] if m and m.group(1) in STACK_KERNEL_NAMES]
    return out, ran, launches


def _check_route(what, expected, ran, launches):
    if expected is None:
        assert ran == [], f"{what}: expected no stack kernel, ran {ran}"
    else:
        assert ran == [expected], f"{what}: expected {expected}, ran {ran}"
        assert launches == 1, f"{what}: {launches} library launches"


def _sensitivity(sd, specs, x, inverse, bn):
    """Per-element sensitivity of the float32 oracle to ~1-ulp relative noise on the weights (6 draws, as
    test_gpu_parity._conditioning): what an implementation with another summation order may legitimately differ by."""
    gen = torch.Generator().manual_seed(0)
    y0, l0 = O.flow_model(sd, "", specs, x, inverse, bn_between=bn)
    cy, cl = torch.zeros_like(y0), torch.zeros(x.shape[0])
    for _ in range(6):
        sdp = {k: (v * (1 + 2e-7 * torch.randn(v.shape, generator=gen)) if v.is_floating_point() and "weight" in k else v)
               for k, v in sd.items()}
        y1, l1 = O.flow_model(sdp, "", specs, x, inverse, bn_between=bn)
        cy = torch.maximum(cy, (y1 - y0).abs().nan_to_num(0.0))
        cl = torch.maximum(cl, (torch.as_tensor(l1) - l0).abs().expand(x.shape[0]).nan_to_num(0.0))
    return cy.double(), cl.double()


def _compare(what, y, ld, ry, rld, y64, ld64, wild, D, L, cond):
    """cond() -> per-element sensitivities (z, log_det) of every row: evaluated only when the strict bound fails.
    An output element has passed through up to L layer transforms and a row log-det sums up to D * L of them, so each
    compared value meets an ill-conditioned transform that many times as often (the `terms` of _within)."""
    y, ld = y.detach().cpu(), ld.detach().cpu()
    calm = ~wild
    memo = []
    sens = lambda i: (memo or memo.append(cond()) or memo)[0][i][calm]
    _within(y[calm], ry[calm], y64[calm], Z_ATOL, Z_RTOL, f"{what} z", lambda: sens(0), terms=L)
    _within(ld[calm], rld[calm], ld64[calm], LD_ATOL, LD_RTOL, f"{what} log_det", lambda: sens(1), terms=D * L)
    if wild.any():
        assert torch.equal(torch.isfinite(y[wild]), torch.isfinite(ry[wild])), f"{what}: finiteness of z (stress rows)"
        assert torch.equal(torch.isfinite(ld[wild]), torch.isfinite(rld[wild])), f"{what}: finiteness of log_det"


def _run_case(name, c, seed):
    old = N.flows.USE_TENSOR_CORES
    N.flows.USE_TENSOR_CORES = c.tc
    try:
        model, sd, specs = _model(c, seed)
        sd64 = _f64(sd)
        x = _inputs(c, seed)
        wild = _wild(x)
        xd = x.to(DEV)
        ref = {}
        with torch.no_grad():
            for inverse, call in ((False, "fwd"), (True, "inv")):
                ry, rld = O.flow_model(sd, "", specs, x, inverse, bn_between=c.bn)
                y64, ld64 = O.flow_model(sd64, "", specs, x.double(), inverse, bn_between=c.bn)
                rld, ld64 = torch.as_tensor(rld).expand(c.B), torch.as_tensor(ld64).expand(c.B)
                ref[call] = (ry, rld, y64, ld64)
                (y, ld), ran, launches = _profiled(lambda: model.inverse(xd) if inverse else model.forward(xd))
                _check_route(f"{name} {call}", c.routes[call], ran, launches)
                _compare(f"{name} {call}", y, ld, ry, rld, y64, ld64, wild, c.D, c.L,
                         lambda: _sensitivity(sd, specs, x, inverse, c.bn))

            if c.routes["log_prob"] != SKIP:
                lp, ran, launches = _profiled(lambda: model.log_prob(xd))
                _check_route(f"{name} log_prob", c.routes["log_prob"], ran, launches)
                rz, rld, z64, ld64 = ref["inv"]
                lp = lp.cpu()
                lp32, lp64 = O.std_normal_log_prob(rz) + rld, O.std_normal_log_prob(z64) + ld64
                calm = ~wild
                _within(lp[calm], lp32[calm], lp64[calm], 2e-4, 1e-5, f"{name} log_prob", terms=c.D)
                if wild.any():
                    assert torch.equal(torch.isfinite(lp[wild]), torch.isfinite(lp32[wild])), f"{name} log_prob stress rows"

            def sample():
                gen = torch.Generator(device=DEV)
                gen.manual_seed(seed)
                return model.sample_and_log_prob(c.B, generator=gen)
            (xs, lq), ran, launches = _profiled(sample)
            _check_route(f"{name} sample", c.routes["sample"], ran, launches)
            z = N.ops.std_normal_draw(seed, 0, c.B, c.D, torch.float32, torch.device(DEV)).cpu()
            rx, rld = O.flow_model(sd, "", specs, z, False, bn_between=c.bn)
            x64, ld64 = O.flow_model(sd64, "", specs, z.double(), False, bn_between=c.bn)
            lq32 = O.std_normal_log_prob(z) - torch.as_tensor(rld).expand(c.B)
            lq64 = O.std_normal_log_prob(z.double()) - torch.as_tensor(ld64).expand(c.B)
            _within(xs.cpu(), rx, x64, Z_ATOL, Z_RTOL, f"{name} sample x")
            _within(lq.cpu(), lq32, lq64, 2e-4, 1e-5, f"{name} sample log_q", terms=c.D)
    finally:
        N.flows.USE_TENSOR_CORES = old


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_stack_kernel_matches_float64_oracle(name):
    _run_case(name, CASES[name], seed=sum(map(ord, name)))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FALLBACK_CASES))
def test_outside_the_envelope_no_stack_kernel_runs(name):
    _run_case(name, FALLBACK_CASES[name], seed=sum(map(ord, name)))


def _tool(name):
    return shutil.which(name) or next((p for p in (os.path.join("/usr/local/cuda/bin", name),) if os.path.exists(p)), None)


def test_library_stack_kernels_match_the_table():
    """The library's stack-kernel entry symbols (cuobjdump -symbols, demangled) are exactly the table's rows: a new
    instantiation needs a case that lands on it."""
    lib, cuobjdump, cxxfilt = N._lib.LIB_PATH, _tool("cuobjdump"), _tool("c++filt")
    if not os.path.exists(lib) or cuobjdump is None or cxxfilt is None:
        pytest.skip("needs the built library, cuobjdump and c++filt")
    out = subprocess.run([cuobjdump, "-symbols", lib], capture_output=True, text=True, check=True).stdout
    mangled = [line.split()[-1] for line in out.splitlines() if "STO_ENTRY" in line]
    names = subprocess.run([cxxfilt], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    found = {f"{m.group(1)}<{m.group(2)}>" for line in names.splitlines()
             for m in [_KERNEL_RE.search(line)] if m and m.group(1) in STACK_KERNEL_NAMES}
    assert found, "no stack kernel entry found in the library's symbols"
    assert found == set(STACK_KERNELS), (f"in the library, not in the table: {sorted(found - set(STACK_KERNELS))}; "
                                         f"in the table, not in the library: {sorted(set(STACK_KERNELS) - found)}")
