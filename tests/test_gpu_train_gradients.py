"""GPU: float32 training gradients against the float64 oracle, on the kernels only a training step runs.

A float32 training step takes the layered route (DESIGN.md, "layered") at sizes where dtype, alignment and row count
select the tensor-core GEMMs (gemm_tc2 / wgrad_tc, masked for MADE), the 128-bit BatchNorm and fused ReLU / bias-gradient
kernels, the streaming spline backward and the float32 transform backward kernels.  test_gpu_gradients.py covers the
float64 route; this file covers the float32 one:

  * model level: one training step's loss -log_prob(x).mean() (the quickstart objective) and every parameter gradient,
    against autograd of the CPU oracle in float64.  The bound is calibrated on the oracle's own float32 error e32;
    the profiler asserts that the kernels each case is meant to cover ran in its backward;
  * the BatchNorm(+ReLU) op against F.batch_norm in float64, over H and B on both sides of every dispatch threshold;
  * the invariant the 128-bit BatchNorm backward relies on: the ReLU mask it re-derives from x equals the one the
    forward wrote into y, bit for bit.
"""
import re

import pytest
import torch
import torch.nn.functional as F

import nfb200 as N
from oracle import flows_oracle as O
from tests import golden_util as G
from tests.test_gpu_gradients import _perturb

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# A tensor passes when e = |g - g64| / |g64| <= max(K_E32 * e32, FLOOR), with e32 the same ratio for the oracle run in
# float32 on the CPU (norms over the whole tensor).  Measured on one B200 (1000 W) over the 14 cases and the BatchNorm
# grid (1398 tensors): median e 1.7e-6 at a median e / e32 of 1.7.
#   * K_E32: the largest e / e32 at an e above 1e-4 was 8.0 (realnvp2_bn_between dflow.flows.1.s_net.1.bias,
#     e = 1.1e-4, e32 = 1.4e-5); K_E32 is twice that.  The BatchNorm op reached at most 3.3.
#   * FLOOR: e / e32 exceeded 16 on 56 tensors of six cases, where the float32 oracle happens to be far more accurate on
#     that tensor than on its neighbours (e32 down to 8.8e-9).  Their largest e were 8.2e-5 (realnvp2_bn_between
#     dflow.flows.1.s_net.6.bias, e32 = 1.0e-6) and 7.0e-5 (spline2 dflows.3.param_net.0.weight, e32 = 7.4e-7); FLOOR
#     is 2.4 times the larger.
K_E32 = 16.0
FLOOR = 2e-4
# Biases of a Linear followed by a train-mode BatchNorm have a zero gradient in exact arithmetic; what both sides compute
# there is rounding noise, compared by the same ratio (|g| against the float32 oracle's |g32|) with its own constant.
# Measured: at most 2.9.
K_ZERO = 10.0
PERTURB = 0.05        # parameter perturbation (the final layers start at zero); larger ones make the deep stacks blow up
# Column reductions (BatchNorm ggamma / gbeta): |g - g64| <= RED_TOL * sum|terms|, as test_col_sum_matches_float64.
RED_TOL = 1e-6


# ---- helpers --------------------------------------------------------------------------------------------------------
def _rel(a, ref):
    a, ref = a.detach().double().cpu(), ref.detach().double().cpu()
    return ((a - ref).norm() / ref.norm()).item()


def _check(what, got, ref64, ref32, failures, k=None):
    """Normwise criterion; prints e, e32 and their ratio, appends a message to `failures` when the bound is missed."""
    n64 = ref64.detach().double().norm().item()
    assert n64 > 0, f"{what}: the float64 reference is zero, the comparison would be vacuous"
    assert torch.isfinite(got.detach()).all(), f"{what}: non-finite values"
    e, e32 = _rel(got, ref64), _rel(ref32, ref64)
    bound = max((K_E32 if k is None else k) * e32, FLOOR)
    print(f"  {what:<48s} e={e:.3e} e32={e32:.3e} ratio={e / max(e32, 1e-300):.2f}")
    if not e <= bound:
        failures.append(f"{what}: e={e:.3e} > bound {bound:.3e} (e32={e32:.3e})")


_NAME_RE = re.compile(r"nf::(\w+)(<[^>(]*>)?")


def _traced(fn):
    """fn() under torch.profiler: (its result, the library kernels it ran, each as its bare name and as
    name<template arguments>).  In long test sessions the first device activity after the profiler starts has been
    missing from the trace (the first of the three kernels of nf_batchnorm_backward, in every one of three traces, while
    the other two were there), so a torch kernel and a synchronisation open every trace before fn runs.  A trace that
    still holds fewer library kernels than the library counted launches is taken again, at most twice more (fn must be
    repeatable), and the last one is used as it is."""
    sentinel = torch.zeros(1, device=DEV)
    for _ in range(3):
        torch.cuda.synchronize()
        before = N._lib.launch_count()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            sentinel.add_(1)
            torch.cuda.synchronize()
            out = fn()
            torch.cuda.synchronize()
        launched = N._lib.launch_count() - before
        found = [m for m in (_NAME_RE.search(ev.name) for ev in prof.events()) if m]
        if found and len(found) >= launched:
            break
    names = {m.group(1) for m in found} | {m.group(1) + m.group(2) for m in found if m.group(2)}
    return out, names


def _backward_traced(loss, leaves):
    """loss.backward() (the graph is retained, so that it can be traced again) with fresh gradients; returns the library
    kernels it ran."""
    def run():
        for t in leaves:
            t.grad = None
        loss.backward(retain_graph=True)
    return _traced(run)[1]


# ---- inputs ---------------------------------------------------------------------------------------------------------
def _moons(n, D, gen):
    """The two-moons-like set of test_training_reduces_nll_realnvp."""
    x = torch.randn(n, D, generator=gen)
    x[:, 1] = 0.5 * x[:, 0] ** 2 + 0.3 * x[:, 1]
    return x


def _normal(n, D, gen):
    return torch.randn(n, D, generator=gen)


def _with_rows(base, values):
    """base(n, D, gen) with its first rows set to the given constants (outliers, values outside the spline interval)."""
    def make(n, D, gen):
        x = base(n, D, gen)
        for i, v in enumerate(values):
            x[i] = v * (1 if i % 2 == 0 else -1)
        return x
    return make


# Spline rows beyond the bound take the identity tails (|x| > 5, or > 3 for data_min / data_max = -+3).
SPLINE_EDGE = (5.5, 7.0, 9.0, 12.0)


def _alt(D, first=1.0):
    return torch.tensor([first, 1 - first] * (D // 2))


def _clamped_s(m):
    """RealNVP(6, 4, 30) whose first layer in the density direction has s near +9.5 on one transformed dim and -9.8 on
    another, so that some rows reach the +10 clamp of s and others the -10 one (where s gets no gradient): 63 and 51 of
    the 1500 rows of the case, which the test checks on the oracle side."""
    with torch.no_grad():
        m.flow.flows[3].s_net[6].bias[:2] += torch.tensor([9.5, -9.8])
    return m


def _clamped_rows(sd0, x):
    """Rows of x for which the float64 oracle's s (before its clamp) of layer 3 is > 10 on dim 0 and < -10 on dim 1."""
    sd = {k: (v.double() if v.is_floating_point() else v) for k, v in sd0.items()}
    with torch.no_grad():
        s = O.coupling_conditioner(sd, "flow.flows.3.s_net", x.double() * sd["flow.flows.3.mask"], training=True)
    return int((s[:, 0] > 10).sum()), int((s[:, 1] < -10).sum())


def _spline2():
    return N.NormalizingFlowModel([N.SplineCouplingLayer(2, 64, _alt(2, 1.0 if i % 2 == 0 else 0.0), num_bins=8)
                                   for i in range(8)])


# name: (model constructor, rows, input generator, oracle case (golden_util.oracle_eval keys), kernels the backward runs)
VEC_BN = {"bn_bwd_partial_vec4_kernel", "bn_bwd_apply_vec4_kernel"}
CASES = {
    "realnvp2": (lambda: N.RealNVP(2, 8, 64), 65536, _moons, dict(kind="realnvp", L=8),
                 VEC_BN | {"wgrad_tc_kernel", "gemm_tc2_kernel", "affine_coupling_vec_bwd_kernel"}),
    "realnvp2_ragged": (lambda: N.RealNVP(2, 8, 64), 4099, _moons, dict(kind="realnvp", L=8),
                        VEC_BN | {"wgrad_tc_kernel", "gemm_tc2_kernel", "affine_coupling_bwd_kernel"}),
    "realnvp2_bn_between": (lambda: N.RealNVP(2, 8, 64, batch_norm_between_layers=True), 4096,
                            _moons, dict(kind="realnvp", L=8, bn=True),
                            VEC_BN | {"wgrad_tc_kernel", "gemm_tc2_kernel", "affine_coupling_vec_bwd_kernel"}),
    "realnvp256": (lambda: N.RealNVP(256, 2, 512), 2048, _normal, dict(kind="realnvp", L=2),
                   VEC_BN | {"wgrad_tc_kernel"}),
    "realnvp_odd": (lambda: N.RealNVP(6, 4, 30), 1500, _normal, dict(kind="realnvp", L=4),
                    {"bn_bwd_partial_kernel", "bn_bwd_apply_kernel", "skinny_k_kernel"}),
    "spline2": (_spline2, 65536, _with_rows(_moons, SPLINE_EDGE), dict(kind="splinestack", L=8, K=8),
                {"relu_bwd_colsum_vec4_kernel", "spline_stream_bwd_kernel<8, 1, true, 1>"}),
    "spline16": (lambda: N.RealNVPSpline(16, 4, 128), 4099, _with_rows(_normal, SPLINE_EDGE),
                 dict(kind="realnvpspline", L=4, K=10),
                 {"relu_bwd_colsum_vec4_kernel", "spline_stream_bwd_kernel<10, 8, true, 0>"}),
    "spline_wide": (lambda: N.SplineCouplingLayer(72, 64, _alt(72)), 2048, _with_rows(_normal, SPLINE_EDGE),
                    dict(kind="spline", K=10, extra={}), {"spline_stream_bwd_kernel<10, 32, true, 2>"}),
    "spline_rescale": (lambda: N.SplineCouplingLayer(8, 64, _alt(8), data_min=-3.0, data_max=3.0), 2048,
                       _with_rows(_normal, (3.5, 4.0, 6.0, 3.2)),
                       dict(kind="spline", K=10, extra=dict(data_min=-3.0, data_max=3.0)),
                       {"feature_affine_bwd_x_kernel"}),
    "maf64": (lambda: N.MaskedAutoregressiveFlow(64, 512), 2048, _normal, dict(kind="maf"),
              {"wgrad_tc_kernel", "gemm_tc2_kernel", "affine_ar_bwd_kernel"}),
    "maf_bn": (lambda: N.MaskedAutoregressiveFlow(16, 128, use_batch_norm=True), 4099, _normal, dict(kind="maf"),
               VEC_BN | {"affine_ar_bwd_kernel"}),
    "iaf_seq": (lambda: N.InverseAutoregressiveFlow(8, 64), 1024, _normal, dict(kind="iaf"),
                {"ar_step_bwd_kernel", "ar_finish_bwd_kernel"}),
    "arqs": (lambda: N.ARQS(5, 64, num_bins=8, data_min=-4.0, data_max=4.0), 1024,
             lambda n, D, gen: _normal(n, D, gen).clamp(-3.9, 3.9),
             dict(kind="arqs", K=8, extra=dict(data_min=-4.0, data_max=4.0)), {"arqs_step_bwd_kernel"}),
    # fine-tuning with frozen statistics: eval-mode BatchNorm with gradients (the apply kernel's training = 0 branch)
    "eval_finetune": (lambda: N.RealNVP(2, 8, 64), 4096, _moons, dict(kind="realnvp", L=8),
                      {"bn_bwd_apply_vec4_kernel", "wgrad_tc_kernel"}),
}


def _perturb_stats(m, seed):
    """Running statistics away from (0, 1), so that eval-mode BatchNorm and the running-statistics update are not
    trivial."""
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, b in m.named_buffers():
            if name.endswith("running_mean"):
                b.add_(0.2 * torch.randn(b.shape, generator=gen))
            elif name.endswith("running_var"):
                b.mul_(torch.exp(0.3 * torch.randn(b.shape, generator=gen)))


def _oracle_step(case, sd0, params, x, dtype, training):
    """Autograd of the oracle's loss in `dtype` on the CPU: (loss, z, log-det, x gradient, parameter gradients)."""
    sd = {k: (v.to(dtype).requires_grad_(k in params) if v.is_floating_point() else v.clone()) for k, v in sd0.items()}
    xo = x.to(dtype).requires_grad_()
    z, ld = G.oracle_eval(dict(case, sd=sd, x=xo), True, grad=True, training=training)
    loss = -(O.std_normal_log_prob(z) + ld).mean()
    loss.backward()
    return loss, z, ld, xo.grad, {k: sd[k].grad for k in params}


def _oracle_running_stats(case, sd0, x, dtype):
    """Running statistics after one train-mode pass of the oracle with update=True."""
    sd = {k: (v.to(dtype) if v.is_floating_point() else v.clone()) for k, v in sd0.items()}
    with torch.no_grad():
        if case["kind"] == "realnvp":
            p, specs = G.stack_specs(case)
            O.flow_model(sd, p, specs, x.to(dtype), True, bn_between=case.get("bn", False), training=True, update=True)
        else:
            O.maf_inverse(sd, "", x.to(dtype), training=True, update=True)
    return sd


def _zero_in_exact_arithmetic(k, sd0):
    """A train-mode BatchNorm removes its input's per-column offset, so the bias of the Linear in front of it has a zero
    gradient."""
    head, _, leaf = k.rpartition(".")
    stem, _, idx = head.rpartition(".")
    return (leaf == "bias" and idx.isdigit() and f"{head}.running_mean" not in sd0
            and f"{stem}.{int(idx) + 1}.running_mean" in sd0)


@pytest.mark.parametrize("name", list(CASES))
def test_float32_training_gradients_match_float64_oracle(name):
    build, rows, data, case, must_run = CASES[name]
    training = name != "eval_finetune"
    torch.manual_seed(0)
    m = build()
    _perturb(m, 17, sigma=PERTURB)
    _perturb_stats(m, 18)
    if name == "realnvp_odd":
        _clamped_s(m)
    sd0 = {k: v.detach().clone() for k, v in m.state_dict().items()}
    D = next(v for k, v in sd0.items() if k.endswith("mask")).shape[-1]
    x = data(rows, D, torch.Generator().manual_seed(19))
    if name == "realnvp_odd":
        up, down = _clamped_rows(sd0, x)
        assert 10 <= up < rows // 2 and 10 <= down < rows // 2, f"rows at the s clamp: {up} at +10, {down} at -10"
    m.to(DEV).train(training)
    if name == "maf64":
        hh = m.conditioner.net[2]
        assert N.ops.mask_plan(hh.mask) is not None, "the MADE hidden mask has no tile plan: the masked wgrad would not run"

    xd = x.to(DEV).requires_grad_()
    # what log_prob runs when autograd is on (flows.flow_log_prob): the inverse, then the N(0, I) head kernel; z and the
    # log-det are compared too, and log_prob itself is checked against this at the end
    z, ld = m.inverse(xd)
    lp = N.ops.std_normal_log_prob(z, ld)
    loss = -lp.mean()
    named = dict(m.named_parameters())
    ran = _backward_traced(loss, list(named.values()) + [xd])

    r64 = _oracle_step(case, sd0, set(named), x, torch.float64, training)
    r32 = _oracle_step(case, sd0, set(named), x, torch.float32, training)
    print(f"\n{name}: {rows} rows, backward ran {sorted(k for k in ran if '<' not in k)}")
    failures = []
    for what, got, i in (("loss", loss, 0), ("z", z, 1), ("log_det", ld, 2), ("x grad", xd.grad, 3)):
        _check(f"{name} {what}", got, r64[i], r32[i], failures)
    checked = 0
    for k, p in named.items():
        if r64[4][k] is None:                       # not used by the density direction (the last between-layer BatchNorm)
            assert p.grad is None or not p.grad.any(), f"{name} d{k}: gradient for a parameter the loss does not use"
            continue
        zero = training and _zero_in_exact_arithmetic(k, sd0)
        _check(f"{name} d{k}" + (" (exact: 0)" if zero else ""), p.grad, r64[4][k], r32[4][k], failures,
               K_ZERO if zero else None)
        checked += 1
    assert checked > 0

    stats = [k for k in sd0 if "running_" in k]
    if training and stats:
        s64, s32 = _oracle_running_stats(case, sd0, x, torch.float64), _oracle_running_stats(case, sd0, x, torch.float32)
        bufs = dict(m.named_buffers())
        for k in stats:
            if torch.equal(s64[k], sd0[k].double()):
                assert torch.equal(bufs[k].cpu(), sd0[k]), f"{name} {k}: moved, the oracle's did not"
            else:
                _check(f"{name} {k}", bufs[k], s64[k], s32[k], failures)
    for k in stats:
        if not training:
            assert torch.equal(dict(m.named_buffers())[k].cpu(), sd0[k]), f"{name} {k}: moved in eval mode"

    missing = sorted(must_run - ran)
    assert not missing, f"{name}: the backward did not run {missing}; it ran {sorted(ran)}"
    assert not failures, "\n".join(failures)
    # last: in train mode it moves the running statistics once more; the batch statistics, and so the result, are the
    # same (up to the order of the double atomics that sum them)
    e_lp = _rel(m.log_prob(xd), lp)
    assert e_lp <= 1e-6, f"{name}: log_prob differs from the inverse + N(0, I) head by {e_lp:.3e}"


# ---- BatchNorm(+ReLU) at op level -----------------------------------------------------------------------------------
def _bn_inputs(B, H, seed, relu):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, H, generator=gen) * 1.5 + 0.3 * torch.randn(H, generator=gen)
    gamma = 1 + 0.3 * torch.randn(H, generator=gen)
    beta = 0.2 * torch.randn(H, generator=gen)
    rm = 0.3 * torch.randn(H, generator=gen)
    rv = torch.exp(0.3 * torch.randn(H, generator=gen))
    gy = torch.randn(B, H, generator=gen)
    return x, gamma, beta, rm, rv, gy


def _bn_ref(x, gamma, beta, rm, rv, gy, training, relu, dtype):
    """F.batch_norm (+ relu) autograd in `dtype` on the GPU: (y, gx, ggamma, gbeta, running_mean, running_var)."""
    xr = x.to(DEV, dtype).requires_grad_()
    g, b = gamma.to(DEV, dtype).requires_grad_(), beta.to(DEV, dtype).requires_grad_()
    rm_, rv_ = rm.to(DEV, dtype), rv.to(DEV, dtype)
    y = F.batch_norm(xr, rm_, rv_, g, b, training, 0.1, 1e-5)
    if relu:
        y = torch.relu(y)
    y.backward(gy.to(DEV, dtype))
    return y.detach(), xr.grad, g.grad, b.grad, rm_, rv_


def _away_from_relu_kink(x, gamma, beta, rm, rv, training):
    """Moves the few elements whose float64 pre-activation lies within 1e-4 |gamma| of 0 to 3e-4 |gamma| on the same
    side.  A float32 pre-activation there may round to the other side of the ReLU kink than the float64 one; that is
    rounding, not an error of the kernel, and it would add a whole gy term to gbeta."""
    xd = x.double()
    mu = xd.mean(0) if training else rm.double()
    var = xd.var(0, unbiased=False) if training else rv.double()
    rs = 1 / torch.sqrt(var + 1e-5)
    pre = (xd - mu) * rs * gamma.double() + beta.double()
    near = pre.abs() < 1e-4 * gamma.double().abs()
    side = torch.where(pre >= 0, 1.0, -1.0) * torch.sign(gamma.double())
    x = torch.where(near, (xd + side * 3e-4 / rs), xd).float()
    return x


BN_H = [4, 16, 30, 64, 512]
BN_B = [2, 255, 1024, 4099, 65536]


@pytest.mark.parametrize("relu", [True, False])
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("B", BN_B)
@pytest.mark.parametrize("H", BN_H)
def test_batchnorm_matches_float64(H, B, training, relu):
    """ops.batchnorm_relu (forward, gx, ggamma, gbeta, running statistics) against F.batch_norm in float64: the 128-bit
    kernels (H % 4 == 0, H >= 16) and the scalar ones, on ragged and tiny batches."""
    x, gamma, beta, rm, rv, gy = _bn_inputs(B, H, 1000 * H + B, relu)
    if relu:
        x = _away_from_relu_kink(x, gamma, beta, rm, rv, training)
    bn = torch.nn.BatchNorm1d(H).to(DEV)
    with torch.no_grad():
        bn.weight.copy_(gamma)
        bn.bias.copy_(beta)
        bn.running_mean.copy_(rm)
        bn.running_var.copy_(rv)
    bn.train(training)
    xd = x.to(DEV).requires_grad_()
    y = N.ops.batchnorm_relu(xd, bn, relu=relu)
    y.backward(gy.to(DEV))
    r64 = _bn_ref(x, gamma, beta, rm, rv, gy, training, relu, torch.float64)
    r32 = _bn_ref(x, gamma, beta, rm, rv, gy, training, relu, torch.float32)
    tag = f"bn H={H} B={B} {'train' if training else 'eval'} relu={int(relu)}"
    failures = []
    _check(f"{tag} y", y, r64[0], r32[0], failures)
    _check(f"{tag} gx", xd.grad, r64[1], r32[1], failures)
    if training:
        _check(f"{tag} running_mean", bn.running_mean, r64[4], r32[4], failures)
        _check(f"{tag} running_var", bn.running_var, r64[5], r32[5], failures)
    else:
        assert torch.equal(bn.running_mean.cpu(), rm) and torch.equal(bn.running_var.cpu(), rv)
    # the reductions, bounded by their condition sum |terms|; xhat comes from the float32 mean and rstd the forward saved,
    # so its rounding error is relative to |x - mean| + |mean| (in units of the standard deviation)
    y64 = r64[0]
    g_eff = gy.to(DEV, torch.float64) * ((y64 > 0) if relu else 1)
    xd64 = x.to(DEV, torch.float64)
    mu = xd64.mean(0) if training else rm.to(DEV, torch.float64)
    var = xd64.var(0, unbiased=False) if training else rv.to(DEV, torch.float64)
    xhat = (xd64 - mu) / torch.sqrt(var + 1e-5)
    xhat_size = xhat.abs() + (mu / torch.sqrt(var + 1e-5)).abs()
    for what, got, ref, terms in (("ggamma", bn.weight.grad, r64[2], g_eff * xhat_size), ("gbeta", bn.bias.grad, r64[3], g_eff)):
        scale = terms.abs().sum(0) + 1e-30
        worst = ((got.double() - ref).abs() / scale).max().item()
        print(f"  {tag} {what:<12s} max |g - g64| / sum|terms| = {worst:.3e}")
        if not worst <= RED_TOL:
            failures.append(f"{tag} {what}: {worst:.3e} > {RED_TOL:.1e} of sum|terms|")
    assert not failures, "\n".join(failures)


# ---- the re-masking invariant, bitwise ------------------------------------------------------------------------------
def _bits(t):
    return t.contiguous().view(torch.int32).cpu()


def _mask_edge_inputs(B, H, training):
    """Columns of {-1, 0, +1} (B/8 each of -1 and +1) with beta in {+-0, +-1 ulp of 0, +-min normal, +-1e-30}: the
    pre-activation of every 0 entry is exactly beta, a signed zero or the smallest float values on either side of the
    ReLU kink.  With eps = 0 the statistics are exact (mean 0, var 1/4, rstd 2 in train mode; running statistics
    0 and 1/4 in eval mode) and so are the backward's sums (dyadic gy), whatever their order: every run computes the
    same bits.  Eval mode adds a NaN in row 5 of the first NAN_COLS columns (ggamma is NaN there)."""
    gen = torch.Generator().manual_seed(B + H)
    col = torch.zeros(B)
    col[: B // 8] = 1.0
    col[B // 8: B // 4] = -1.0
    x = torch.stack([col[torch.randperm(B, generator=gen)] for _ in range(H)], dim=1)
    if not training:
        x[5, :NAN_COLS] = float("nan")
    tiny = torch.tensor([0.0, -0.0, 2.0 ** -149, -2.0 ** -149, 2.0 ** -126, -2.0 ** -126, 1e-30, -1e-30])
    beta = tiny.repeat(H // 8)
    gamma = torch.tensor([1.0, -1.0, 0.5, -2.0]).repeat_interleave(2).repeat(H // 8).roll(3)
    gy = torch.randint(-64, 65, (B, H), generator=gen).float() / 16
    return x, gamma, beta, gy


NAN_COLS = 8


@pytest.mark.parametrize("training", [True, False])
def test_batchnorm_relu_mask_rederivation_is_bitwise(training):
    """nf_batchnorm_forward writes the same y through the 128-bit apply kernel (y 16-byte aligned) and the scalar one
    (y at a 4-byte offset), and nf_batchnorm_backward computes the same gx, ggamma, gbeta bits whether its 128-bit
    kernels re-derive the ReLU mask from bn_affine(x) (beta given) or read it from y (beta = NULL)."""
    call, ptr, st, F32 = N._lib.call, N._lib.ptr, N._lib.stream, N._lib.NF_F32
    B, H = 4096, 64
    x, gamma, beta, gy = (t.to(DEV) for t in _mask_edge_inputs(B, H, training))
    rm = torch.zeros(H, device=DEV)
    rv = torch.full((H,), 0.25, device=DEV)
    sm, sr = torch.empty(H, device=DEV), torch.empty(H, device=DEV)
    ws = torch.empty(2 * H, dtype=torch.float64, device=DEV)

    def forward(y):
        rm_, rv_ = rm.clone(), rv.clone()          # train mode moves them: each pass gets its own copy
        call("nf_batchnorm_forward", ptr(x), ptr(gamma), ptr(beta), ptr(rm_), ptr(rv_), ptr(y), ptr(sm),
             ptr(sr), ptr(ws), B, H, int(training), 0.1, 0.0, 1, F32, st())

    y_al = torch.empty(B, H, device=DEV)
    ran_al = _traced(lambda: forward(y_al))[1]
    buf = torch.empty(B * H + 1, device=DEV)
    y_off = buf[1:].view(B, H)
    ran_off = _traced(lambda: forward(y_off))[1]
    assert "bn_apply_vec4_kernel" in ran_al and "bn_apply_kernel" in ran_off, (ran_al, ran_off)
    if training:
        assert torch.equal(sr.cpu(), torch.full((H,), 2.0)), "the statistics are not the exact ones the inputs encode"
    assert torch.equal(_bits(y_al), _bits(y_off)), "the two apply kernels wrote different y"
    assert (y_al == 0).any() and (y_al > 0).any() and (y_al[y_al > 0] < 1e-29).any()

    results = []
    for y in (y_al, y_off.clone()):                 # the copy is 16-byte aligned: the backward takes its 128-bit kernels
        for b in (beta, None):
            gx, gg, gb = torch.empty(B, H, device=DEV), torch.empty(H, device=DEV), torch.empty(H, device=DEV)
            ran = _traced(lambda: call("nf_batchnorm_backward", ptr(x), ptr(y), ptr(gamma), ptr(sm), ptr(sr), ptr(gy),
                                       ptr(gx), ptr(gg), ptr(gb), ptr(ws), B, H, 1, int(training), F32, ptr(b), st()))[1]
            assert VEC_BN <= ran, ran
            results.append((_bits(gx), _bits(gg), _bits(gb)))
    for r in results[1:]:
        for a, b, what in zip(results[0], r, ("gx", "ggamma", "gbeta")):
            assert torch.equal(a, b), f"{what} depends on where the backward takes its ReLU mask from"
    # none of the compared reductions is vacuous: ggamma is finite and not all zero outside the NaN columns, gbeta everywhere
    gg, gb = results[0][1].view(torch.float32), results[0][2].view(torch.float32)
    gg_clean = gg if training else gg[NAN_COLS:]
    assert torch.isfinite(gg_clean).all() and gg_clean.abs().sum() > 0
    assert torch.isfinite(gb).all() and gb.abs().sum() > 0
