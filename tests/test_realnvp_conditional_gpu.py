"""Conditional affine coupling flows, p(x | c), on the GPU against the float64 reference of
tests/conditional_affine_oracle.py.

A stack of CouplingLayer(context_dim = C) in eval mode inside the tcgen05 envelope (data_dim <= 8, hidden <= 128,
1 <= C <= 8) runs as one launch of coupling_stack_ctx_tc_kernel; CTX_KERNELS lists its instantiations and CASES states
which one each model must run.  Every case is checked four ways through the module -- forward, inverse, log_prob and
sample_and_log_prob -- against the reference in float32 and float64 (tests.test_gpu_parity._within), with one library
launch per fused call; and under torch.profiler (one trace per case) exactly the expected instantiation ran, in a process
of its own (tests/test_spline_conditional_gpu.py, _child, says why).  The conditioner BatchNorms carry perturbed running
statistics, so a pack that forgot to fold them into the context columns fails.
FALLBACK_CASES sit outside the envelope: no stack kernel runs and the layered route still matches.  Further tests tie the
conditional kernel to the unconditional one (zero context weights give identical outputs), pin the sampling layout and
the device generator, check the layered route's gradients and a model mixing conditional affine and spline layers.
test_library_ctx_kernels_match_the_table (no GPU) reads the library's symbols: an instantiation without a case fails."""
import json
import os
import subprocess
import sys
from dataclasses import dataclass

import pytest
import torch

import nfb200 as N
from oracle import flows_oracle as O
from tests import conditional_affine_oracle as CAO
from tests.test_gpu_parity import LD_ATOL, LD_RTOL, Z_ATOL, Z_RTOL, _within
from tests.test_gpu_published import _perturbed
from tests.test_gpu_stack_envelope import _KERNEL_RE, _tool
from tests.test_spline_conditional_gpu import _f64, _routes, _traced, _with_params

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CTX_KERNEL = "coupling_stack_ctx_tc_kernel"
# stack_tc.cu, coupling_stack_tc_launch<true>: DM 2 (D <= 2) / 4 (D = 3) / 8; HP 64 (H <= 64) / 128
_INST = [f"{CTX_KERNEL}<{dm}, {hp}" for dm in (2, 4, 8) for hp in (64, 128)]
CTX_KERNELS = [f"{k}, {s}>" for k in _INST for s in ("false", "true")]
assert len(CTX_KERNELS) == 12


@dataclass(frozen=True)
class Case:
    D: int
    H: int
    L: int
    C: int
    B: int
    kernel: object           # expected instantiation without the SAMPLE argument, or None (no stack kernel)
    bn: bool = False
    broadcast: bool = False  # context [1, C] instead of [B, C]
    train: bool = False      # train mode: conditioner BatchNorm on batch statistics (the layered route)
    f64: bool = False        # a float64 model (the layered route)


CASES = {
    "D2_H64_C4_bn": Case(2, 64, 8, 4, 65539, _INST[0], bn=True),
    "D1_H33_C8": Case(1, 33, 2, 8, 127, _INST[0]),
    "D2_H128_C8_broadcast": Case(2, 128, 4, 8, 4099, _INST[1], broadcast=True),
    "D2_H100_C1_bn_B1": Case(2, 100, 2, 1, 1, _INST[1], bn=True),
    "D3_H64_C1_broadcast": Case(3, 64, 2, 1, 4099, _INST[2], broadcast=True),
    "D3_H128_C4_bn": Case(3, 128, 2, 4, 4099, _INST[3], bn=True),
    "D5_H64_C8_bn": Case(5, 64, 2, 8, 4099, _INST[4], bn=True),
    "D8_H33_C1": Case(8, 33, 2, 1, 4099, _INST[4]),
    "D8_H100_C4_broadcast": Case(8, 100, 2, 4, 127, _INST[5], broadcast=True),
}
FALLBACK_CASES = {
    "hidden160": Case(2, 160, 2, 4, 4099, None, bn=True),
    "context9": Case(2, 64, 2, 9, 4099, None),
    "train": Case(2, 64, 2, 4, 50, None, train=True),
    "float64": Case(3, 64, 2, 4, 4099, None, bn=True, f64=True),
}
_claimed = {k for c in CASES.values() for k in (c.kernel + ", false>", c.kernel + ", true>")}
assert _claimed == set(CTX_KERNELS), sorted(set(CTX_KERNELS) - _claimed)


# ---- model, reference and inputs -----------------------------------------------------------------------------------
def _masks(c):
    first = [1.0] * (c.D // 2) + [0.0] * (c.D - c.D // 2)
    return [torch.tensor(first if i % 2 == 0 else [1.0 - v for v in first]) for i in range(c.L)]


def _model(c, seed, context_dim=None):
    torch.manual_seed(seed)
    C = c.C if context_dim is None else context_dim
    layers = [N.CouplingLayer(c.D, c.H, m, context_dim=C) for m in _masks(c)]
    model = _perturbed(N.NormalizingFlowModel(layers, batch_norm_between_layers=c.bn), seed)
    if c.train:
        model.train()
    if c.f64:
        model.double()
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    return model.to(DEV), sd, [dict(kind="affine")] * c.L


def _inputs(c, seed):
    """x with a few stress rows (NaN, +-Inf, 1e8) and a context whose own stress rows hold NaN / Inf (per-row context:
    in rows of their own, so that each meets a calm x)."""
    g = torch.Generator().manual_seed(seed)
    x = 1.5 * torch.randn(c.B, c.D, generator=g)
    ctx = torch.randn(1 if c.broadcast else c.B, c.C, generator=g)
    if c.B >= 64:
        for i, v in enumerate((float("nan"), float("inf"), -float("inf"), 1e8)):
            x[c.B - 1 - i] = v
        if not c.broadcast:
            ctx[c.B - 8, 0] = float("nan")
            ctx[c.B - 9, -1] = float("inf")
            ctx[c.B - 10, :] = -float("inf")
    dt = torch.float64 if c.f64 else torch.float32
    return x.to(dt), ctx.to(dt)


def _wild(x, ctx):
    bad = (x.abs() > 50).any(dim=1) | ~torch.isfinite(x).all(dim=1)
    return bad | ~torch.isfinite(ctx).all(dim=1).expand(x.shape[0])


def _compare(what, y, ld, ry, rld, y64, ld64, wild, D, L):
    y, ld = y.detach().cpu(), ld.detach().cpu()
    calm = ~wild
    _within(y[calm], ry[calm], y64[calm], Z_ATOL, Z_RTOL, f"{what} z", terms=L)
    _within(ld[calm], rld[calm], ld64[calm], LD_ATOL, LD_RTOL, f"{what} log_det", terms=D * L)
    if wild.any():
        assert torch.equal(torch.isfinite(y[wild]), torch.isfinite(ry[wild])), f"{what}: finiteness of z (stress rows)"
        assert torch.equal(torch.isfinite(ld[wild]), torch.isfinite(rld[wild])), f"{what}: finiteness of log_det"


def _setup(c, seed):
    """Model, reference inputs and the four calls of a case: forward, inverse, log_prob with the [B, C] (or [1, C])
    context, and sample_and_log_prob with m context rows (the per-row context's last rows, NaN / Inf ones included when
    there) of n samples each."""
    model, sd, specs = _model(c, seed)
    x, ctx = _inputs(c, seed)
    xd, cd = x.to(DEV), ctx.to(DEV)
    m = 1 if c.broadcast else min(c.B, 12)
    n = max(c.B // m, 1)
    cs = ctx[c.B - m:] if (not c.broadcast and c.B >= 64) else ctx[:m]

    def sample():
        gen = torch.Generator(device=DEV)
        gen.manual_seed(seed)
        return model.sample_and_log_prob(n, generator=gen, context=cs.to(DEV))
    calls = {"fwd": lambda: model.forward(xd, context=cd), "inv": lambda: model.inverse(xd, context=cd),
             "log_prob": lambda: model.log_prob(xd, context=cd), "sample": sample}
    return sd, specs, x, ctx, cs, m, n, calls


def _expected(c):
    fused = None if c.kernel is None else c.kernel + ", false>"
    return dict(fwd=fused, inv=fused, log_prob=fused, sample=None if c.kernel is None else c.kernel + ", true>")


def _ref(sd, specs, x, ctx, inverse, c):
    """The float32 and float64 reference of one direction (a float64 case: float64 both times)."""
    sd32 = sd if c.f64 else {k: (v.float() if v.is_floating_point() else v) for k, v in sd.items()}
    x32, c32 = (x, ctx) if c.f64 else (x.float(), ctx.float())
    ry, rld = CAO.flow_model(sd32, "", specs, x32, c32, inverse, bn_between=c.bn, training=c.train)
    y64, ld64 = CAO.flow_model(_f64(sd), "", specs, x.double(), ctx.double(), inverse, bn_between=c.bn, training=c.train)
    B = x.shape[0]
    return ry, torch.as_tensor(rld).expand(B), y64, torch.as_tensor(ld64).expand(B)


def _run_case(name, c, seed):
    sd, specs, x, ctx, cs, m, n, calls = _setup(c, seed)
    wild = _wild(x, ctx)
    out = {}
    with torch.no_grad():
        for call, fn in calls.items():
            fn()                                              # packs the weights
            torch.cuda.synchronize()
            before = N._lib.launch_count()
            out[call] = fn()
            torch.cuda.synchronize()
            if _expected(c)[call] is not None:
                assert N._lib.launch_count() - before == 1, f"{name} {call}: not one library launch"
    ref = {}
    for inverse, call in ((False, "fwd"), (True, "inv")):
        ref[call] = _ref(sd, specs, x, ctx, inverse, c)
        _compare(f"{name} {call}", *out[call], *ref[call], wild, c.D, c.L)

    rz, rld, z64, ld64 = ref["inv"]
    lp = out["log_prob"].cpu()
    calm = ~wild
    _within(lp[calm], (O.std_normal_log_prob(rz) + rld)[calm], (O.std_normal_log_prob(z64) + ld64)[calm], 2e-4, 1e-5,
            f"{name} log_prob", terms=c.D)
    if wild.any():
        assert torch.equal(torch.isfinite(lp[wild]), torch.isfinite(O.std_normal_log_prob(rz) + rld)[wild])

    xs, lq = out["sample"]
    assert xs.shape == (m, n, c.D) and lq.shape == (m, n)
    z = N.ops.std_normal_draw(seed, 0, m * n, c.D, torch.float32, torch.device(DEV)).cpu().to(x.dtype)
    crep = cs.repeat_interleave(n, 0)
    rx, rld, x64, ld64 = _ref(sd, specs, z, crep, False, c)
    lq32 = O.std_normal_log_prob(z) - rld
    lq64 = O.std_normal_log_prob(z.double()) - ld64
    calm = torch.isfinite(crep).all(dim=1)
    xs, lq = xs.reshape(m * n, c.D).cpu(), lq.reshape(m * n).cpu()
    _within(xs[calm], rx[calm], x64[calm], Z_ATOL, Z_RTOL, f"{name} sample x", terms=c.L)
    _within(lq[calm], lq32[calm], lq64[calm], 2e-4, 1e-5, f"{name} sample log_q", terms=c.D * c.L)
    if not calm.all():
        assert torch.equal(torch.isfinite(xs[~calm]), torch.isfinite(rx[~calm])), f"{name} sample stress rows"


def _route_report():
    """Every case's four calls under the profiler: name -> (stack kernels in call order, library launches per call)."""
    report = {}
    for name, c in list(CASES.items()) + list(FALLBACK_CASES.items()):
        calls = _setup(c, sum(map(ord, name)))[-1]
        with torch.no_grad():
            _, ran, launches = _traced(calls)
        report[name] = (ran, launches)
    return report


def _run_named(name):
    _run_case(name, CASES.get(name) or FALLBACK_CASES[name], seed=sum(map(ord, name)))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_conditional_stack_matches_float64_reference(name):
    _run_named(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FALLBACK_CASES))
def test_outside_the_envelope_no_stack_kernel_runs(name):
    _run_named(name)


def _child(fn, *args):
    """Run tests.test_realnvp_conditional_gpu.<fn>(*args) in a new interpreter; its JSON result follows 'RESULT=' (the
    reason is in tests/test_spline_conditional_gpu.py, _child)."""
    code = (f"import json, sys; from tests.test_realnvp_conditional_gpu import {fn}; "
            f"print('RESULT=' + json.dumps({fn}(*json.loads(sys.argv[1]))))")
    argv = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code, json.dumps(args)]
    return subprocess.run(argv, capture_output=True, text=True, cwd=ROOT)


def _in_child(fn, *args):
    r = _child(fn, *args)
    assert r.returncode == 0, f"{fn}{args} failed in its process:\n" + r.stdout[-4000:] + r.stderr[-6000:]
    return json.loads(next(l for l in r.stdout.splitlines() if l.startswith("RESULT="))[len("RESULT="):])


@pytest.mark.gpu
def test_routes_under_the_profiler():
    """Under torch.profiler, each case's forward / inverse / log_prob run exactly the expected instantiation and its
    sampling call the SAMPLE twin, one library launch each; outside the envelope no stack kernel runs."""
    report = _in_child("_route_report")
    assert set(report) == set(CASES) | set(FALLBACK_CASES)
    for name, (ran, launches) in report.items():
        c = CASES.get(name) or FALLBACK_CASES[name]
        _routes(name, _expected(c), ran, launches)


def test_library_ctx_kernels_match_the_table():
    """The library's conditional affine stack-kernel entry symbols are exactly CTX_KERNELS."""
    lib, cuobjdump, cxxfilt = N._lib.LIB_PATH, _tool("cuobjdump"), _tool("c++filt")
    if not os.path.exists(lib) or cuobjdump is None or cxxfilt is None:
        pytest.skip("needs the built library, cuobjdump and c++filt")
    out = subprocess.run([cuobjdump, "-symbols", lib], capture_output=True, text=True, check=True).stdout
    mangled = [line.split()[-1] for line in out.splitlines() if "STO_ENTRY" in line]
    names = subprocess.run([cxxfilt], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    found = {f"{m.group(1)}<{m.group(2)}>" for line in names.splitlines()
             for m in [_KERNEL_RE.search(line)] if m and m.group(1) == CTX_KERNEL}
    assert found == set(CTX_KERNELS), (f"in the library, not in the table: {sorted(found - set(CTX_KERNELS))}; "
                                       f"in the table, not in the library: {sorted(set(CTX_KERNELS) - found)}")


# ---- the conditional kernel against the unconditional one ----------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["D2_H64_C4_bn", "D2_H128_C8_broadcast", "D3_H128_C4_bn", "D5_H64_C8_bn"])
def test_zero_context_weights_give_the_unconditional_outputs(name):
    """With its context columns zeroed, a conditional model computes bit for bit what the unconditional model with the
    remaining weights computes (coupling_stack_tc_kernel): same x FMAs in the same order, the context's only adding
    exact zeros."""
    c = CASES[name]
    cond, sd, _ = _model(c, 1)
    plain, _, _ = _model(c, 1, context_dim=0)
    with torch.no_grad():
        for f in cond.flows:
            f.s_net[0].weight[:, c.D:] = 0
            f.b_net[0].weight[:, c.D:] = 0
        sd0 = {k: (v[:, :c.D] if k.endswith("net.0.weight") else v) for k, v in cond.state_dict().items()}
        plain.load_state_dict(sd0)
        x, _ = _inputs(c, 2)
        ctx = torch.randn(c.B, c.C)                       # finite: 0 * NaN would not be 0
        xd, cd = x.to(DEV), ctx.to(DEV)
        for a, b in ((cond.forward(xd, context=cd), plain.forward(xd)), (cond.inverse(xd, context=cd), plain.inverse(xd))):
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        assert torch.equal(cond.log_prob(xd, context=cd), plain.log_prob(xd))
        g1, g2 = torch.Generator(device=DEV).manual_seed(9), torch.Generator(device=DEV).manual_seed(9)
        xs, lq = cond.sample_and_log_prob(c.B, generator=g1, context=cd[:1])
        xp, lp = plain.sample_and_log_prob(c.B, generator=g2)
        assert torch.equal(xs[0], xp) and torch.equal(lq[0], lp)


# ---- sampling ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
def test_sample_is_forward_of_the_same_draw(fused):
    """sample_and_log_prob(n, context=c) with m rows: row r of the flat draw is conditioned on context row r // n.  It
    equals forward on the same draw with c.repeat_interleave(n, 0), then the log-q head.  fused=False: hidden 160,
    outside the kernel's envelope (the layered route)."""
    c = CASES["D2_H64_C4_bn"] if fused else FALLBACK_CASES["hidden160"]
    model, _, _ = _model(c, 4)
    m, n = 5, 1001
    cs = torch.randn(m, c.C, device=DEV)
    with torch.no_grad():
        gen = torch.Generator(device=DEV).manual_seed(11)
        xs, lq = model.sample_and_log_prob(n, generator=gen, context=cs)
        assert xs.shape == (m, n, c.D) and lq.shape == (m, n)
        z = N.ops.std_normal_draw(11, 0, m * n, c.D, torch.float32, torch.device(DEV))
        xf, ld = model.forward(z, context=cs.repeat_interleave(n, 0))
        assert torch.equal(xs.reshape(m * n, c.D), xf)
        torch.testing.assert_close(lq.reshape(m * n), N.ops.std_normal_log_q(z, ld), atol=2e-5, rtol=1e-6)
        x2 = model.sample(n, context=cs)
        assert x2.shape == (m, n, c.D) and torch.isfinite(x2).all()


@pytest.mark.gpu
def test_device_generator_capture_draws_new_samples():
    """Captured in a CUDA graph with a DeviceGenerator, the conditional sampling launch draws new samples on every
    replay, equal to the host-key call at the offset it read, and the offset moves on by 4 per replay."""
    model = _perturbed(N.RealNVP(2, 10, 128, context_dim=4), 5).to(DEV)
    cs = torch.randn(3, 4, device=DEV)
    g = N.DeviceGenerator(DEV, seed=21)
    with torch.no_grad():
        model.sample_and_log_prob(1000, generator=g, context=cs)       # warm-up outside the capture
        assert g.get_offset() == 4
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            x, lq = model.sample_and_log_prob(1000, generator=g, context=cs)
        assert g.get_offset() == 4                                       # capture records the draw, it does not run it
        seen = []
        for i in range(3):
            graph.replay()
            torch.cuda.synchronize()
            assert g.get_offset() == 8 + 4 * i
            seen.append(x.clone())
            gen = torch.Generator(device=DEV).manual_seed(21)
            gen.set_offset(4 + 4 * i)
            xe, lqe = model.sample_and_log_prob(1000, generator=gen, context=cs)
            assert torch.equal(x, xe) and torch.equal(lq, lqe)
        assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])


# ---- gradients on the layered route --------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("broadcast", [False, True])
def test_gradcheck_float64(broadcast, train):
    """torch.autograd.gradcheck of log_prob with respect to x, the context and every parameter of a small conditional
    RealNVP in float64 (the layered route: linear_ctx without its ReLU, then the conditioner BatchNorm on running
    statistics, or in train mode on the batch's)."""
    torch.manual_seed(0)
    model = _perturbed(N.RealNVP(3, 2, 8, batch_norm_between_layers=True, context_dim=3), 3).double().to(DEV)
    if train:
        for mod in model.modules():
            if isinstance(mod, torch.nn.BatchNorm1d) and mod not in list(model.flow.batch_norms):
                mod.train()
    names = [k for k, _ in model.named_parameters()]
    params = [p.detach().clone().requires_grad_() for _, p in model.named_parameters()]
    x = (0.7 * torch.randn(6, 3, dtype=torch.float64, device=DEV)).requires_grad_()
    c = torch.randn(1 if broadcast else 6, 3, dtype=torch.float64, device=DEV, requires_grad=True)
    fn = lambda x, c, *ps: _with_params(model, names, ps, lambda: model.log_prob(x, context=c))
    assert torch.autograd.gradcheck(fn, (x, c, *params), eps=1e-6, atol=1e-5, rtol=1e-4)


@pytest.mark.gpu
def test_float32_training_step_matches_float64_reference():
    """One NLL step at 65 536 rows in train mode (conditioner BatchNorm on batch statistics, the layered route): the loss,
    the input and context gradients and every parameter gradient against float64 autograd of the reference, with the
    normwise bound of tests/test_gpu_train_gradients.py.  The seed is 8: with seed 7, one of the 4.2 M first-layer
    BatchNorm outputs of flows.2.b_net lies 1.8e-8 from the ReLU kink and lands on the other side in float32 (float64
    input to that layer matched to 2.7e-7), which alone moves that net's first-layer gradients by 5e-4."""
    from tests.test_gpu_train_gradients import _check
    c = Case(2, 64, 8, 4, 65536, None, bn=True, train=True)
    model, sd, specs = _model(c, 8)
    g = torch.Generator().manual_seed(8)
    x = 1.5 * torch.randn(c.B, c.D, generator=g)
    ctx = torch.randn(c.B, c.C, generator=g)
    xd, cd = x.to(DEV).requires_grad_(), ctx.to(DEV).requires_grad_()
    before = N._lib.launch_count()
    loss = -model.log_prob(xd, context=cd).mean()
    loss.backward()
    assert N._lib.launch_count() > before

    def ref(dtype):
        sdr = {k: (v.to(dtype).requires_grad_() if v.is_floating_point() and "running" not in k else v.to(dtype)
                   if v.is_floating_point() else v) for k, v in sd.items()}
        xr, cr = x.to(dtype).requires_grad_(), ctx.to(dtype).requires_grad_()
        z, ld = CAO.flow_model(sdr, "", specs, xr, cr, True, bn_between=c.bn, training=True)
        lr = -(O.std_normal_log_prob(z) + ld).mean()
        lr.backward()
        return lr, xr.grad, cr.grad, {k: v.grad for k, v in sdr.items() if isinstance(v, torch.Tensor) and v.requires_grad}
    l64, gx64, gc64, gp64 = ref(torch.float64)
    l32, gx32, gc32, gp32 = ref(torch.float32)
    failures = []
    _check("loss", loss.detach().reshape(1), l64.reshape(1), l32.reshape(1), failures)
    _check("x.grad", xd.grad, gx64, gx32, failures)
    _check("context.grad", cd.grad, gc64, gc32, failures)
    for k, p in model.named_parameters():
        if p.grad is None:                        # the last between-layer BatchNorm: no layer follows it
            assert gp64[k] is None, k
            continue
        _check(k + ".grad", p.grad, gp64[k], gp32[k], failures)
    assert not failures, "\n".join(failures)


# ---- a model of conditional affine and spline layers ---------------------------------------------------------------
@pytest.mark.gpu
def test_mixed_affine_and_spline_model_matches_the_reference():
    """NormalizingFlowModel of alternating conditional CouplingLayers and SplineCouplingLayers reading one context: the
    layers run one by one (each conditional layer on its own one-launch route) and match the reference."""
    torch.manual_seed(3)
    D, C, B = 2, 4, 4099
    masks = [torch.tensor([1.0, 0.0]) if i % 2 == 0 else torch.tensor([0.0, 1.0]) for i in range(4)]
    layers = [N.CouplingLayer(D, 64, m, context_dim=C) if i % 2 == 0 else
              N.SplineCouplingLayer(D, 64, m, num_bins=8, context_dim=C) for i, m in enumerate(masks)]
    model = _perturbed(N.NormalizingFlowModel(layers, batch_norm_between_layers=True), 3)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    specs = [dict(kind="affine") if i % 2 == 0 else dict(kind="spline", num_bins=8) for i in range(4)]
    model = model.to(DEV)
    g = torch.Generator().manual_seed(4)
    x, ctx = 1.5 * torch.randn(B, D, generator=g), torch.randn(B, C, generator=g)
    c = Case(D, 64, 4, C, B, None, bn=True)
    with torch.no_grad():
        lp = model.log_prob(x.to(DEV), context=ctx.to(DEV)).cpu()
        for inverse in (False, True):
            y, ld = model.inverse(x.to(DEV), context=ctx.to(DEV)) if inverse else model.forward(x.to(DEV), context=ctx.to(DEV))
            _compare(f"mixed {'inv' if inverse else 'fwd'}", y, ld, *_ref(sd, specs, x, ctx, inverse, c),
                     torch.zeros(B, dtype=torch.bool), D, 4)
    rz, rld, z64, ld64 = _ref(sd, specs, x, ctx, True, c)
    _within(lp, O.std_normal_log_prob(rz) + rld, O.std_normal_log_prob(z64) + ld64, 2e-4, 1e-5, "mixed log_prob", terms=D)
