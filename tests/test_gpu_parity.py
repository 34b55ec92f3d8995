"""GPU parity: the CUDA path (through the nn.Module surface -> ctypes -> C ABI -> sm_100a kernels) against
  * the committed golden vectors produced by the unmodified reference (tests/golden), and
  * the CPU oracle on seeded inputs.
Tolerances (north_star): z within 1e-5*max(1,|z|), row log-det within 1e-4 absolute; written at each assert."""
import json
import os
import re

import pytest
import torch

import nfb200 as N
from oracle import flows_oracle as O
from tests import golden_util as G
from tests.build_util import MODULE_KINDS, assert_close, build

pytestmark = pytest.mark.gpu

Z_ATOL, Z_RTOL = 1e-5, 1e-5      # fp32 z: |dz| <= 1e-5 * (1 + |z|)
LD_ATOL, LD_RTOL = 1e-4, 1e-5    # row log-det: 1e-4 absolute (+1e-5 relative for |ld| >> 1)

MODULE_CASES = [n for n in G.golden_names() if G.load(n)["kind"] in MODULE_KINDS]


def _dev():
    return torch.device("cuda:0")


def _run(m, x, inverse):
    return m.inverse(x) if inverse else m.forward(x)


def _loose(g):
    """stress rows drive the conditioners to 1e10-scale activations where fp32 GEMM summation order decides
    between saturated values; compare those rows only for NaN pattern / finiteness + clamped log-det"""
    x = g["x"]
    return (x.abs() > 50).any(dim=1) | ~torch.isfinite(x).all(dim=1)


_ORACLE64 = {}
_COND = {}


def _oracle64(g, name, inverse):
    """float64 oracle on the calm rows of a golden case (cached): the yardstick for how much of a deviation is
    the reference's own float32 rounding noise (SURVEY D10 / A.3)."""
    key = (name, inverse)
    if key not in _ORACLE64:
        calm = ~_loose(g)
        sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in g["sd"].items()}
        y, ld = G.oracle_eval(dict(g, sd=sd64, x=g["x"][calm].double()), inverse)
        _ORACLE64[key] = (y, torch.as_tensor(ld).expand(y.shape[0]))
    return _ORACLE64[key]


def _conditioning(g, name, inverse):
    """Per-element sensitivity of the float32 oracle to ~1-ulp relative noise on the weights (6 draws): what any
    implementation with a different GEMM summation order may legitimately differ by on that element."""
    key = (name, inverse)
    if key not in _COND:
        calm = ~_loose(g)
        x = g["x"][calm]
        y0, l0 = G.oracle_eval(dict(g, x=x), inverse)
        l0 = torch.as_tensor(l0).expand(y0.shape[0])
        gen = torch.Generator().manual_seed(0)
        cy, cl = torch.zeros_like(y0), torch.zeros_like(l0)
        for _ in range(6):
            sdp = {k: (v * (1 + 2e-7 * torch.randn(v.shape, generator=gen)) if v.is_floating_point() and "weight" in k
                       else v) for k, v in g["sd"].items()}
            y1, l1 = G.oracle_eval(dict(g, sd=sdp, x=x), inverse)
            cy = torch.maximum(cy, (y1 - y0).abs().nan_to_num(0.0))
            cl = torch.maximum(cl, (torch.as_tensor(l1).expand(l0.shape) - l0).abs().nan_to_num(0.0))
        _COND[key] = (cy.double(), cl.double())
    return _COND[key]


FALLBACK_LOG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "parity_fallbacks.jsonl")
MAX_FALLBACK_FRACTION = 1e-3     # at most 0.1 % of a comparison's elements (and never fewer than 2 allowed) may need a fallback clause


def _within(mine, ref32, ref64, atol, rtol, what, cond=None, terms=1):
    """Per-element clauses only:
      (1) strict      |mine-ref32| <= atol + rtol|ref32|                                       (north_star's bound)
      (2) fallback A  ill-conditioned element, i.e. the reference's own float32 result is already e_ref away from its
                      float64 result: |mine-ref64| <= atol + rtol|ref64| + 2*e_ref  (THIS element's e_ref);
      (3) fallback B  |mine-ref32| <= atol + rtol|ref32| + 2*c with c = THIS element's measured sensitivity of the
                      float32 oracle to 1-ulp weight noise (`cond`, a callable evaluated only when needed).
    The number of elements that needed (2) or (3) is printed, logged to gpurun_out/parity_fallbacks.jsonl and bounded:
    at most 0.1 % of the compared values -- times `terms` when a compared value is a sum of `terms` transformed
    elements (a row log-det over Dt dims meets an ill-conditioned element Dt times as often as a single element does)."""
    mine, ref32 = mine.double(), ref32.double()
    assert torch.equal(torch.isnan(mine), torch.isnan(ref32)), f"{what}: NaN pattern differs"
    strict = ((mine - ref32).abs() <= atol + rtol * ref32.abs()) | (mine == ref32) | torch.isnan(mine)   # equal infinities are equal
    e_ref = (ref32 - ref64).abs().nan_to_num(0.0, posinf=0.0)
    ok = strict | ((mine - ref64).abs() <= atol + rtol * ref64.abs() + 2 * e_ref)
    if not bool(ok.all()) and cond is not None:
        ok |= (mine - ref32).abs() <= atol + rtol * ref32.abs() + 2 * cond()
    n, n_fb = strict.numel(), int((ok & ~strict).sum())
    print(f"[parity] {what}: {n} elements, {n_fb} through a fallback clause, worst |mine-ref32| "
          f"{(mine - ref32).abs().nan_to_num(0.0, posinf=0.0).max().item() if n else 0.0:.3e}")
    try:
        os.makedirs(os.path.dirname(FALLBACK_LOG), exist_ok=True)
        with open(FALLBACK_LOG, "a") as f:
            f.write(json.dumps({"what": what, "elements": n, "terms": terms, "fallback": n_fb}) + "\n")
    except OSError:
        pass
    bad = ~ok
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())} elements off, worst |mine-ref32| "
                                 f"{(mine - ref32).abs()[bad].max().item():.3e}, reference's own fp32 error "
                                 f"max {e_ref.max().item():.3e}")
    assert n_fb <= max(2, int(MAX_FALLBACK_FRACTION * n * terms)), (
        f"{what}: {n_fb} of {n} values ({terms} term(s) each) pass only through a fallback clause")


def _compare(g, y, ld, key, tag, name):
    ref_y, ref_ld = g[key], torch.as_tensor(g[key + "_ld"])
    y, ld = y.detach().cpu(), ld.detach().cpu()
    if ref_ld.dim() == 0:
        ref_ld = ref_ld.expand(ld.shape)
    wild = _loose(g)
    calm = ~wild
    y64, ld64 = _oracle64(g, name, key == "inv")
    inv = key == "inv"
    _within(y[calm], ref_y[calm], y64, Z_ATOL, Z_RTOL, f"{tag} {key} z", lambda: _conditioning(g, name, inv)[0])
    _within(ld[calm], ref_ld[calm], ld64, LD_ATOL, LD_RTOL, f"{tag} {key} log_det",
            lambda: _conditioning(g, name, inv)[1])
    if wild.any():
        assert torch.equal(torch.isfinite(y[wild]), torch.isfinite(ref_y[wild])), f"{tag} {key} finiteness (stress rows)"
        assert torch.equal(torch.isfinite(ld[wild]), torch.isfinite(ref_ld[wild]))


@pytest.mark.parametrize("tensor_cores", [True, False])
@pytest.mark.parametrize("name", MODULE_CASES)
def test_fused_route_matches_reference_golden(name, tensor_cores, monkeypatch):
    """no_grad + eval: single-launch kernels (tcgen05 / FP32-pipe stacks, MADE chain, incremental sequential)."""
    monkeypatch.setattr(N.flows, "USE_TENSOR_CORES", tensor_cores)
    g = G.load(name)
    m = build(g).to(_dev())
    x = g["x"].to(_dev())
    before = N._lib.launch_count()
    with torch.no_grad():
        for inverse, key in ((False, "fwd"), (True, "inv")):
            y, ld = _run(m, x, inverse)
            _compare(g, y, ld, key, name + (" [fused tc]" if tensor_cores else " [fused simt]"), name)
    assert N._lib.launch_count() > before


def test_tensor_core_stack_is_taken_and_handles_ragged_batches():
    """config-2 shape through the tcgen05 kernel explicitly, at batch sizes around the 512-row tile."""
    g = G.load("splinestack_2_8_64_K8")
    m = build(g).to(_dev())
    pk = N.packing.pack_spline_stack_tc(list(m.flows), None)
    assert pk is not None
    gen = torch.Generator().manual_seed(3)
    for B in (1, 127, 128, 129, 511, 512, 513, 5000):
        x = (torch.randn(B, 2, generator=gen) * 1.5)
        for inverse in (False, True):
            out = N.ops.stack("nf_spline_stack_tc", pk[0], pk[1], x.to(_dev()), inverse)
            assert out is not None
            ry, rld = O.flow_model(g["sd"], "", [dict(kind="spline", num_bins=8)] * 8, x, inverse)
            sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in g["sd"].items()}
            y64, ld64 = O.flow_model(sd64, "", [dict(kind="spline", num_bins=8)] * 8, x.double(), inverse)
            _within(out[0].cpu(), ry, y64, Z_ATOL, Z_RTOL, f"tc stack B={B} z")
            _within(out[1].cpu(), rld, ld64, LD_ATOL, LD_RTOL, f"tc stack B={B} ld")


@pytest.mark.parametrize("name", MODULE_CASES)
def test_layered_route_matches_reference_golden(name):
    """grad enabled: conditioner GEMMs + BatchNorm + transform kernels, one autograd Function each."""
    g = G.load(name)
    m = build(g).to(_dev())
    x = g["x"].to(_dev()).requires_grad_()
    for inverse, key in ((False, "fwd"), (True, "inv")):
        y, ld = _run(m, x, inverse)
        assert y.requires_grad and ld.requires_grad
        _compare(g, y, ld, key, name + " [layered]", name)


@pytest.mark.parametrize("name", MODULE_CASES)
def test_float64_route_matches_float64_oracle(name):
    g = G.load(name)
    finite = torch.isfinite(g["x"]).all(dim=1) & (g["x"].abs() < 50).all(dim=1)
    x = g["x"][finite].double()
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in g["sd"].items()}
    g64 = dict(g, sd=sd64, x=x)
    m = build(g).double().to(_dev())
    with torch.no_grad():
        for inverse in (False, True):
            ry, rld = G.oracle_eval(g64, inverse)
            y, ld = _run(m, x.to(_dev()), inverse)
            assert y.dtype == torch.float64
            assert_close(y, ry, 1e-9, 1e-9, f"{name} f64 z inv={inverse}")
            # ARQS keeps its log-det in a float32 vector whatever the data dtype (arqs.py:52): one float32 ulp
            ld_atol, ld_rtol = (1e-6, 2e-7) if g["kind"] == "arqs" else (1e-8, 1e-9)
            assert ld.dtype == torch.as_tensor(rld).dtype
            assert_close(ld, torch.as_tensor(rld).expand(ld.shape), ld_atol, ld_rtol, f"{name} f64 ld inv={inverse}")


@pytest.mark.parametrize("name", G.golden_names("coupling_train"))
def test_train_mode_coupling_batch_statistics(name):
    """BatchNorm batch statistics + running-stat side effects (coupling_layer.py:20,23)."""
    g = G.load(name)
    m = build(g).to(_dev())
    m.train()
    with torch.no_grad():
        y, ld = m.forward(g["x"].to(_dev()))
    assert_close(y, g["fwd"], Z_ATOL, Z_RTOL, name + " z")
    assert_close(ld, g["fwd_ld"], LD_ATOL, LD_RTOL, name + " ld")
    after = m.state_dict()
    for k, v in g["sd_after"].items():
        if v.is_floating_point():
            assert_close(after[k], v, 1e-6, 1e-5, f"{name} {k}")
        else:
            assert torch.equal(after[k].cpu(), v), k


@pytest.mark.parametrize("name", G.golden_names("mafbn_train") + G.golden_names("iafbn_train"))
def test_train_mode_made_batch_norm(name):
    """MAF / IAF with use_batch_norm=True in train mode, parallel direction: batch statistics + running-stat updates."""
    g = G.load(name)
    m = build(g).to(_dev())
    m.train()
    with torch.no_grad():
        y, ld = m.inverse(g["x"].to(_dev())) if g["kind"] == "maf_train" else m.forward(g["x"].to(_dev()))
    assert_close(y, g["out"], Z_ATOL, Z_RTOL, name + " z")
    assert_close(ld, g["out_ld"], LD_ATOL, LD_RTOL, name + " ld")
    after = m.state_dict()
    for k, v in g["sd_after"].items():
        if v.is_floating_point():
            assert_close(after[k], v, 1e-6, 1e-5, f"{name} {k}")
        else:
            assert torch.equal(after[k].cpu(), v), k


def test_train_mode_between_layer_batchnorm():
    g = G.load("realnvp_4_4_16_bn_train")
    m = build(g).to(_dev())
    m.train()
    with torch.no_grad():
        y, ld = m.forward(g["x"].to(_dev()))
    assert_close(y, g["fwd"], Z_ATOL, Z_RTOL, "bn-train z")
    assert_close(ld, g["fwd_ld"], LD_ATOL, LD_RTOL, "bn-train ld")
    after = m.state_dict()
    for k, v in g["sd_after"].items():
        if v.is_floating_point():
            assert_close(after[k], v, 1e-6, 1e-5, k)
        else:
            assert torch.equal(after[k].cpu(), v), k


def _param_noise(fn, params, trials=6):
    """elementwise max deviation of fn(*params) under ~1-ulp relative noise on the spline parameters"""
    gen = torch.Generator().manual_seed(0)
    y0, l0 = fn(*params)
    cy, cl = torch.zeros_like(y0), torch.zeros_like(l0)
    for _ in range(trials):
        pp = [p * (1 + 2e-7 * torch.randn(p.shape, generator=gen)) for p in params]
        y1, l1 = fn(*pp)
        cy = torch.maximum(cy, (y1 - y0).abs().nan_to_num(0.0))
        cl = torch.maximum(cl, (l1 - l0).abs().nan_to_num(0.0))
    return cy.double().reshape(-1), cl.double().reshape(-1)


@pytest.mark.parametrize("name", G.golden_names("rqs_unit"))
def test_public_spline_function(name):
    g = G.load(name)
    d = _dev()
    for inverse, key in ((False, "fwd"), (True, "inv")):
        y, ld = N.rational_quadratic_spline(g["x"].to(d), g["w"].to(d), g["h"].to(d), g["d"].to(d), inverse=inverse)
        assert y.shape == g["x"].shape and ld.shape == g["x"].shape
        y64, l64 = O.rqs_unit(g["x"].double(), g["w"].double(), g["h"].double(), g["d"].double(), inverse)
        noise = lambda: _param_noise(lambda w, h, dd: O.rqs_unit(g["x"], w, h, dd, inverse), [g["w"], g["h"], g["d"]])
        _within(y.cpu(), g[key], y64, Z_ATOL, Z_RTOL, f"{name} {key} y", lambda: noise()[0])
        _within(ld.cpu(), g[key + "_ld"], l64, LD_ATOL, LD_RTOL, f"{name} {key} ld", lambda: noise()[1])


@pytest.mark.parametrize("name", [n for n in G.golden_names("spline_") if n.endswith("_rqs")])
def test_bounded_spline_transform_kernel(name):
    """a6 through the C ABI: every element its own row (D=1), so the row log-det is the element log-det."""
    g = G.load(name)
    K = g["K"]
    d = _dev()
    x = g["x"].reshape(-1, 1).to(d)
    params = torch.cat([g["uw"], g["uh"], g["ud"]], dim=-1).reshape(-1, 3 * K - 1).contiguous().to(d)
    mask = torch.zeros(1, device=d)
    tidx = torch.zeros(1, dtype=torch.int32, device=d)
    for inverse, key in ((False, "fwd"), (True, "inv")):
        y, ld = N.ops.spline_transform(x, params, mask, tidx, K, inverse, g["bound"], (1e-3, 1e-3, 1e-3))
        y64, l64 = O.rqs_bounded(g["x"].double(), g["uw"].double(), g["uh"].double(), g["ud"].double(), inverse)
        noise = lambda: _param_noise(lambda a, b, c: O.rqs_bounded(g["x"], a, b, c, inverse, bound=g["bound"]),
                                     [g["uw"], g["uh"], g["ud"]])
        _within(y.cpu().reshape(-1), g[key].reshape(-1), y64.reshape(-1), Z_ATOL, Z_RTOL, f"{name} {key} y",
                lambda: noise()[0])
        _within(ld.cpu().reshape(-1), g[key + "_ld"].reshape(-1), l64.reshape(-1), LD_ATOL, LD_RTOL,
                f"{name} {key} ld", lambda: noise()[1])


@pytest.mark.parametrize("D,K,B", [(2, 8, 200003), (16, 10, 40001), (5, 4, 150001)])
@pytest.mark.parametrize("compact", [True, False])
def test_spline_transform_large_batch(D, K, B, compact):
    """Forward transform kernels at large, ragged batch sizes (warp-transposed compact-layout kernel and the
    register-path kernel for the reference layout) against the oracle's bounded spline, alternating mask."""
    gen = torch.Generator().manual_seed(D * 100 + K)
    P = 3 * K - 1
    mask = torch.zeros(D)
    mask[::2] = 1
    tl = torch.nonzero(mask == 0).flatten()
    Dt = tl.numel()
    x = torch.randn(B, D, generator=gen) * 3
    full = torch.randn(B, D, P, generator=gen)
    par = (full[:, tl, :] if compact else full).reshape(B, -1).contiguous()
    d = _dev()
    tidx = tl.to(torch.int32).to(d)
    for inverse in (False, True):
        y, ld = N.ops.spline_transform(x.to(d), par.to(d), mask.to(d), tidx, K, inverse, 5.0, (1e-3, 1e-3, 1e-3), None,
                                       compact)
        uw, uh, ud = full[:, tl, :K], full[:, tl, K:2 * K], full[:, tl, 2 * K:]
        yt, lt = O.rqs_bounded(x[:, tl], uw, uh, ud, inverse, bound=5.0)
        y64, l64 = O.rqs_bounded(x[:, tl].double(), uw.double(), uh.double(), ud.double(), inverse, bound=5.0)
        ref = x.clone()
        ref[:, tl] = yt
        ref64 = x.double().clone()
        ref64[:, tl] = y64
        # 10^5..10^6 elements with randn(0, 1) raw parameters (far wilder than conditioner outputs): the per-element
        # sensitivity is measured under 1-ulp noise on the parameters AND the input, 16 draws
        xt = x[:, tl]
        noise = lambda: tuple(2 * t for t in _param_noise(lambda xx, a, b, c: O.rqs_bounded(xx, a, b, c, inverse, bound=5.0),
                                                          [xt, uw, uh, ud], 16))
        def ynoise():
            n = torch.zeros(B, D, dtype=torch.float64)
            n[:, tl] = noise()[0].reshape(B, Dt)
            return n
        _within(y.cpu(), ref, ref64, Z_ATOL, Z_RTOL, f"staged z inv={inverse}", ynoise)
        _within(ld.cpu(), lt.sum(1), l64.sum(1), LD_ATOL, LD_RTOL, f"staged ld inv={inverse}",
                lambda: noise()[1].reshape(B, Dt).sum(1), terms=Dt)


# the in-block kernel each layout reaches (ar_blocked.cu picks it from the block layout alone): whole 8-unit tiles of at
# most 16 units per degree -> mma.sync; degrees not padded to multiples of 4 (the padding would cost > 10 % more units)
# -> warp-private FP32 tiles; blocks of more than ~148 units (~34 per degree at MAF(16, 512)) -> CTA barriers
_IN_BLOCK_KERNEL = {(64, 512): "ar_block_mma_kernel", (32, 256): "ar_block_mma_kernel", (20, 128): "ar_block_warp_kernel",
                    (36, 288): "ar_block_mma_kernel", (12, 96): "ar_block_warp_kernel", (16, 512): "ar_block_kernel"}
# shapes the module's own blocked route takes, with a launch count the route exceeds (in-block kernels, pull and push
# products, finish; MAF(16, 512) has two blocks: 7 launches) and the one-launch kernel does not
_MODULE_BLOCKED_LAUNCHES = {(64, 512): 8, (32, 256): 8, (20, 128): 8, (16, 512): 6}


@pytest.mark.parametrize("kind,D,H,B", [("maf", 64, 512, 2048), ("iaf", 32, 256, 1500), ("maf", 20, 128, 1024),
                                       ("maf", 36, 288, 1001), ("iaf", 12, 96, 777),      # last block of 4 degrees; ragged row tiles
                                       ("maf", 16, 512, 1024)])
def test_blocked_sequential_direction_matches_oracle(kind, D, H, B):
    """MAF.forward / IAF.inverse through the blocked tensor-core evaluation (ar_blocked.cu) against the oracle's
    D-step loop and against the one-launch incremental kernel; the profiler confirms which in-block kernel ran."""
    sd = O.init_made_sd(D, H, seed=D + H, sigma=0.03, prefix="conditioner.")
    cls = N.MaskedAutoregressiveFlow if kind == "maf" else N.InverseAutoregressiveFlow
    m = cls(D, H)
    m.load_state_dict(sd, strict=True)
    m.to(_dev()).eval()
    gen = torch.Generator().manual_seed(B)
    v = torch.randn(B, D, generator=gen)
    v[3, 5] = float("nan")                     # poison: every later dim of that row must follow the dense reference
    v[7, D - 1] = float("inf")
    with torch.no_grad():
        ref_y, ref_ld = O.maf_forward(sd, "", v) if kind == "maf" else O.iaf_inverse(sd, "", v)
        folded = m.conditioner.folded()
        mode = N._lib.AR_MAF_FORWARD if kind == "maf" else N._lib.AR_IAF_INVERSE
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            blocked = N.ops.ar_sequential_blocked(v.to(_dev()), folded, mode)
            torch.cuda.synchronize()
        assert blocked is not None
        in_block = {hit.group(1) for e in prof.events()
                    for hit in [re.search(r"\b(ar_block(?:_mma|_warp)?_kernel)\b", e.name)] if hit}
        assert in_block == {_IN_BLOCK_KERNEL[(D, H)]}, in_block
        sd64 = {k: (t.double() if t.is_floating_point() else t) for k, t in sd.items()}
        y64, ld64 = (O.maf_forward(sd64, "", v.double())) if kind == "maf" else O.iaf_inverse(sd64, "", v.double())
        _within(blocked[0].cpu(), ref_y, y64, Z_ATOL, Z_RTOL, f"blocked {kind} z")
        _within(blocked[1].cpu(), ref_ld, ld64, LD_ATOL, LD_RTOL, f"blocked {kind} ld")
        # module entry point takes the blocked route at this size
        before = N._lib.launch_count()
        y2, ld2 = m.forward(v.to(_dev())) if kind == "maf" else m.inverse(v.to(_dev()))
        assert torch.equal(torch.isnan(y2), torch.isnan(blocked[0]))
        if (D, H) in _MODULE_BLOCKED_LAUNCHES:
            assert N._lib.launch_count() - before > _MODULE_BLOCKED_LAUNCHES[(D, H)]
            assert torch.allclose(y2.nan_to_num(), blocked[0].nan_to_num())
        else:                          # the added shapes are too small for the module's blocked route: the one-launch kernel
            _within(y2.cpu(), ref_y, y64, Z_ATOL, Z_RTOL, f"module route {kind} z")


def _randomised(m, seed, sigma):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(sigma * torch.randn(p.shape, generator=g))
        for n, b in m.named_buffers():
            if n.endswith("running_mean"):
                b.copy_(0.2 * torch.randn(b.shape, generator=g))
            elif n.endswith("running_var"):
                b.copy_(0.5 + torch.rand(b.shape, generator=g))
    return m


@pytest.mark.parametrize("kind,D,H,B", [("coupling", 8, 32, 700), ("coupling", 256, 512, 512), ("spline", 16, 64, 600),
                                        ("spline", 784, 1024, 300)])
def test_wide_eval_route_matches_oracle(kind, D, H, B):
    """Large data_dim, no autograd: cached mask / BatchNorm folds + TF32 splits, three tcgen05 GEMMs per conditioner
    (flows.py `_fold_wide`), against the oracle on the module's own state_dict; and against the layered route."""
    mask = torch.tensor([1.0 if i % 2 == 0 else 0.0 for i in range(D)])
    sigma = 0.3 / H ** 0.5
    if kind == "coupling":
        m = _randomised(N.CouplingLayer(D, H, mask), D + H, sigma)
    else:
        m = _randomised(N.SplineCouplingLayer(D, H, mask, num_bins=10), D + H, sigma)
    m.eval()
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    x = torch.randn(B, D, generator=torch.Generator().manual_seed(B)) * 1.5
    m = m.to(_dev())
    for inverse in (False, True):
        if kind == "coupling":
            ry, rld = O.affine_coupling(sd, "", x, inverse)
            y64, ld64 = O.affine_coupling(sd64, "", x.double(), inverse)
        else:
            ry, rld = O.spline_coupling(sd, "", x, inverse, num_bins=10)
            y64, ld64 = O.spline_coupling(sd64, "", x.double(), inverse, num_bins=10)
        with torch.no_grad():
            _run(m, x.to(_dev()), inverse)                                     # first call builds the cached folds
            before = N._lib.launch_count()
            y, ld = _run(m, x.to(_dev()), inverse)
        launches = N._lib.launch_count() - before
        assert launches <= (7 if kind == "coupling" else 4), launches          # 6 GEMMs + transform / 3 GEMMs + transform
        if H >= 1024:
            # 1024-long contractions: the short-chain tensor-core kernel (gemm_tc2.cu) keeps every TMEM accumulation chain at
            # 48 MMAs and folds chains with round-to-nearest adds; the single-chain kernel (384 truncating MMAs) showed a
            # coherent log-det bias of 4e-4 here (DESIGN.md).  SURVEY 8d's C4 bound: err <= 2 x err_ref32 + 1e-4.
            _within(y.cpu(), ry, y64, Z_ATOL, Z_RTOL, f"wide {kind} z inv={inverse}")
            e_ref = (rld.double() - ld64).abs().max().item()
            assert (ld.cpu().double() - ld64).abs().max().item() <= 2 * e_ref + 1e-4
            N.set_strict_fp32(True)                                            # FP32-pipe route: the same bound
            try:
                with torch.no_grad():
                    ys, lds = _run(m, x.to(_dev()), inverse)
            finally:
                N.set_strict_fp32(False)
            assert (lds.cpu().double() - ld64).abs().max().item() <= 2 * e_ref + 1e-4
            _within(ys.cpu(), ry, y64, Z_ATOL, Z_RTOL, f"strict {kind} z inv={inverse}")
        else:
            _within(y.cpu(), ry, y64, Z_ATOL, Z_RTOL, f"wide {kind} z inv={inverse}")
            _within(ld.cpu(), rld, ld64, LD_ATOL, LD_RTOL, f"wide {kind} ld inv={inverse}")
        yl, ldl = _run(m, x.to(_dev()).requires_grad_(), inverse)              # layered route, same module
        assert torch.allclose(yl, y, atol=2e-5, rtol=2e-5) and torch.allclose(ldl, ld, atol=3e-4, rtol=2e-5)
