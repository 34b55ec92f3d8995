"""GPU: sample_and_log_prob.  Every route -- the in-kernel draw of the fused stacks, the bf16 chain, and draw + forward
+ log-q head -- returns x == forward(z)[0] bit for bit for the z of the N(0, I) stream at the same (seed, offset), and
log_q == log N(z) - log_det; the stream's statistics; gradients; train-mode side effects; other bases; launch counts."""
import math

import numpy as np
import pytest
import torch
from torch import distributions as td

import nfb200 as N

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LOG2PI = math.log(2 * math.pi)


def _perturbed(m, sigma, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(sigma * torch.randn(p.shape, generator=g, dtype=p.dtype))
    return m


def _bn_stats(m, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for bn in m.modules():
            if isinstance(bn, torch.nn.BatchNorm1d):
                bn.running_mean.add_(0.2 * torch.randn(bn.running_mean.shape, generator=g))
                bn.running_var.mul_(1 + 0.3 * torch.rand(bn.running_var.shape, generator=g))
    return m


def draw(seed, offset, n, D, dtype=torch.float32):
    return N.ops.std_normal_draw(seed, offset, n, D, dtype, torch.device(DEV))


def _spline_model(D, L, H, K, bn=False):
    masks = [torch.tensor([1. if (d < D // 2) == (i % 2 == 0) else 0. for d in range(D)]) for i in range(L)]
    return N.NormalizingFlowModel([N.SplineCouplingLayer(D, H, m, num_bins=K) for m in masks], batch_norm_between_layers=bn)


def check_route(model, n, D, gen_seed=123):
    """sample_and_log_prob against forward(draw) at the same (seed, offset); returns (library launches of the call,
    library launches of forward alone)."""
    dtype = next(model.parameters()).dtype
    with torch.no_grad():                       # the first call builds the packed / folded weights (launches of its own)
        model.sample_and_log_prob(n)
        model.forward(draw(0, 0, n, D, dtype))
    gen = torch.Generator(device=DEV)
    gen.manual_seed(gen_seed)
    seed, off = gen.initial_seed(), gen.get_offset()
    torch.cuda.synchronize()
    c0 = N._lib.launch_count()
    with torch.no_grad():
        x, lq = model.sample_and_log_prob(n, generator=gen)
    torch.cuda.synchronize()
    launches = N._lib.launch_count() - c0
    assert gen.get_offset() == off + 4
    z = draw(seed, off, n, D, dtype)
    c1 = N._lib.launch_count()
    with torch.no_grad():
        xr, ld = model.forward(z)
    torch.cuda.synchronize()
    fwd = N._lib.launch_count() - c1
    assert x.shape == (n, D) and lq.shape == (n,) and x.dtype == dtype and lq.dtype == dtype
    assert torch.equal(x, xr), f"max |x - forward(z)| {(x - xr).abs().max().item():.3e}"
    ref = -0.5 * (z.double() ** 2).sum(1) - 0.5 * D * LOG2PI - ld.double()
    err = (lq.double() - ref).abs() - 1e-5 * (1 + ref.abs())
    assert bool((err <= 0).all()), f"log_q exceeds 1e-5 (1 + |log_q|) by {err.max().item():.3e}"
    return launches, fwd


# ---- fused families: one launch ------------------------------------------------------------------------------------
FUSED = {
    "spline_tc_D2": lambda: _spline_model(2, 8, 64, 8),
    "spline_tc_D2_K10": lambda: N.RealNVPSpline(2, 4, 64),
    "spline_fp32pipe_D6": lambda: _spline_model(6, 4, 32, 8),
    "spline_fp32pipe_D8_K10": lambda: _spline_model(8, 4, 64, 10),
    "spline_tc_bn": lambda: _bn_stats(_spline_model(2, 4, 64, 8, bn=True), 5),
    "coupling_tc_H64": lambda: N.RealNVP(2, 8, 64),
    "coupling_tc_H128": lambda: N.RealNVP(2, 10, 128),
    "coupling_tc_D8_bn": lambda: _bn_stats(N.RealNVP(8, 4, 64, batch_norm_between_layers=True), 6),
    "iaf_stack": lambda: N.NormalizingFlowModel([N.InverseAutoregressiveFlow(2, 64) for _ in range(6)]),
    "maf_stack": lambda: N.NormalizingFlowModel([N.MaskedAutoregressiveFlow(2, 64) for _ in range(6)]),
    "iaf_stack_D5_bn": lambda: _bn_stats(N.NormalizingFlowModel([N.InverseAutoregressiveFlow(5, 32) for _ in range(4)],
                                                                batch_norm_between_layers=True), 7),
    "sequential_coupling": lambda: N.SequentialFlow([N.CouplingLayer(2, 64, torch.tensor([float(i % 2), 1. - i % 2]))
                                                     for i in range(4)]),
    "single_spline_layer": lambda: N.SplineCouplingLayer(2, 64, torch.tensor([1., 0.]), num_bins=8),
    "single_coupling_layer": lambda: N.CouplingLayer(4, 64, torch.tensor([1., 1., 0., 0.])),
}


@pytest.mark.parametrize("name", sorted(FUSED))
@pytest.mark.parametrize("n", [5000, 70001])
def test_fused_stack_route_identity_one_launch(name, n):
    model = _perturbed(FUSED[name](), 0.05, 1).to(DEV).eval()
    D = N.flows._event_dim(model)
    launches, fwd = check_route(model, n, D)
    assert fwd == 1 and launches == 1


def test_fp32_pipe_coupling_stack():
    old = N.flows.USE_TENSOR_CORES
    N.flows.USE_TENSOR_CORES = False
    try:
        for model in (N.RealNVP(2, 6, 64), N.RealNVP(4, 4, 128)):
            model = _perturbed(model, 0.05, 2).to(DEV).eval()
            launches, fwd = check_route(model, 9000, N.flows._event_dim(model))
            assert fwd == 1 and launches == 1
    finally:
        N.flows.USE_TENSOR_CORES = old


# ---- routes without an in-kernel draw: draw + forward + head --------------------------------------------------------
def test_unfused_routes():
    m = torch.tensor([1., 1., 0., 0.])
    cases = [
        (N.InverseAutoregressiveFlow(64, 512), 4096, 0.02),
        (N.MaskedAutoregressiveFlow(64, 512), 2048, 0.02),                 # blocked sequential direction
        (N.ARQS(4, 32, num_bins=8), 3000, 0.05),
        (N.SequentialFlow([N.CouplingLayer(4, 32, m), N.InverseAutoregressiveFlow(4, 32),
                           N.SplineCouplingLayer(4, 32, 1 - m, num_bins=6)]), 3001, 0.05),
        (N.RealNVP(2, 4, 16).double(), 2500, 0.05),                        # float64 widens the float32 draw
    ]
    for model, n, sigma in cases:
        model = _perturbed(model, sigma, 3).to(DEV).eval()
        launches, fwd = check_route(model, n, N.flows._event_dim(model))
        assert launches == fwd + 2, (type(model).__name__, launches, fwd)


def test_iaf_bf16_chain_two_launches():
    model = _perturbed(N.InverseAutoregressiveFlow(64, 512), 0.02, 4).to(DEV).eval()
    N.set_gemm_precision("bf16")
    try:
        launches, fwd = check_route(model, 8192, 64)
        assert fwd == 1 and launches == 2
    finally:
        N.set_gemm_precision("fp32")


@pytest.mark.parametrize("n", [0, 1, 127, 513])
def test_small_and_ragged_row_counts(n):
    for model in (_perturbed(_spline_model(2, 8, 64, 8), 0.05, 1), _perturbed(N.RealNVP(2, 10, 128), 0.05, 1),
                  _perturbed(N.InverseAutoregressiveFlow(3, 16), 0.05, 1)):
        model = model.to(DEV).eval()
        if n == 0:
            with torch.no_grad():
                x, lq = model.sample_and_log_prob(0)
            assert x.shape == (0, N.flows._event_dim(model)) and lq.shape == (0,)
        else:
            check_route(model, n, N.flows._event_dim(model))


# ---- consistency with the density --------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", ["c1", "c2"])
def test_log_q_agrees_with_log_prob(cfg):
    if cfg == "c1":
        model, n = _perturbed(N.RealNVP(2, 8, 64), 0.05, 1), 5000
    else:
        model, n = _perturbed(_spline_model(2, 8, 64, 8), 0.05, 2), 1 << 20
    model = model.to(DEV).eval()
    torch.manual_seed(0)
    with torch.no_grad():
        x, lq = model.sample_and_log_prob(n)
        lp = model.log_prob(x)
    d = (lq.double() - lp.double()).abs()
    assert bool(torch.isfinite(d).all())
    q999 = float(torch.quantile(d.float().cpu()[:: max(1, n // 200000)], 0.999))
    assert q999 <= 1e-4 and d.max().item() <= 1e-2, (q999, d.max().item())


# ---- the stream ------------------------------------------------------------------------------------------------------
def test_prefix_seed_and_offset_behaviour():
    model = _perturbed(_spline_model(2, 8, 64, 8), 0.05, 1).to(DEV).eval()
    z1, z2 = draw(99, 8, 1000, 5), draw(99, 8, 100000, 5)
    assert torch.equal(z1, z2[:1000])
    with torch.no_grad():
        torch.manual_seed(7)
        a = model.sample_and_log_prob(3000)
        b = model.sample_and_log_prob(3000)
        torch.manual_seed(7)
        c = model.sample_and_log_prob(3000)
        torch.manual_seed(7)
        small = model.sample_and_log_prob(1000)
    assert torch.equal(a[0], c[0]) and torch.equal(a[1], c[1])
    assert not torch.equal(a[0], b[0])
    assert torch.equal(small[0], a[0][:1000])


def test_draw_matches_numpy_box_muller():
    from tests.test_hostcheck_rng import box_muller64, py_philox, ulp_err, KEY_XOR, MASK
    seed, offset, D = 0xDEADBEEF12345, 4 * 77, 6
    z = draw(seed, offset, 64, D).cpu().numpy()
    key = ((seed & MASK) ^ KEY_XOR, seed >> 32)
    for r in range(64):
        w = np.array(py_philox([0, r, offset // 4, 0], key) + py_philox([1, r, offset // 4, 0], key), dtype=np.uint32)
        c, s = box_muller64(w[0::2], w[1::2])
        ref = np.stack([c, s], axis=1).reshape(-1)[:D]
        assert ulp_err(z[r], ref).max() <= 4


def test_moments_ks_and_correlations():
    from scipy import stats
    n = 1 << 24
    z = draw(2024, 0, n // 4, 4).reshape(-1).double()
    m, v = z.mean().item(), z.var().item()
    c = z - m
    skew = (c ** 3).mean().item() / v ** 1.5
    kurt = (c ** 4).mean().item() / v ** 2 - 3
    assert abs(m) <= 5 / math.sqrt(n) and abs(v - 1) <= 5 * math.sqrt(2 / n)
    assert abs(skew) <= 5 * math.sqrt(6 / n) and abs(kurt) <= 5 * math.sqrt(24 / n)
    p = stats.kstest(z[: 1 << 20].cpu().numpy(), "norm").pvalue
    assert p > 1e-3, p
    # dims of a row, adjacent rows, and torch.randn from the same generator state
    rows = 1 << 20
    zz = draw(5, 0, rows, 8).double()
    lim = 5 / math.sqrt(rows)
    cc = torch.corrcoef(zz.T)
    assert (cc - torch.eye(8, dtype=cc.dtype, device=cc.device)).abs().max().item() < lim
    adj = torch.corrcoef(torch.stack([zz[:-1, 3], zz[1:, 3]]))[0, 1].item()
    assert abs(adj) < lim
    gen = torch.Generator(device=DEV)
    gen.manual_seed(31)
    off = gen.get_offset()
    mine = draw(gen.initial_seed(), off, rows, 2).double()
    gen.set_offset(off)
    theirs = torch.randn(rows, 2, generator=gen, device=DEV).double()
    for d in range(2):
        assert abs(torch.corrcoef(torch.stack([mine[:, d], theirs[:, d]]))[0, 1].item()) < lim


# ---- gradients ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["iaf", "spline"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_reparameterised_gradient(kind, dtype):
    torch.manual_seed(3)
    base = N.InverseAutoregressiveFlow(4, 32) if kind == "iaf" else N.RealNVPSpline(2, 4, 32)
    model = _perturbed(base, 0.05, 4).to(DEV, dtype).train()
    twin = _perturbed(N.InverseAutoregressiveFlow(4, 32) if kind == "iaf" else N.RealNVPSpline(2, 4, 32), 0.05, 4)
    twin = twin.to(DEV).double().train()
    twin.load_state_dict({k: v.double() for k, v in model.state_dict().items()})
    D = N.flows._event_dim(model)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(11)
    seed, off = gen.initial_seed(), gen.get_offset()
    x, lq = model.sample_and_log_prob(2048, generator=gen)
    assert lq.requires_grad
    lq.mean().backward()
    z = draw(seed, off, 2048, D).double()
    xr, ld = twin.forward(z)
    (-0.5 * (z ** 2).sum(1) - 0.5 * D * LOG2PI - ld).mean().backward()
    for (name, p), q in zip(model.named_parameters(), twin.parameters()):
        g, gr = p.grad.double(), q.grad
        tol = 1e-9 * (1 + gr.abs()) if dtype == torch.float64 else 1e-5 * (gr.abs().max() + 1e-6)
        assert bool(((g - gr).abs() <= tol).all()), (name, (g - gr).abs().max().item())


# ---- semantics ---------------------------------------------------------------------------------------------------------
def test_train_mode_batchnorm_moves_running_stats_like_forward():
    a = _perturbed(N.RealNVPSpline(2, 4, 32, batch_norm_between_layers=True), 0.05, 5).to(DEV).train()
    b = _perturbed(N.RealNVPSpline(2, 4, 32, batch_norm_between_layers=True), 0.05, 5).to(DEV).train()
    b.load_state_dict(a.state_dict())
    gen = torch.Generator(device=DEV)
    gen.manual_seed(2)
    seed, off = gen.initial_seed(), gen.get_offset()
    with torch.no_grad():
        x, lq = a.sample_and_log_prob(4096, generator=gen)
        xr, ld = b.forward(draw(seed, off, 4096, 2))
    assert torch.equal(x, xr)
    for (k, v), w in zip(a.state_dict().items(), b.state_dict().values()):
        assert torch.equal(v, w), k


@pytest.mark.parametrize("which", ["normal", "mvn"])
def test_non_normal_base_matches_torch_composition(which):
    model = _perturbed(N.RealNVP(2, 4, 32), 0.05, 6).to(DEV).eval()
    if which == "normal":
        base = td.Normal(torch.ones(2, device=DEV), 2 * torch.ones(2, device=DEV))
    else:
        base = td.MultivariateNormal(torch.zeros(2, device=DEV), torch.tensor([[1.0, 0.6], [0.6, 2.0]], device=DEV))
    torch.manual_seed(9)
    with torch.no_grad():
        x, lq = model.sample_and_log_prob(3000, base_dist=base)
    torch.manual_seed(9)
    z = base.rsample((3000,))
    with torch.no_grad():
        xr, ld = model.forward(z)
    lp = base.log_prob(z)
    lp = lp.sum(1) if lp.dim() > 1 else lp
    assert torch.equal(x, xr) and torch.equal(lq, lp - ld)


def test_std_normal_base_object_uses_the_device_draw():
    model = _perturbed(N.RealNVP(2, 4, 32), 0.05, 6).to(DEV).eval()
    with torch.no_grad():
        torch.manual_seed(4)
        a = model.sample_and_log_prob(1000)
        torch.manual_seed(4)
        b = model.sample_and_log_prob(1000, base_dist=td.Normal(torch.zeros(2, device=DEV), torch.ones(2, device=DEV)))
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_stream_capture_raises():
    model = _perturbed(N.RealNVP(2, 4, 32), 0.05, 6).to(DEV).eval()
    with torch.no_grad():
        model.sample_and_log_prob(256)                    # warm-up outside the capture
        s = torch.cuda.Stream()
        g = torch.cuda.CUDAGraph()
        with pytest.raises(RuntimeError, match="CUDA graph"):
            with torch.cuda.graph(g, stream=s):
                model.sample_and_log_prob(256)


def test_no_torch_kernels_on_the_fused_and_unfused_routes():
    from torch.profiler import ProfilerActivity, profile
    models = [_perturbed(_spline_model(2, 8, 64, 8), 0.05, 1), _perturbed(N.InverseAutoregressiveFlow(16, 128), 0.02, 1)]
    for model in models:
        model = model.to(DEV).eval()
        with torch.no_grad():
            model.sample_and_log_prob(4096)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                model.sample_and_log_prob(4096)
                torch.cuda.synchronize()
        names = [e.name for e in prof.events()]
        assert any("nf::" in k for k in names), names          # the library's kernels live in namespace nf
        torch_kernels = [k for k in names if "at::native" in k or "elementwise_kernel" in k]
        assert not torch_kernels, torch_kernels
