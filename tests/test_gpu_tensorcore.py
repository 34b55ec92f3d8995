"""GPU: the tcgen05 tile primitive (TMEM operands, SWIZZLE_128B weight images, 3xTF32) against a float64 product."""
import numpy as np
import pytest
import torch

import nfb200 as N
N_ = N

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n_out", [16, 32, 64, 128])
def test_tc_gemm128_3xtf32(n_out):
    rng = np.random.default_rng(n_out)
    a = rng.standard_normal((128, 64)).astype(np.float32) * 2
    w = rng.standard_normal((n_out, 64)).astype(np.float32)
    img = torch.from_numpy(N.packing.umma_sw128_images(w)).cuda()
    ad = torch.from_numpy(a).cuda()
    ref = a.astype(np.float64) @ w.astype(np.float64).T
    scale = np.abs(a).astype(np.float64) @ np.abs(w).astype(np.float64).T
    for passes, tol in ((3, 1e-6), (1, 2e-3)):
        d = torch.full((128, n_out), float("nan"), device="cuda")
        N._lib.call("nf_debug_tc_gemm128", ad.data_ptr(), img.data_ptr(), d.data_ptr(), n_out, passes, None, 1,
                    N._lib.stream())
        torch.cuda.synchronize()
        err = np.abs(d.cpu().numpy().astype(np.float64) - ref) / scale
        assert np.isfinite(err).all()
        assert err.max() < tol, f"passes={passes}: max scaled error {err.max():.3e}"
        if passes == 1:
            assert err.max() > 1e-6      # a single TF32 pass must NOT be fp32-accurate (sanity of the test itself)


@pytest.mark.parametrize("M,N,K", [(128, 128, 32), (1000, 512, 64), (4096, 512, 512), (777, 130, 100), (300, 64, 1024),
                                   (257, 22736 // 8, 128)])
@pytest.mark.parametrize("relu", [False, True])
def test_linear_tc_matches_float64(M, N, K, relu):
    gen = torch.Generator().manual_seed(M + N + K)
    x = torch.randn(M, K, generator=gen) * 1.5
    w = torch.randn(N, K, generator=gen) / K ** 0.5
    b = torch.randn(N, generator=gen)
    xd, wd, bd = x.cuda(), w.cuda(), b.cuda()
    hi, lo = N_.ops.split_tf32(wd)
    assert torch.equal(hi.cpu().view(torch.int32) & 0x1FFF, torch.zeros(N, K, dtype=torch.int32))
    assert torch.equal(lo.cpu().view(torch.int32) & 0x1FFF, torch.zeros(N, K, dtype=torch.int32))
    assert bool((((hi + lo).cpu().double() - w.double()).abs() <= 2.0 ** -23 * w.double().abs()).all())
    hn, ln = N_.packing.split_tf32(w.numpy())
    assert torch.equal(hi.cpu(), torch.from_numpy(hn)) and torch.equal(lo.cpu(), torch.from_numpy(ln))
    y = N_.ops.linear_tc(xd, hi, lo, bd, relu)
    assert y is not None
    ref = x.double() @ w.double().T + b.double()
    scale = x.double().abs() @ w.double().abs().T + b.double().abs()
    if relu:
        ref = ref.clamp_min(0)
    err = ((y.cpu().double() - ref).abs() / scale).max().item()
    assert err < 2e-6, f"scaled error {err:.3e}"      # K up to 1024: fp32 accumulation in TMEM adds ~sqrt(K) ulp
    # and against the FP32-pipe GEMM (same inputs): both are fp32-accurate
    y2 = N_.ops.linear_raw(xd, wd, bd, relu)
    assert ((y - y2).abs() / scale.cuda().float()).max().item() < 2e-6


def test_linear_tc_k_extent_matches_masked_dense():
    gen = torch.Generator().manual_seed(0)
    M, N, K = 512, 256, 256
    x = torch.randn(M, K, generator=gen)
    w = torch.randn(N, K, generator=gen)
    ext = torch.tensor([64, 100, 200, 256], dtype=torch.int32)
    for t in range(4):
        w[t * 64:(t + 1) * 64, int(ext[t]):] = 0
    hi, lo = N_.ops.split_tf32(w.cuda())
    y = N_.ops.linear_tc(x.cuda(), hi, lo, None, False, ext.cuda())
    ref = x.double() @ w.double().T
    scale = x.double().abs() @ w.double().abs().T + 1e-30
    err = ((y.cpu().double() - ref).abs() / scale).max().item()
    assert err < 2e-6, f"scaled error {err:.3e}"


@pytest.mark.parametrize("B,N,K", [(32, 128, 128), (256, 128, 128), (4096, 512, 512), (5000, 512, 64), (777, 132, 100),
                                   (100000, 128, 256), (3000, 2844, 1024), (1, 64, 64), (0, 64, 32), (30000, 23, 64),
                                   (5000, 29, 1024), (1000, 11369, 128)])
def test_linear_wgrad_tc_matches_float64(B, N, K):
    """dW = dY^T X on tcgen05 (MN-major operands, split over the batch) against a float64 product."""
    gen = torch.Generator().manual_seed(B + N + K)
    g = torch.randn(B, N, generator=gen) * 1.5
    x = torch.randn(B, K, generator=gen)
    gd, xd = g.cuda(), x.cuda()
    dw = N_.ops.linear_wgrad_tc(gd, xd, out=torch.full((N, K), float("nan"), device="cuda"))
    assert dw is not None
    torch.cuda.synchronize()
    ref = g.double().T @ x.double()
    scale = g.double().abs().T @ x.double().abs() + 1e-30
    err = ((dw.cpu().double() - ref).abs() / scale).max().item()
    # the tensor core's fp32 accumulation truncates: measured bias 2^-25 of the running sum per MMA (scripts/
    # wgrad_accuracy.py); a TMEM chain is at most 64 K blocks x 12 MMAs long => <= 2.3e-5 of sum|a||b| in the worst
    # (same-sign) case, ~1e-6 for random signs; the split partials are then added with round-to-nearest
    assert err < 1e-5, f"scaled error {err:.3e}"
    if B:
        dw2 = N_.ops.gemm(gd, xd, N, K, B, 1, N, K, 1)
        assert ((dw - dw2).abs() / scale.cuda().float()).max().item() < 1e-5
        rms = (dw.cpu().double() - ref).pow(2).mean().sqrt().item() / max(ref.pow(2).mean().sqrt().item(), 1e-30)
        assert rms < 3e-5, f"rms error / rms(dW) {rms:.3e}"
        # deterministic: the split partials are summed in a fixed order
        assert torch.equal(dw, N_.ops.linear_wgrad_tc(gd, xd))


def test_linear_autograd_uses_tc_wgrad_and_matches_float64():
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(2048, 256, generator=gen)
    w = torch.randn(512, 256, generator=gen) / 16
    b = torch.randn(512, generator=gen)
    xd = x.cuda().requires_grad_(True)
    wd = w.cuda().requires_grad_(True)
    bd = b.cuda().requires_grad_(True)
    y = N_.ops.linear(xd, wd, bd, relu=True)
    (y * y).sum().backward()
    x64, w64, b64 = (t.double().requires_grad_(True) for t in (x, w, b))
    y64 = torch.relu(x64 @ w64.T + b64)
    (y64 * y64).sum().backward()
    for got, ref in ((xd.grad, x64.grad), (wd.grad, w64.grad), (bd.grad, b64.grad)):
        rel = (got.cpu().double() - ref).abs().max().item() / ref.abs().max().item()
        assert rel < 2e-5, rel


@pytest.mark.parametrize("rows,cols", [(5, 8), (1024, 4), (1500, 132), (65536, 512), (4096, 11368), (3000, 7), (0, 16)])
def test_col_sum_matches_float64(rows, cols):
    """bias gradient reduction (autograd of F.linear's bias): vectorised and scalar kernels."""
    gen = torch.Generator().manual_seed(rows + cols)
    a = torch.randn(rows, cols, generator=gen) + 0.25
    got = N_.ops.col_sum(a.cuda()).cpu().double()
    ref = a.double().sum(0)
    scale = a.double().abs().sum(0) + 1e-30
    assert ((got - ref).abs() / scale).max().item() < 1e-6


@pytest.mark.parametrize("rows,cols,dtype", [(5, 8, torch.float32), (1500, 132, torch.float32), (65536, 64, torch.float32),
                                             (70001, 512, torch.float32), (4096, 1024, torch.float32), (3000, 23, torch.float32),
                                             (2048, 64, torch.float64), (0, 16, torch.float32)])
def test_relu_backward_colsum_matches_the_two_pass_result(rows, cols, dtype):
    """nf_relu_backward_colsum (ReLU backward of a Linear(+ReLU) fused with that Linear's bias gradient): gx is exactly
    gy masked by y > 0 (NaN in y masks like torch.relu's backward: NaN > 0 is false), the column sums match float64; the
    fused 128-bit kernel and the fallback (two kernels) are both covered."""
    gen = torch.Generator().manual_seed(rows * 7 + cols)
    y = torch.relu(torch.randn(rows, cols, generator=gen, dtype=dtype))
    gy = torch.randn(rows, cols, generator=gen, dtype=dtype) + 0.1
    if rows > 4:
        y[3, 1] = float("nan")
    gx, cs = N_.ops.relu_backward_colsum(y.cuda(), gy.cuda())
    ref = torch.where(y > 0, gy, torch.zeros_like(gy))
    assert torch.equal(gx.cpu(), ref)
    ref_cs = ref.double().sum(0)
    scale = ref.double().abs().sum(0) + 1e-30
    assert ((cs.cpu().double() - ref_cs).abs() / scale).max().item() < (1e-6 if dtype == torch.float32 else 1e-13) if cols else True


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("B,H,D", [(5000, 64, 2), (300, 64, 2), (70000, 128, 3), (4096, 40, 8), (1000, 16, 1), (30000, 64, 23),
                                   (9000, 300, 29), (2000, 64, 17), (1001, 256, 2), (777, 128, 4), (67, 1024, 6), (4099, 100, 5)])
def test_skinny_products_match_float64(B, H, D, dtype):
    """nf_gemm's skinny routes (one dimension <= 8): first / last Linear of a low-dimensional conditioner, forward,
    input gradient and weight gradient, against float64 products."""
    gen = torch.Generator().manual_seed(B + H + D)
    x = torch.randn(B, D, generator=gen, dtype=torch.float64)
    h = torch.randn(B, H, generator=gen, dtype=torch.float64)
    w1 = torch.randn(H, D, generator=gen, dtype=torch.float64)          # first Linear  [H, D]
    w3 = torch.randn(D, H, generator=gen, dtype=torch.float64)          # last Linear   [D, H]
    b1 = torch.randn(H, generator=gen, dtype=torch.float64)
    b3 = torch.randn(D, generator=gen, dtype=torch.float64)
    gy1 = torch.randn(B, H, generator=gen, dtype=torch.float64)         # grad of the first Linear's output
    gy3 = torch.randn(B, D, generator=gen, dtype=torch.float64)
    c = lambda t: t.to(dtype).cuda().contiguous()
    tol = 2e-6 if dtype == torch.float32 else 1e-12

    def check(got, ref, scale, what):
        err = ((got.cpu().double() - ref).abs() / (scale + 1e-30)).max().item()
        assert err < tol, f"{what}: scaled error {err:.3e}"

    # forward, K = D small (bias + ReLU) and N = D small (bias)
    check(N_.ops.linear_raw(c(x), c(w1), c(b1), relu=True), torch.relu(x @ w1.T + b1), x.abs() @ w1.abs().T + b1.abs(), "fwd K small")
    check(N_.ops.linear_raw(c(h), c(w3), c(b3)), h @ w3.T + b3, h.abs() @ w3.abs().T + b3.abs(), "fwd N small")
    # input gradient of the last Linear: dX[B,H] = dY[B,D] W3[D,H]
    check(N_.ops.gemm(c(gy3), c(w3), B, H, D, D, 1, H, 1), gy3 @ w3, gy3.abs() @ w3.abs(), "dX K small")
    # input gradient of the first Linear: dX[B,D] = dY[B,H] W1[H,D]
    check(N_.ops.gemm(c(gy1), c(w1), B, D, H, H, 1, D, 1), gy1 @ w1, gy1.abs() @ w1.abs(), "dX N small")
    # weight gradients: dW1[H,D] = dY1^T x, dW3[D,H] = dY3^T h
    check(N_.ops.gemm(c(gy1), c(x), H, D, B, 1, H, D, 1), gy1.T @ x, gy1.abs().T @ x.abs(), "dW narrow K")
    check(N_.ops.gemm(c(gy3), c(h), D, H, B, 1, D, H, 1), gy3.T @ h, gy3.abs().T @ h.abs(), "dW narrow N")
    # bias gradient of the last Linear
    check(N_.ops.col_sum(c(gy3)), gy3.sum(0), gy3.abs().sum(0), "col_sum small")


@pytest.mark.parametrize("D,H,B", [(64, 512, 1024), (256, 1024, 512), (20, 256, 700)])
def test_mask_plans_skip_only_exact_zeros(D, H, B):
    """MADE-masked linear layers (masked_linear.py:14-18) through the autograd op with and without the zero-structure
    plans (K-range / tile skipping in the forward, input-gradient and weight-gradient GEMMs): same results, and both
    match a float64 masked product."""
    made = N_.MADE(D, H)
    gen = torch.Generator().manual_seed(D + H)
    for idx in (2, 6):                                   # hidden->hidden [H,H] and hidden->out [2D,H]
        lin = made.net[idx]
        w = (torch.randn(lin.weight.shape, generator=gen) / lin.weight.shape[1] ** 0.5)
        b = torch.randn(lin.weight.shape[0], generator=gen)
        mask = lin.mask.clone()
        x = torch.randn(B, lin.weight.shape[1], generator=gen)
        gy = torch.randn(B, lin.weight.shape[0], generator=gen)
        res = {}
        for use in (True, False):
            N_.ops.USE_MASK_PLANS = use
            try:
                xd = x.cuda().requires_grad_(True)
                wd = w.cuda().requires_grad_(True)
                bd = b.cuda().requires_grad_(True)
                y = N_.ops.linear(xd, wd, bd, mask=mask.cuda(), relu=True)
                y.backward(gy.cuda())
                res[use] = (y.detach().cpu(), xd.grad.cpu(), wd.grad.cpu(), bd.grad.cpu())
            finally:
                N_.ops.USE_MASK_PLANS = True
        plan = N_.ops.mask_plan(mask.cuda())
        if min(mask.shape) >= 512:                      # 4 x 4 tiles or more: the upper triangle is skippable
            assert plan is not None and plan.live_fraction < 0.9
        x64, w64, b64 = (t.double().requires_grad_(True) for t in (x, w, b))
        y64 = torch.relu(x64 @ (w64 * mask.double()).T + b64)
        y64.backward(gy.double())
        refs = (y64.detach(), x64.grad, w64.grad, b64.grad)
        for got_a, got_b, ref, what in zip(res[True], res[False], refs, ("y", "dx", "dw", "db")):
            scale = ref.abs().max().item() + 1e-30
            assert (got_a.double() - ref).abs().max().item() / scale < 2e-5, what
            assert (got_a - got_b).abs().max().item() / scale < 2e-5, what
        assert torch.equal(res[True][2] == 0, res[False][2] == 0) or bool((res[True][2][mask == 0] == 0).all())


@pytest.mark.parametrize("M,N,K", [(4096, 512, 512), (2048, 1024, 1024), (1000, 300, 2048), (512, 128, 4096)])
def test_long_contractions_are_fp32_grade(M, N, K):
    """Short-chain kernel (gemm_tc2.cu): the rms error of a K-long product stays at the FFMA-GEMM level whatever K is
    (a single TMEM accumulation chain grows linearly: 4e-6 at K = 1024, 3e-5 at K = 4096), also for same-sign data
    (no bias)."""
    gen = torch.Generator().manual_seed(K)
    for positive in (False, True):
        x = torch.randn(M, K, generator=gen)
        w = torch.randn(N, K, generator=gen) / K ** 0.5
        if positive:
            x, w = x.abs(), w.abs()
        hi, lo = N_.ops.split_tf32(w.cuda())
        y = N_.ops.linear_tc(x.cuda(), hi, lo)
        ref = x.double() @ w.double().T
        rms = ref.pow(2).mean().sqrt().item()
        e = y.cpu().double() - ref
        assert e.pow(2).mean().sqrt().item() / rms < 1.5e-6, (positive, e.pow(2).mean().sqrt().item() / rms)
        # same-sign data: a 48-MMA chain still loses ~48 * 2^-25 = 1.4e-6 of the running sum (384 MMAs: 1.2e-5)
        assert abs(e.mean().item()) / rms < (2e-6 if positive else 5e-7), (positive, e.mean().item() / rms)


@pytest.fixture
def tf32_mode():
    N_.set_gemm_precision("tf32")
    try:
        yield
    finally:
        N_.set_gemm_precision("fp32")


# Reduced-precision mode (set_gemm_precision("tf32"), BASELINE config C4's "bf16 conditioner GEMMs" slot): one TF32
# pass, both operands rounded to the nearest TF32 (relative rounding error <= 2^-11 each) => every product is within
# 2^-10 of |a||b|, i.e. the scaled error max|err| / sum|a||b| is bounded by 2^-10 = 9.8e-4 (+ fp32 accumulation);
# a bf16 product would be bounded by 2^-7 = 7.8e-3.  Bounds written here are the documented ones (DESIGN.md).
TF32_SCALED_BOUND = 1.0e-3
TF32_RMS_BOUND = 6.0e-4          # rms error / rms(result) for random-sign data: ~2^-11 * sqrt(2/3)


@pytest.mark.parametrize("M,N,K", [(128, 128, 32), (1000, 512, 64), (4096, 512, 512), (777, 130, 100), (300, 64, 1024),
                                   (2048, 1024, 1024), (512, 128, 4096)])
@pytest.mark.parametrize("relu", [False, True])
def test_linear_tc_tf32_mode_bounds(tf32_mode, M, N, K, relu):
    gen = torch.Generator().manual_seed(M + N + K)
    x = torch.randn(M, K, generator=gen) * 1.5
    w = torch.randn(N, K, generator=gen) / K ** 0.5
    b = torch.randn(N, generator=gen)
    hi, lo = N_.ops.split_tf32(w.cuda())
    y = N_.ops.linear_tc(x.cuda(), hi, lo, b.cuda(), relu)
    assert y is not None
    ref = x.double() @ w.double().T + b.double()
    scale = x.double().abs() @ w.double().abs().T + b.double().abs()
    if relu:
        ref = ref.clamp_min(0)
    e = y.cpu().double() - ref
    err = (e.abs() / scale).max().item()
    assert err < TF32_SCALED_BOUND, f"scaled error {err:.3e}"
    assert err > 1e-6                       # the mode must really be the single-pass one
    if not relu:
        assert e.pow(2).mean().sqrt().item() / ref.pow(2).mean().sqrt().item() < TF32_RMS_BOUND
    # w_lo is not read in this mode
    y_nolo = N_.ops.linear_tc(x.cuda(), hi, torch.full_like(lo, float("nan")), b.cuda(), relu)
    assert torch.equal(y, y_nolo)
    # and the default mode is back to fp32 grade afterwards (checked by the other tests through the fixture's finally)


@pytest.mark.parametrize("B,N,K", [(256, 128, 128), (4096, 512, 512), (777, 132, 100), (100000, 128, 256),
                                   (5000, 29, 1024), (3000, 2844, 1024)])
def test_linear_wgrad_tc_tf32_mode_bounds(tf32_mode, B, N, K):
    gen = torch.Generator().manual_seed(B + N + K)
    g = torch.randn(B, N, generator=gen) * 1.5
    x = torch.randn(B, K, generator=gen)
    dw = N_.ops.linear_wgrad_tc(g.cuda(), x.cuda(), out=torch.full((N, K), float("nan"), device="cuda"))
    assert dw is not None
    ref = g.double().T @ x.double()
    scale = g.double().abs().T @ x.double().abs() + 1e-30
    e = dw.cpu().double() - ref
    err = (e.abs() / scale).max().item()
    assert 1e-6 < err < TF32_SCALED_BOUND, f"scaled error {err:.3e}"
    assert e.pow(2).mean().sqrt().item() / ref.pow(2).mean().sqrt().item() < TF32_RMS_BOUND
    assert torch.equal(dw, N_.ops.linear_wgrad_tc(g.cuda(), x.cuda()))


def test_tf32_mode_flow_parity_bounds(tf32_mode):
    """Whole-layer effect of the reduced-precision mode against the default mode on the same weights: MAF(64, 512)
    density pass and a RealNVPSpline(784, 2, 1024) pass.  Documented bounds (DESIGN.md, measured values in
    profiles/r01t_tf32_mode_accuracy.log): z within 5e-3 * max(1, |z|) and log-det within 5e-2 at D = 64; z within 2e-2
    and log-det within 2e-1 at D = 784 (392 spline elements per row and layer, each sensitive to its 29 parameters)."""
    torch.manual_seed(0)
    for make, D, z_tol, ld_tol in ((lambda: N_.MaskedAutoregressiveFlow(64, 512), 64, 5e-3, 5e-2),
                                   (lambda: N_.RealNVPSpline(784, 2, 1024), 784, 2e-2, 2e-1)):
        m = make().cuda().eval()
        with torch.no_grad():
            for p in m.parameters():
                p.add_(0.02 * torch.randn_like(p))
        x = torch.randn(2048, D, device="cuda")
        with torch.no_grad():
            z_f, ld_f = m.inverse(x)
            N_.set_gemm_precision("fp32")
            z_r, ld_r = m.inverse(x)
            N_.set_gemm_precision("tf32")
        assert torch.isfinite(z_f).all() and torch.isfinite(ld_f).all()
        dz = ((z_f - z_r).abs() / z_r.abs().clamp_min(1)).max().item()
        dl = (ld_f - ld_r).abs().max().item()
        assert dz < z_tol, (D, dz)
        assert dl < ld_tol, (D, dl)
        assert dz > 0 or dl > 0            # the mode changed something


def test_set_gemm_precision_rejects_unknown_modes():
    with pytest.raises(ValueError):
        N_.set_gemm_precision("bf16x")
    assert N_.get_gemm_precision() == "fp32"


@pytest.mark.parametrize("M,N,K", [(4096, 512, 512), (777, 130, 100), (300, 64, 1024), (1000, 512, 64)])
def test_linear_tc_one_pass_ss_option_bounds(tf32_mode, M, N, K):
    """nf_set_option(10, 1): the one-pass mode with the A operand straight from shared memory.  The tensor core truncates
    x to TF32 (relative error < 2^-10, toward zero) where the converters round (2^-11), w_hi is rounded:
    max|err| / sum|a||b| <= 2^-10 + 2^-11 = 1.5e-3."""
    gen = torch.Generator().manual_seed(M + N + K)
    x = torch.randn(M, K, generator=gen) * 1.5
    w = torch.randn(N, K, generator=gen) / K ** 0.5
    b = torch.randn(N, generator=gen)
    hi, lo = N_.ops.split_tf32(w.cuda())
    N_._lib.call("nf_set_option", 10, 1)
    try:
        y = N_.ops.linear_tc(x.cuda(), hi, lo, b.cuda(), True)
    finally:
        N_._lib.call("nf_set_option", 10, 0)
    ref = (x.double() @ w.double().T + b.double()).clamp_min(0)
    scale = x.double().abs() @ w.double().abs().T + b.double().abs()
    err = ((y.cpu().double() - ref).abs() / scale).max().item()
    assert 1e-6 < err < 1.6e-3, f"scaled error {err:.3e}"
