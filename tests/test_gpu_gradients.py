"""GPU: hand-written backward kernels against torch autograd of the CPU oracle (float64), plus the reference's
own property tests restated for CUDA modules (tests/correctness/*.py in the reference; SURVEY 4)."""
import pytest
import torch

import nfb200 as N
from oracle import flows_oracle as O
from tests import golden_util as G
from tests.build_util import assert_close, build

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

GRAD_CASES = ["coupling_eval_D4_H16_alt", "coupling_eval_D5_H8_alt", "spline_D4_H16_K10_alt", "spline_D3_H8_K4_alt",
              "spline_D4_H16_K6_alt_bound", "spline_D4_H16_K10_half_data_min_data_max", "maf_D5_H32", "iaf_D5_H32",
              "maf_D2_H16", "iaf_D3_H8", "realnvp_4_4_16_bn", "realnvpspline_6_4_32_bn", "mixed_4", "sequential_3"]


def _oracle_loss(g, sd, x, inverse, wy, wl):
    y, ld = G.oracle_eval(dict(g, sd=sd, x=x), inverse, grad=True)
    return (y * wy).sum() + (ld * wl).sum()


@pytest.mark.parametrize("name", GRAD_CASES)
@pytest.mark.parametrize("inverse", [False, True])
def test_backward_matches_oracle_autograd_f64(name, inverse):
    g = G.load(name)
    gen = torch.Generator().manual_seed(5)
    D = g["x"].shape[1]
    x = (torch.randn(24, D, generator=gen, dtype=torch.float64) * 1.5)
    wy = torch.randn(24, D, generator=gen, dtype=torch.float64)
    wl = torch.randn(24, generator=gen, dtype=torch.float64)
    # oracle side (CPU, float64, autograd through ATen)
    sd = {k: (v.double().requires_grad_() if v.is_floating_point() and "running" not in k and not k.endswith("mask")
              else (v.double() if v.is_floating_point() else v)) for k, v in g["sd"].items()}
    xo = x.clone().requires_grad_()
    _oracle_loss(g, sd, xo, inverse, wy, wl).backward()
    # product side
    m = build(g).double().to(DEV)
    xp = x.to(DEV).requires_grad_()
    y, ld = m.inverse(xp) if inverse else m.forward(xp)
    ((y * wy.to(DEV)).sum() + (ld * wl.to(DEV)).sum()).backward()
    assert_close(xp.grad, xo.grad, 1e-8, 1e-7, f"{name} dx")
    named = dict(m.named_parameters())
    checked = 0
    for k, v in sd.items():
        if isinstance(v, torch.Tensor) and v.requires_grad:
            ref = v.grad if v.grad is not None else torch.zeros_like(v)
            got = named[k].grad
            got = torch.zeros_like(named[k]) if got is None else got
            assert_close(got, ref, 1e-8, 1e-7, f"{name} d{k}")
            checked += 1
    assert checked > 0


@pytest.mark.parametrize("name", ["coupling_train_D4_H16_alt", "coupling_train_D2_H64_half"])
def test_backward_train_mode_batchnorm(name):
    g = G.load(name)
    gen = torch.Generator().manual_seed(9)
    x = g["x"].double()
    wy = torch.randn(x.shape, generator=gen, dtype=torch.float64)
    wl = torch.randn(x.shape[0], generator=gen, dtype=torch.float64)
    sd = {k: (v.double().requires_grad_() if v.is_floating_point() and "running" not in k and k != "mask"
              else (v.double() if v.is_floating_point() else v)) for k, v in g["sd"].items()}
    xo = x.clone().requires_grad_()
    y, ld = O.affine_coupling(sd, "", xo, True, training=True, update=False)
    ((y * wy).sum() + (ld * wl).sum()).backward()
    m = build(dict(g, kind="coupling")).double().to(DEV)
    m.train()
    xp = x.to(DEV).requires_grad_()
    y2, ld2 = m.inverse(xp)
    ((y2 * wy.to(DEV)).sum() + (ld2 * wl.to(DEV)).sum()).backward()
    assert_close(y2, y, 1e-9, 1e-9, "train z")
    assert_close(xp.grad, xo.grad, 1e-7, 1e-6, "train dx")
    for k, p in m.named_parameters():
        assert_close(p.grad, sd[k].grad, 1e-7, 1e-6, f"train d{k}")


# ---- the reference's property tests, restated on CUDA modules --------------------------------------------
def _layers(dim=4, hidden=16):
    alt = torch.tensor([1., 0.] * (dim // 2))
    return {
        "coupling_alt": lambda: N.CouplingLayer(dim, hidden, alt.clone()),
        "coupling_rev": lambda: N.CouplingLayer(dim, hidden, 1 - alt),
        "spline_alt": lambda: N.SplineCouplingLayer(dim, hidden, alt.clone()),
        "spline_rev": lambda: N.SplineCouplingLayer(dim, hidden, 1 - alt),
        "maf": lambda: N.MaskedAutoregressiveFlow(dim, hidden),
        "iaf": lambda: N.InverseAutoregressiveFlow(dim, hidden),
        "realnvp_bn": lambda: N.RealNVP(dim, 4, hidden, batch_norm_between_layers=True),
        "realnvpspline_bn": lambda: N.RealNVPSpline(dim, 4, hidden, batch_norm_between_layers=True),
    }


def _perturb(m, seed, sigma=0.2):
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(sigma * torch.randn(p.shape, generator=gen).to(p.device))


@pytest.mark.parametrize("kind", list(_layers()))
def test_log_determinant_symmetry(kind):
    """reference tests/correctness/test_invertibility.py:132-161 (train mode, B=8, dim 4)."""
    torch.manual_seed(0)
    m = _layers()[kind]()
    _perturb(m, 1)
    m.to(DEV)
    m.eval() if kind.startswith("coupling") or "realnvp_bn" == kind else m.train()
    x = torch.randn(8, 4, device=DEV)
    y, ld_f = m.forward(x)
    x2, ld_i = m.inverse(y)
    tol = 1e-3 if kind in ("maf", "iaf") else 1e-5
    assert (ld_f + ld_i).abs().max().item() < max(tol, 2e-5)
    assert (x2 - x).abs().max().item() < 1e-4


@pytest.mark.parametrize("kind", ["maf", "iaf"])
@pytest.mark.parametrize("dim", [3, 5, 10])
def test_autoregressive_jacobian_is_triangular(kind, dim):
    """reference tests/correctness/test_autoregressive_mask_correctness.py:24-63."""
    torch.manual_seed(dim)
    m = (N.MaskedAutoregressiveFlow if kind == "maf" else N.InverseAutoregressiveFlow)(dim, 32)
    _perturb(m, dim, 0.3)
    m.double().to(DEV).eval()
    x = torch.randn(1, dim, dtype=torch.float64, device=DEV)
    fn = (lambda v: m.forward(v)[0]) if kind == "maf" else (lambda v: m.inverse(v)[0])
    J = torch.autograd.functional.jacobian(fn, x).reshape(dim, dim)
    assert torch.triu(J, diagonal=1).abs().max().item() < 1e-6
    assert J.diagonal().abs().min().item() > 0


@pytest.mark.parametrize("kind", ["coupling_alt", "spline_alt", "maf", "iaf"])
@pytest.mark.parametrize("direction", ["forward", "inverse"])
def test_logdet_matches_autograd_jacobian(kind, direction):
    """reference tests/correctness/test_logdet_autodiff.py:107-239 (eval mode, per-row Jacobian)."""
    torch.manual_seed(3)
    m = _layers(4, 8)[kind]()
    _perturb(m, 7, 0.3)
    m.double().to(DEV).eval()
    for r in range(3):
        x = torch.randn(1, 4, dtype=torch.float64, device=DEV)
        f = getattr(m, direction)
        _, ld = f(x)
        J = torch.autograd.functional.jacobian(lambda v: f(v)[0], x).reshape(4, 4)
        ref = torch.linalg.slogdet(J)[1]
        assert abs(ld.item() - ref.item()) < 1e-6


@pytest.mark.parametrize("kind", ["coupling_alt", "spline_alt", "maf", "iaf"])
def test_gradcheck_float64(kind):
    """reference tests/correctness/test_gradcheck.py:137-255 (dim 3/4, float64)."""
    torch.manual_seed(4)
    if kind == "spline_alt":
        m = N.SplineCouplingLayer(4, 8, torch.tensor([1., 0., 1., 0.]), num_bins=4)
    else:
        m = _layers(4, 8)[kind]()
    _perturb(m, 11, 0.3)
    m.double().to(DEV).eval()
    x = (torch.randn(2, 4, dtype=torch.float64, device=DEV) * 0.7).requires_grad_()
    for direction in ("forward", "inverse"):
        f = getattr(m, direction)
        assert torch.autograd.gradcheck(lambda v: f(v)[0], (x,), eps=1e-6, atol=1e-4, rtol=1e-3, nondet_tol=1e-9)
        assert torch.autograd.gradcheck(lambda v: f(v)[1], (x,), eps=1e-6, atol=1e-4, rtol=1e-3, nondet_tol=1e-9)


def test_training_reduces_nll_realnvp():
    """README quickstart loop (README.md:105-123): inverse -> NLL -> backward -> Adam, train mode."""
    torch.manual_seed(0)
    gen = torch.Generator().manual_seed(0)
    data = torch.randn(2048, 2, generator=gen)
    data[:, 1] = 0.5 * data[:, 0] ** 2 + 0.3 * data[:, 1]
    data = data.to(DEV)
    m = N.RealNVP(2, 4, 32).to(DEV)
    opt = torch.optim.Adam(m.parameters(), lr=2e-3)
    base = torch.distributions.Normal(torch.zeros(2, device=DEV), torch.ones(2, device=DEV))
    losses = []
    for _ in range(150):
        opt.zero_grad()
        z, ld = m.inverse(data)
        loss = -(base.log_prob(z).sum(1) + ld).mean()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(torch.isfinite(torch.tensor(losses)))
    assert losses[-1] < losses[0] - 0.3


@pytest.mark.parametrize("name", ["arqs_D3_H16_K8", "arqs_D5_H32_K10", "arqs_D8_H32_K8_rescale"])
@pytest.mark.parametrize("inverse", [False, True])
def test_arqs_backward_matches_oracle_autograd_f64(name, inverse):
    """ARQS (arqs.py): D sequential steps, each = masked-linear chain + head slice + spline-step kernel, all with
    hand-written backward kernels; inputs inside the spline's domain so the bin gradients are exercised."""
    g = G.load(name)
    gen = torch.Generator().manual_seed(7)
    D = g["D"]
    x = torch.rand(24, D, generator=gen, dtype=torch.float64)
    if g["extra"]:
        x = x * (g["extra"]["data_max"] - g["extra"]["data_min"]) + g["extra"]["data_min"]
    wy = torch.randn(24, D, generator=gen, dtype=torch.float64)
    wl = torch.randn(24, generator=gen, dtype=torch.float64)
    sd = {k: (v.double().requires_grad_() if v.is_floating_point() and not k.endswith("mask") else v)
          for k, v in g["sd"].items()}
    xo = x.clone().requires_grad_()
    _oracle_loss(g, sd, xo, inverse, wy, wl).backward()
    m = build(g).double().to(DEV)
    xp = x.to(DEV).requires_grad_()
    y, ld = m.inverse(xp) if inverse else m.forward(xp)
    assert ld.dtype == torch.float32
    ((y * wy.to(DEV)).sum() + (ld * wl.to(DEV)).sum()).backward()
    assert xo.grad.abs().max() > 0
    # the float32 log-det vector rounds its incoming gradient to float32 (both here and in the oracle's autograd)
    assert_close(xp.grad, xo.grad, 1e-7, 1e-6, f"{name} dx")
    named = dict(m.named_parameters())
    for k, v in sd.items():
        if isinstance(v, torch.Tensor) and v.requires_grad:
            ref = v.grad if v.grad is not None else torch.zeros_like(v)
            got = named[k].grad
            got = torch.zeros_like(named[k]) if got is None else got
            assert_close(got, ref, 1e-7, 1e-6, f"{name} d{k}")
