"""GPU: DeviceGenerator, the device-resident seed and offset of sample_and_log_prob's N(0, I) draw.  A DeviceGenerator
at (s, o) draws the same bits as a torch.Generator with seed s at offset o on every route, with the same launches, and
each call moves its offset on by exactly 4 in device memory (ticket protocol, csrc/nf_rng.cuh) -- under load, under
CUDA-graph capture and replay, and inside a graphed reverse-KL training step."""
import copy
import math

import pytest
import torch
from torch import distributions as td

import nfb200 as N
from tests.test_gpu_sample_log_prob import FUSED, _perturbed, _spline_model

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _host_key(model, n, seed, offset):
    gen = torch.Generator(device=DEV)
    gen.manual_seed(seed)
    gen.set_offset(offset)
    with torch.no_grad():
        return model.sample_and_log_prob(n, generator=gen)


def _state(g):
    return [int(v) for v in g._state.cpu()]


def _both_paths(model, n, seed=1234, offset=40):
    """(host-key x, lq, launches), (device-state x, lq, launches) at (seed, offset); checks the generator's advance."""
    with torch.no_grad():                       # the first call builds the packed / folded weights (launches of its own)
        model.sample_and_log_prob(n)
    torch.cuda.synchronize()
    c0 = N._lib.launch_count()
    xh, lh = _host_key(model, n, seed, offset)
    torch.cuda.synchronize()
    c1 = N._lib.launch_count()
    g = N.DeviceGenerator(DEV, seed=seed)
    g.set_offset(offset)
    torch.cuda.synchronize()
    c2 = N._lib.launch_count()
    with torch.no_grad():
        xd, ld = model.sample_and_log_prob(n, generator=g)
    torch.cuda.synchronize()
    c3 = N._lib.launch_count()
    assert g.get_offset() == offset + 4 and _state(g) == [seed, offset + 4, 0, 0]
    return (xh, lh, c1 - c0), (xd, ld, c3 - c2)


def _iaf_bf16():
    return _perturbed(N.InverseAutoregressiveFlow(64, 512), 0.02, 4)


# D = 3 spline stacks on tcgen05: spline_stack_tc2_kernel<4, 8, 8, true> and <4, 10, 10, true>, the DM = 4 twins with a
# compile-time bin count (the launch function the host-key path shares picks them; test_gpu_stack_envelope checks it)
SPLINE_D3 = {
    "spline_tc_D3_K8": lambda: _spline_model(3, 4, 64, 8),
    "spline_tc_D3_K10": lambda: _spline_model(3, 4, 64, 10),
}

OTHER = {
    "iaf_gemm_16_128": lambda: _perturbed(N.InverseAutoregressiveFlow(16, 128), 0.02, 3),
    "maf_sequential_4_32": lambda: _perturbed(N.MaskedAutoregressiveFlow(4, 32), 0.05, 3),
    "arqs": lambda: _perturbed(N.ARQS(4, 32, num_bins=8), 0.05, 3),
    "float64": lambda: _perturbed(N.RealNVP(2, 4, 16).double(), 0.05, 3),
    "mixed_sequential": lambda: _perturbed(N.SequentialFlow([
        N.CouplingLayer(4, 32, torch.tensor([1., 1., 0., 0.])), N.InverseAutoregressiveFlow(4, 32),
        N.SplineCouplingLayer(4, 32, torch.tensor([0., 0., 1., 1.]), num_bins=6)]), 0.05, 3),
}


@pytest.mark.parametrize("name", sorted(FUSED) + sorted(SPLINE_D3) + sorted(OTHER) + ["coupling_fp32pipe", "iaf_bf16"])
def test_same_bits_as_the_host_key_path(name):
    n = 5000
    old_tc = N.flows.USE_TENSOR_CORES
    try:
        if name == "coupling_fp32pipe":
            N.flows.USE_TENSOR_CORES = False
            model = _perturbed(N.RealNVP(2, 6, 64), 0.05, 2)
        elif name == "iaf_bf16":
            N.set_gemm_precision("bf16")
            model = _iaf_bf16()
        elif name in FUSED:
            model = _perturbed(FUSED[name](), 0.05, 1)
        elif name in SPLINE_D3:
            model = _perturbed(SPLINE_D3[name](), 0.05, 1)
        else:
            model = OTHER[name]()
        model = model.to(DEV).eval()
        (xh, lh, ch), (xd, ld, cd) = _both_paths(model, n)
    finally:
        N.flows.USE_TENSOR_CORES = old_tc
        N.set_gemm_precision("fp32")
    assert torch.equal(xh, xd) and torch.equal(lh, ld)
    assert ch == cd, (ch, cd)
    if name in FUSED or name in SPLINE_D3 or name == "coupling_fp32pipe":
        assert cd == 1
    if name == "iaf_bf16":
        assert cd == 2


def test_ticket_under_load():
    models = [
        _perturbed(_spline_model(2, 8, 64, 8), 0.05, 1),                          # tcgen05 spline stack
        _perturbed(N.RealNVP(2, 10, 128), 0.05, 1),                               # tcgen05 coupling stack, H = 128
        _perturbed(_spline_model(6, 4, 32, 8), 0.05, 1),                          # FP32-pipe spline stack
        _perturbed(N.NormalizingFlowModel([N.InverseAutoregressiveFlow(2, 64) for _ in range(4)]), 0.05, 1),  # MADE stack
        _perturbed(N.InverseAutoregressiveFlow(3, 16), 0.05, 1),                  # draw + forward + head
    ]
    models = [m.to(DEV).eval() for m in models]
    sizes = [0, 1, 127, 5000, 70001, (1 << 20) + 3]
    for m in models:
        with torch.no_grad():
            m.sample_and_log_prob(300)
    g = N.DeviceGenerator(DEV, seed=77)
    calls, outs = [], []
    with torch.no_grad():
        for i in range(50):                     # queued back to back: no host read of the state in between
            m, n = models[i % len(models)], sizes[(i // len(models)) % len(sizes)]     # every model at every size
            calls.append((m, n))
            outs.append(m.sample_and_log_prob(n, generator=g))
    assert _state(g) == [77, 200, 0, 0]
    assert {n for _, n in calls} == set(sizes)
    for i, ((m, n), (x, lq)) in enumerate(zip(calls, outs)):
        xr, lr = _host_key(m, n, 77, 4 * i)
        assert torch.equal(x, xr) and torch.equal(lq, lr), (i, n)


def _capture(model, n, g):
    with torch.no_grad():
        model.sample_and_log_prob(n, generator=g)           # warm-up outside the capture
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            x, lq = model.sample_and_log_prob(n, generator=g)
    return graph, x, lq


@pytest.mark.parametrize("route", ["fused_spline_stack", "unfused_iaf_gemm", "iaf_bf16_chain"])
def test_capture_and_replay(route):
    n = 4096
    if route == "fused_spline_stack":
        model = _perturbed(_spline_model(2, 8, 64, 8), 0.05, 1)
    elif route == "unfused_iaf_gemm":
        model = _perturbed(N.InverseAutoregressiveFlow(16, 128), 0.02, 3)
    else:
        N.set_gemm_precision("bf16")
        model = _iaf_bf16()
    try:
        model = model.to(DEV).eval()
        g = N.DeviceGenerator(DEV, seed=0)
        graph, x, lq = _capture(model, n, g)
        g.manual_seed(7)
        outs = []
        for _ in range(3):
            graph.replay()
            outs.append((x.clone(), lq.clone()))
        assert g.get_offset() == 12
        for i, (xo, lo) in enumerate(outs):
            xr, lr = _host_key(model, n, 7, 4 * i)
            assert torch.equal(xo, xr) and torch.equal(lo, lr), i
        assert not torch.equal(outs[0][0], outs[1][0]) and not torch.equal(outs[1][0], outs[2][0])
        assert not torch.equal(outs[0][0], outs[2][0])
        g.manual_seed(7)
        graph.replay()
        assert torch.equal(x, outs[0][0]) and torch.equal(lq, outs[0][1])
        assert g.get_offset() == 4
    finally:
        N.set_gemm_precision("fp32")


_MEANS = None


def _target_log_prob(x):
    """A fixed 2-D mixture of two unit Gaussians at (-2, 0) and (2, 0), equal weights."""
    d = x[:, None, :] - _MEANS[None]
    lp = -0.5 * (d * d).sum(-1) - math.log(2 * math.pi)
    return torch.logsumexp(lp, dim=1) - math.log(2.0)


@pytest.mark.parametrize("make", [lambda: N.RealNVP(2, 4, 32),
                                  lambda: N.NormalizingFlowModel([N.InverseAutoregressiveFlow(2, 64) for _ in range(6)])],
                         ids=["realnvp_2_4_32", "iaf_6x_2_64"])
def test_graphed_reverse_kl_step_follows_eager(make):
    global _MEANS
    _MEANS = torch.tensor([[-2.0, 0.0], [2.0, 0.0]], device=DEV)
    torch.manual_seed(0)
    base = make().to(DEV).train()
    n = 2000

    def make_loss(g):
        def loss_fn(m, _):
            x, lq = m.sample_and_log_prob(n, generator=g)
            return (lq - _target_log_prob(x)).mean()
        return loss_fn

    eager_m = copy.deepcopy(base)
    opt_e = torch.optim.SGD(eager_m.parameters(), lr=1e-2, momentum=0.9)
    graph_m = copy.deepcopy(base)
    opt_g = torch.optim.SGD(graph_m.parameters(), lr=1e-2, momentum=0.9)
    g_graph, g_eager = N.DeviceGenerator(DEV, seed=5), N.DeviceGenerator(DEV, seed=5)
    loss_g, loss_e = make_loss(g_graph), make_loss(g_eager)
    step = N.graphs.GraphedTrainStep(graph_m, opt_g, loss_g, torch.empty(1, device=DEV), warmup=2)
    for _ in range(2):                      # the 2 warm-up steps (capture records the step, it does not run it)
        opt_e.zero_grad(set_to_none=True)
        loss_e(eager_m, None).backward()
        opt_e.step()
    assert g_graph.get_offset() == g_eager.get_offset() == 8
    losses_g, losses_e = [], []
    for _ in range(3):
        losses_g.append(float(step()))
        opt_e.zero_grad(set_to_none=True)
        le = loss_e(eager_m, None)
        le.backward()
        opt_e.step()
        losses_e.append(float(le.detach()))
    assert g_graph.get_offset() == g_eager.get_offset() == 20
    assert len(set(losses_g)) == 3                       # every replay drew new samples
    assert all(abs(a - b) <= 1e-4 * (1 + abs(b)) for a, b in zip(losses_g, losses_e)), (losses_g, losses_e)
    for (k, p), (_, q) in zip(graph_m.named_parameters(), eager_m.named_parameters()):
        assert torch.allclose(p, q, atol=1e-5, rtol=1e-4), k


def test_refusals():
    model = _perturbed(N.RealNVP(2, 4, 32), 0.05, 6).to(DEV).eval()
    g = N.DeviceGenerator(DEV, seed=3)
    for base in (td.Normal(torch.ones(2, device=DEV), 2 * torch.ones(2, device=DEV)),
                 td.MultivariateNormal(torch.zeros(2, device=DEV), torch.tensor([[1.0, 0.5], [0.5, 1.0]], device=DEV))):
        with pytest.raises(ValueError, match="generator"):
            model.sample_and_log_prob(8, base_dist=base, generator=g)
    with pytest.raises(ValueError, match="DeviceGenerator"):
        N.RealNVP(2, 2, 8).sample_and_log_prob(8, generator=g)          # the model on the CPU, the generator on cuda:0
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="DeviceGenerator"):
            model.sample_and_log_prob(8, generator=N.DeviceGenerator("cuda:1", seed=3))
    assert g.get_offset() == 0                                        # nothing was drawn
    with pytest.raises(ValueError, match="multiple of 4"):
        g.set_offset(6)
    with torch.no_grad():
        model.sample_and_log_prob(8, generator=g)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        for what in ("manual_seed", "get_offset", "set_offset"):
            with pytest.raises(RuntimeError, match=what):
                with torch.cuda.graph(graph):
                    if what == "manual_seed":
                        g.manual_seed(1)
                    elif what == "get_offset":
                        g.get_offset()
                    else:
                        g.set_offset(0)
            graph = torch.cuda.CUDAGraph()
    assert g.get_offset() == 4 and g.initial_seed() == 3


def test_default_seed_follows_torch_manual_seed_and_nan_free_draw_with_high_seed():
    torch.manual_seed(4242)
    g = N.DeviceGenerator()
    assert g.initial_seed() == 4242 and g.get_offset() == 0 and g.device == torch.device(DEV)
    seed = (1 << 64) - 5                                              # a seed above 2^63 round-trips through int64
    g.manual_seed(seed)
    assert g.initial_seed() == seed
    model = _perturbed(_spline_model(2, 8, 64, 8), 0.05, 1).to(DEV).eval()
    with torch.no_grad():
        x, lq = model.sample_and_log_prob(1000, generator=g)
    xr, lr = _host_key(model, 1000, seed, 0)
    assert torch.equal(x, xr) and torch.equal(lq, lr)
