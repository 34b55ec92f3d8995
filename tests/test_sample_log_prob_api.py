"""CPU: the public surface of sample_and_log_prob -- present on every flow class and model container, no CPU route,
and a generator only with the on-device N(0, I) draw."""
import pytest
import torch
from torch import distributions as td

import nfb200 as N


def _modules():
    m = torch.tensor([1., 0.])
    return [
        N.CouplingLayer(2, 8, m), N.SplineCouplingLayer(2, 8, m, num_bins=4), N.MaskedAutoregressiveFlow(2, 8),
        N.InverseAutoregressiveFlow(2, 8), N.ARQS(2, 8, num_bins=4),
        N.SequentialFlow([N.CouplingLayer(2, 8, m), N.InverseAutoregressiveFlow(2, 8)]),
        N.NormalizingFlowModel([N.CouplingLayer(2, 8, m), N.CouplingLayer(2, 8, 1 - m)], batch_norm_between_layers=True),
        N.RealNVP(2, 2, 8), N.RealNVPSpline(2, 2, 8),
    ]


def test_every_public_class_has_sample_and_log_prob():
    for cls in (N.Flow, N.SequentialFlow, N.CouplingLayer, N.SplineCouplingLayer, N.MaskedAutoregressiveFlow,
                N.InverseAutoregressiveFlow, N.ARQS, N.NormalizingFlowModel, N.RealNVP, N.RealNVPSpline):
        assert callable(getattr(cls, "sample_and_log_prob", None)), cls.__name__
    for mod in _modules():
        assert callable(mod.sample_and_log_prob)


@pytest.mark.parametrize("idx", range(9))
def test_cpu_module_has_no_cpu_path(idx):
    mod = _modules()[idx]
    with pytest.raises(RuntimeError, match="no CPU path"):
        mod.sample_and_log_prob(4)
    with pytest.raises(RuntimeError, match="no CPU path"):
        mod.sample_and_log_prob(4, base_dist=td.Normal(torch.zeros(2), torch.ones(2)))


def test_generator_with_a_non_normal_base_is_refused():
    layer = N.CouplingLayer(2, 8, torch.tensor([1., 0.]))
    gen = torch.Generator().manual_seed(0)
    for base in (td.Normal(torch.ones(2), 2 * torch.ones(2)),
                 td.MultivariateNormal(torch.zeros(2), torch.tensor([[1.0, 0.5], [0.5, 1.0]]))):
        with pytest.raises(ValueError, match="generator"):
            layer.sample_and_log_prob(4, base_dist=base, generator=gen)
