"""Layer stacks: same classes, constructor arguments and state_dict layout as the reference's `src.models`.

    NormalizingFlowModel   src/models/normalizing_flow_model.py:4-128
    RealNVP                src/models/real_nvp.py:6-49
    RealNVPSpline          src/models/real_nvp_spline.py:6-48
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .flows import (ChainPlan, CouplingLayer, SplineCouplingLayer, _apply_layer, _as_context, _context_dim, _shared_context_dim,
                    flow_log_prob, flow_sample_and_log_prob, on_input_device, sample_from)


class _DensityAPI:
    """log_prob / sample on the model containers (north_star: `NormalizingFlowModel.log_prob/sample`; same meaning as
    Flow.log_prob / Flow.sample, flow.py:40-73).  base_dist=None means the standard normal N(0, I); a standard-normal
    base is evaluated by the fused head (one launch for a fused stack, z never written).
    A model with conditional layers (context_dim > 0) takes context= on every call: [B, C] or [1, C] for log_prob,
    forward and inverse, [m, C] for sample / sample_and_log_prob (n rows per context row, returned as [m, n, ...])."""

    def _data_dim(self):
        flows = self.flows if hasattr(self, "flows") else self.flow.flows
        return getattr(flows[0], "data_dim", None)

    def log_prob(self, x, base_dist=None, context=None):
        return flow_log_prob(self, x, base_dist, getattr(self, "_log_prob_fused", None), context)

    def sample(self, num_samples, base_dist=None, device=None, context=None):
        if device is None:
            device = next(self.parameters()).device
        return sample_from(self, self._data_dim(), num_samples, base_dist, device, context)

    def sample_and_log_prob(self, num_samples, base_dist=None, device=None, generator=None, context=None):
        """(x, log_q) with z ~ base, (x, log_det) = forward(z), log_q = log p_base(z) - log_det: Flow.sample_and_log_prob.
        A standard-normal base is drawn on the GPU (one launch for a fused stack, z never written)."""
        return flow_sample_and_log_prob(self, num_samples, base_dist, device, generator, context)


class NormalizingFlowModel(_DensityAPI, nn.Module):
    """Chain of flow layers, optionally with an invertible BatchNorm affine between consecutive layers.

    The between-layer BatchNorm always transforms with its *running* statistics (so that forward, inverse and
    log-det share constants); train mode only moves the running statistics towards the batch statistics
    (momentum, biased variance) before using them (normalizing_flow_model.py:67-85).  Its log-det is the scalar
    sum(log|gamma| - 0.5*log(var+eps)), broadcast over rows (:87-108).
    """

    def __init__(self, flows, batch_norm_between_layers=False):
        super().__init__()
        self.batch_norm_between_layers = batch_norm_between_layers
        if self.batch_norm_between_layers:
            data_dim = getattr(flows[0], "data_dim", None)
            if data_dim is None:
                raise ValueError("Cannot use batch_norm_between_layers if flows do not have a 'data_dim' attribute.")
            self.batch_norms = nn.ModuleList([nn.BatchNorm1d(data_dim) for _ in range(len(flows))])
        self.flows = nn.ModuleList(flows)
        self.context_dim = _shared_context_dim(self.flows)    # the between-layer BatchNorms never see the context
        self._chain = ChainPlan()

    # -- between-layer BatchNorm pieces: [B,D] work in kernels, [D]-sized constants on the parameter vectors ----
    @staticmethod
    def _bn_sd(bn):
        return torch.sqrt(bn.running_var + bn.eps)

    def _apply_batch_norm(self, bn_layer, x):
        if self.training:
            mean, var = ops.col_stats(x)
            with torch.no_grad():
                momentum = bn_layer.momentum if bn_layer.momentum is not None else 0.1
                bn_layer.running_mean.mul_(1 - momentum).add_(momentum * mean.to(bn_layer.running_mean.dtype))
                bn_layer.running_var.mul_(1 - momentum).add_(momentum * var.to(bn_layer.running_var.dtype))
        return ops.feature_affine(x, bn_layer.running_mean, self._bn_sd(bn_layer), bn_layer.weight, bn_layer.bias)

    def _inverse_batch_norm(self, bn_layer, y):
        return ops.feature_affine(y, bn_layer.bias, bn_layer.weight, self._bn_sd(bn_layer), bn_layer.running_mean)

    def _batch_norm_log_det_jacobian(self, bn_layer, x):
        return (torch.log(torch.abs(bn_layer.weight)) - 0.5 * torch.log(bn_layer.running_var + bn_layer.eps)).sum()

    def _bns(self):
        return self.batch_norms if self.batch_norm_between_layers else None

    def _log_prob_fused(self, x, ctx=None):
        out = self._chain.run(self.flows, self._bns(), self.training, x, True, head=True, ctx=ctx)
        return None if out is None else out[1]

    def _sample_fused(self, x, draw, ctx=None):
        return self._chain.run(self.flows, self._bns(), self.training, x, False, sample=draw, ctx=ctx)

    @on_input_device
    def forward(self, z, context=None):
        """Sampling direction z -> x (:25-46)."""
        ctx = _as_context(self, context, z)
        fused = self._chain.run(self.flows, self._bns(), self.training, z, False, ctx=ctx)
        if fused is not None:
            return fused
        log_det_sum = 0
        last = len(self.flows) - 1
        for i, flow in enumerate(self.flows):
            z, log_det = flow(z) if ctx is None or not _context_dim(flow) else _apply_layer(flow, z, False, ctx)
            log_det_sum = log_det_sum + log_det
            if self.batch_norm_between_layers and i < last:
                bn = self.batch_norms[i]
                z = self._apply_batch_norm(bn, z)
                log_det_sum = log_det_sum + self._batch_norm_log_det_jacobian(bn, z)
        return z, log_det_sum

    @on_input_device
    def inverse(self, x, context=None):
        """Density direction x -> z (:48-65)."""
        ctx = _as_context(self, context, x)
        fused = self._chain.run(self.flows, self._bns(), self.training, x, True, ctx=ctx)
        if fused is not None:
            return fused
        log_det_sum = 0
        last = len(self.flows) - 1
        for i in range(last, -1, -1):
            if self.batch_norm_between_layers and i < last:
                bn = self.batch_norms[i]
                x = self._inverse_batch_norm(bn, x)
                log_det_sum = log_det_sum - self._batch_norm_log_det_jacobian(bn, x)
            x, log_det = _apply_layer(self.flows[i], x, True, ctx)
            log_det_sum = log_det_sum + log_det
        return x, log_det_sum


def _half_masks(data_dim, n_layers):
    """Alternating half masks: even layers condition on the first half, odd layers on the second
    (real_nvp.py:24-33, real_nvp_spline.py:22-31)."""
    first = torch.zeros(data_dim)
    first[: data_dim // 2] = 1
    return [first.clone() if i % 2 == 0 else 1 - first for i in range(n_layers)]


class _HalfMaskStack(_DensityAPI, nn.Module):
    """RealNVP / RealNVPSpline: n_layers coupling layers of class `_layer` on alternating half masks, wrapped in a
    NormalizingFlowModel at `self.flow` (the reference's state_dict keys)."""
    _layer = None

    def __init__(self, data_dim, n_layers, hidden_dim, batch_norm_between_layers=False, **layer_kwargs):
        super().__init__()
        assert n_layers % 2 == 0, "Number of layers must be even to ensure all dimensions are transformed."
        layers = [self._layer(data_dim, hidden_dim, m, **layer_kwargs) for m in _half_masks(data_dim, n_layers)]
        self.flow = NormalizingFlowModel(layers, batch_norm_between_layers)
        self.context_dim = self.flow.context_dim

    def _log_prob_fused(self, x, ctx=None):
        return self.flow._log_prob_fused(x, ctx)

    def _sample_fused(self, x, draw, ctx=None):
        return self.flow._sample_fused(x, draw, ctx)

    def forward(self, z, context=None):
        return self.flow.forward(z, context)

    def inverse(self, x, context=None):
        return self.flow.inverse(x, context)


class RealNVP(_HalfMaskStack):
    """context_dim = C > 0: every layer is a conditional CouplingLayer reading the one context."""
    _layer = CouplingLayer

    def __init__(self, data_dim, n_layers, hidden_dim, batch_norm_between_layers=False, context_dim=0):
        super().__init__(data_dim, n_layers, hidden_dim, batch_norm_between_layers, context_dim=context_dim)


class RealNVPSpline(_HalfMaskStack):
    """context_dim = C > 0: every layer is a conditional SplineCouplingLayer reading the one context."""
    _layer = SplineCouplingLayer

    def __init__(self, data_dim, n_layers, hidden_dim, batch_norm_between_layers=False, context_dim=0):
        super().__init__(data_dim, n_layers, hidden_dim, batch_norm_between_layers, context_dim=context_dim)
