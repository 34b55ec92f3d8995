"""Reference for conditional spline coupling flows, p(x | c), in plain torch.

A conditional SplineCouplingLayer (context_dim = C > 0) feeds [x_rescaled * mask, c] to its conditioner, the context
columns last as in nflows; the context is neither rescaled nor masked.  Everything after the first Linear -- the spline,
its tails, the scrubs and the between-layer BatchNorm -- is the unconditional oracle's (oracle/flows_oracle.py), which
these functions call.  With C = 0 they compute exactly what O.spline_coupling / O.flow_model compute (eval mode)."""
from typing import Sequence, Tuple

import torch
import torch.nn.functional as F
from torch import Tensor

from oracle import flows_oracle as O


def spline_coupling(sd, p: str, x: Tensor, context: Tensor, inverse: bool, num_bins=10, bound=5.0, min_bin_width=1e-3,
                    min_bin_height=1e-3, min_derivative=1e-3, data_min=None, data_max=None) -> Tuple[Tensor, Tensor]:
    """O.spline_coupling with context [B, C] (or [1, C], broadcast) appended to the conditioner input."""
    m = sd[p + "mask"]
    D, K = m.numel(), num_bins
    W0 = sd[p + "param_net.0.weight"]
    rescale = data_min is not None and data_max is not None
    xr = (2 * bound) / (data_max - data_min) * (x - data_min) - bound if rescale else x
    x_a = xr * m
    if W0.shape[1] > D:
        x_a = torch.cat([x_a, context.to(x.dtype).expand(x.shape[0], -1)], dim=1)
    h = torch.relu(F.linear(x_a, W0, sd[p + "param_net.0.bias"]))
    h = torch.relu(F.linear(h, sd[p + "param_net.2.weight"], sd[p + "param_net.2.bias"]))
    params = F.linear(h, sd[p + "param_net.4.weight"], sd[p + "param_net.4.bias"]).view(-1, D, 3 * K - 1)
    uw, uh, ud = torch.split(params, [K, K, K - 1], dim=-1)
    tr = m == 0
    out_b, ld_b = O.rqs_bounded(xr[:, tr], uw[:, tr], uh[:, tr], ud[:, tr], inverse, bound, min_bin_width,
                                min_bin_height, min_derivative)
    if rescale:
        out_b = (out_b + bound) * ((data_max - data_min) / (2 * bound)) + data_min
    y = x.clone()
    y[:, tr] = out_b
    return O._scrub_zero(y), O._scrub_zero(ld_b.sum(dim=1))


def flow_model(sd, p: str, specs: Sequence[dict], x: Tensor, context: Tensor, inverse: bool,
               bn_between=False) -> Tuple[Tensor, Tensor]:
    """O.flow_model (eval mode) over spline layers that all read `context`; the between-layer BatchNorm does not."""
    L = len(specs)
    total = 0
    order = reversed(range(L)) if inverse else range(L)
    for i in order:
        kw = {k: v for k, v in specs[i].items() if k != "kind"}
        q = f"{p}batch_norms.{i}"
        if inverse and bn_between and i < L - 1:
            x = (x - sd[q + ".bias"]) / sd[q + ".weight"] * torch.sqrt(sd[q + ".running_var"] + O.BN_EPS) \
                + sd[q + ".running_mean"]
            total = total - O._bn_between_logdet(sd, q)
        x, ld = spline_coupling(sd, f"{p}flows.{i}.", x, context, inverse, **kw)
        total = total + ld
        if not inverse and bn_between and i < L - 1:
            x = (x - sd[q + ".running_mean"]) / torch.sqrt(sd[q + ".running_var"] + O.BN_EPS) * sd[q + ".weight"] \
                + sd[q + ".bias"]
            total = total + O._bn_between_logdet(sd, q)
    return x, total
