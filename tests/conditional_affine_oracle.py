"""Reference for conditional affine coupling flows, p(x | c), in plain torch.

A conditional CouplingLayer (context_dim = C > 0) feeds [x * mask, c] to both s_net and b_net, the context columns last
as in nflows and in the conditional spline layer; the context is not masked.  Everything after the first Linear -- the
conditioner BatchNorms, the clamps, the affine transform, the scrubs and the between-layer BatchNorm -- is the
unconditional oracle's (oracle/flows_oracle.py), and conditional spline layers are tests/conditional_oracle.py's.  With
C = 0, affine_coupling computes exactly what O.affine_coupling computes."""
from typing import Sequence, Tuple

import torch
from torch import Tensor

from oracle import flows_oracle as O
from tests import conditional_oracle as CO


def affine_coupling(sd, p: str, x: Tensor, context: Tensor, inverse: bool, training=False) -> Tuple[Tensor, Tensor]:
    """O.affine_coupling with context [B, C] (or [1, C], broadcast) appended to the input of s_net and b_net.
    training=True: the conditioner BatchNorms normalise with the batch statistics of their input (the first Linear of the
    concatenated input, context included) and leave `sd` untouched."""
    m = sd[p + "mask"]
    x_a = x * m
    inp = x_a
    if sd[p + "s_net.0.weight"].shape[1] > m.numel():
        inp = torch.cat([x_a, context.to(x.dtype).expand(x.shape[0], -1)], dim=1)
    s = torch.clamp(O.coupling_conditioner(sd, p + "s_net", inp, training), -10.0, 10.0)
    b = torch.clamp(O.coupling_conditioner(sd, p + "b_net", inp, training), -10.0, 10.0)
    if not inverse:
        y = x_a + (1 - m) * (x * torch.exp(s) + b)
        ld = ((1 - m) * s).sum(dim=1)
    else:
        y = x_a + (1 - m) * ((x - b) * torch.exp(-s))
        ld = ((1 - m) * -s).sum(dim=1)
    return O._scrub_zero(y), O._scrub_zero(ld)


def flow_model(sd, p: str, specs: Sequence[dict], x: Tensor, context: Tensor, inverse: bool,
               bn_between=False, training=False) -> Tuple[Tensor, Tensor]:
    """CO.flow_model over coupling layers that all read `context`, spec["kind"] "affine" or "spline" (the other keys:
    the spline layer's arguments).  The between-layer BatchNorm does not see the context and uses its running statistics.
    training=True: the affine layers' conditioner BatchNorms use batch statistics."""
    L = len(specs)
    total = 0
    order = reversed(range(L)) if inverse else range(L)
    for i in order:
        q = f"{p}batch_norms.{i}"
        if inverse and bn_between and i < L - 1:
            x = (x - sd[q + ".bias"]) / sd[q + ".weight"] * torch.sqrt(sd[q + ".running_var"] + O.BN_EPS) \
                + sd[q + ".running_mean"]
            total = total - O._bn_between_logdet(sd, q)
        if specs[i]["kind"] == "affine":
            x, ld = affine_coupling(sd, f"{p}flows.{i}.", x, context, inverse, training)
        else:
            kw = {k: v for k, v in specs[i].items() if k != "kind"}
            x, ld = CO.spline_coupling(sd, f"{p}flows.{i}.", x, context, inverse, **kw)
        total = total + ld
        if not inverse and bn_between and i < L - 1:
            x = (x - sd[q + ".running_mean"]) / torch.sqrt(sd[q + ".running_var"] + O.BN_EPS) * sd[q + ".weight"] \
                + sd[q + ".bias"]
            total = total + O._bn_between_logdet(sd, q)
    return x, total
