"""Load golden fixtures (tests/golden/*.pt) and evaluate the oracle on them."""
import glob
import os

import torch

from oracle import flows_oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_names(prefix=""):
    return sorted(os.path.basename(p)[:-3] for p in glob.glob(os.path.join(GOLDEN_DIR, prefix + "*.pt")))


def load(name):
    return torch.load(os.path.join(GOLDEN_DIR, name + ".pt"), map_location="cpu", weights_only=False)


def stack_specs(g):
    """Layer spec list for the stacked-model goldens."""
    k = g["kind"]
    if k in ("realnvp", "realnvp_train"):
        return "flow.", [dict(kind="coupling")] * g["L"]
    if k == "realnvpspline":
        return "flow.", [dict(kind="spline", num_bins=g["K"])] * g["L"]
    if k == "splinestack":
        return "", [dict(kind="spline", num_bins=g["K"])] * g["L"]
    if k in ("mixed", "sequential"):
        return "", g["specs"]
    raise ValueError(k)


def oracle_eval(g, inverse, grad=False, training=False):
    """Run the oracle on golden case `g` in one direction; returns (y, ld).  grad=True keeps the autograd graph (the
    state_dict `g["sd"]` may hold leaves that require grad); training=True evaluates the conditioners' BatchNorms on
    batch statistics without moving their running statistics (update=False)."""
    with torch.set_grad_enabled(grad):
        return _oracle_eval(g, inverse, training)


def _oracle_eval(g, inverse, training):
    k = g["kind"]
    x = g["x"]
    if k == "coupling":
        return O.affine_coupling(g["sd"], "", x, inverse, training=training)
    if k == "spline":
        return O.spline_coupling(g["sd"], "", x, inverse, num_bins=g["K"], **g["extra"])
    if k == "rqs_bounded":
        return O.rqs_bounded(x, g["uw"], g["uh"], g["ud"], inverse, bound=g["bound"])
    if k == "rqs_unit":
        return O.rqs_unit(x, g["w"], g["h"], g["d"], inverse)
    if k == "maf":
        return O.maf_inverse(g["sd"], "", x, training=training) if inverse else O.maf_forward(g["sd"], "", x)
    if k == "iaf":
        return O.iaf_inverse(g["sd"], "", x) if inverse else O.iaf_forward(g["sd"], "", x, training=training)
    if k == "arqs":
        return O.arqs(g["sd"], "", x, inverse, num_bins=g["K"], **g["extra"])
    p, specs = stack_specs(g)
    if k == "sequential":
        return O.sequential_flow(g["sd"], p, specs, x, inverse)
    return O.flow_model(g["sd"], p, specs, x, inverse, bn_between=g.get("bn", False), training=training)
