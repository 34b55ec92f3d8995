"""CPU: pin oracle/flows_oracle.py to golden vectors produced by the unmodified reference
(tests/golden/make_golden.py).  The oracle issues the same ATen ops as the reference, so
the comparison is bit-exact except where noted."""
import pytest
import torch

from oracle import flows_oracle as O
from tests import golden_util as G

EVAL_KINDS = ("coupling", "spline", "rqs_bounded", "rqs_unit", "maf", "iaf", "realnvp", "realnvpspline",
              "splinestack", "mixed", "sequential", "arqs")
# ATen's CPU BatchNorm splits the batch statistics across the intra-op threads, so their float32 rounding depends on the
# thread count; the train-mode goldens were produced with 8 threads and reproduce bit for bit only with 8.
GOLDEN_THREADS = 8


@pytest.fixture
def golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def _same(a, b):
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    assert a.shape == b.shape
    assert torch.equal(torch.isnan(a), torch.isnan(b))
    ok = torch.isnan(a) | (a == b)
    assert bool(ok.all()), f"max abs diff {(a - b)[~ok].abs().max().item():.3e}"


@pytest.mark.parametrize("name", G.golden_names())
def test_oracle_matches_reference_golden(name):
    g = G.load(name)
    if g["kind"] not in EVAL_KINDS:
        pytest.skip("train-mode case, see test_oracle_train_mode")
    for inverse, key in ((False, "fwd"), (True, "inv")):
        y, ld = G.oracle_eval(g, inverse)
        _same(y, g[key])
        _same(ld, g[key + "_ld"])


@pytest.mark.parametrize("name", G.golden_names("coupling_train"))
def test_oracle_train_mode_coupling(name, golden_threads):
    """BatchNorm batch statistics + running-stat side effects (coupling_layer.py:20,23)."""
    g = G.load(name)
    sd = {k: v.clone() for k, v in g["sd"].items()}
    with torch.no_grad():
        y, ld = O.affine_coupling(sd, "", g["x"], False, training=True, update=True)
    _same(y, g["fwd"])
    _same(ld, g["fwd_ld"])
    for k, v in g["sd_after"].items():
        _same(sd[k], v)


@pytest.mark.parametrize("name", G.golden_names("mafbn_train") + G.golden_names("iafbn_train"))
def test_oracle_train_mode_made_batch_norm(name, golden_threads):
    """MADE(use_batch_norm=True) in train mode: batch statistics + running-stat side effects (made.py:93-108)."""
    g = G.load(name)
    sd = {k: v.clone() for k, v in g["sd"].items()}
    with torch.no_grad():
        fn = O.maf_inverse if g["kind"] == "maf_train" else O.iaf_forward
        y, ld = fn(sd, "", g["x"], training=True, update=True)
    _same(y, g["out"])
    _same(ld, g["out_ld"])
    for k, v in g["sd_after"].items():
        _same(sd[k], v)


def test_oracle_train_mode_between_layer_bn(golden_threads):
    """normalizing_flow_model.py:74-79: running stats updated, affine uses running stats."""
    g = G.load("realnvp_4_4_16_bn_train")
    sd = {k: v.clone() for k, v in g["sd"].items()}
    with torch.no_grad():
        y, ld = O.flow_model(sd, "flow.", [dict(kind="coupling")] * g["L"], g["x"], False,
                             bn_between=True, training=True, update=True)
    _same(y, g["fwd"])
    _same(ld, g["fwd_ld"])
    for k, v in g["sd_after"].items():
        _same(sd[k], v)


@pytest.mark.parametrize("name", G.golden_names("maf_") + G.golden_names("iaf_"))
def test_made_masks_and_degrees(name):
    g = G.load(name)
    D, H = g["D"], g["H"]
    _, m_h = O.made_degrees(D, H)
    assert torch.equal(torch.as_tensor(m_h), g["degrees"])
    masks = O.made_masks(D, H)
    for idx, mk in zip((0, 2, 4, 6), (masks[0], masks[1], masks[1], masks[2])):
        assert torch.equal(mk, g["sd"][f"conditioner.net.{idx}.mask"])


def test_init_builders_have_reference_key_layout():
    """oracle.init_* produce exactly the reference's state_dict keys/shapes (SURVEY A.2)."""
    g = G.load("realnvpspline_2_8_64")
    sd = O.init_spline_stack_sd(2, 8, 64, 10)
    assert {k: tuple(v.shape) for k, v in sd.items()} == {k: tuple(v.shape) for k, v in g["sd"].items()}
    g = G.load("realnvp_4_4_16_bn")
    sd = O.init_coupling_stack_sd(4, 4, 16, bn_between=True)
    assert {k: tuple(v.shape) for k, v in sd.items()} == {k: tuple(v.shape) for k, v in g["sd"].items()}
    g = G.load("maf_D5_H32")
    sd = O.init_made_sd(5, 32)
    assert {k: tuple(v.shape) for k, v in sd.items()} == {k: tuple(v.shape) for k, v in g["sd"].items()}
