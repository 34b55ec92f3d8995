"""CPU: the conditional spline-coupling surface (context_dim), without launching a kernel.

- context_dim = 0 builds today's modules: same state_dict keys, shapes and seeded initial weights.
- context_dim = C widens param_net[0] to data_dim + C inputs and keeps every other parameter as it was.
- Every misuse of context raises ValueError before anything runs: a conditional model without context, a context for a
  model without conditional layer, and a context of the wrong width, row count, dtype or device.
- The conditional layout's packed bytes and host header are pinned by SHA-256, as tests/test_stack_plumbing.py pins the
  unconditional ones, and a conditional layer never reaches the unconditional packers.
- The three conditional entry points' refusal codes are pinned for every check they make before a CUDA call.
"""
import ctypes
import hashlib

import numpy as np
import pytest
import torch

import nfb200 as N
from nfb200 import _lib, packing
from tests.test_stack_plumbing import _between, _fill, _masks

OK, BAD_SHAPE, UNSUPPORTED, MISALIGNED, NULL, WORKSPACE = 0, -1, -2, -3, -5, -6


# ------------------------------------------------------------------------------------------------
# module surface
# ------------------------------------------------------------------------------------------------
def _sd(m):
    return {k: v.clone() for k, v in m.state_dict().items()}


@pytest.mark.parametrize("ctor", [
    lambda **kw: N.SplineCouplingLayer(4, 16, torch.tensor([1., 1., 0., 0.]), num_bins=6, **kw),
    lambda **kw: N.RealNVPSpline(6, 2, 32, **kw),
    lambda **kw: N.RealNVPSpline(2, 4, 8, batch_norm_between_layers=True, **kw),
])
def test_context_dim_zero_is_todays_module(ctor):
    torch.manual_seed(3)
    plain = _sd(ctor())
    torch.manual_seed(3)
    zero = _sd(ctor(context_dim=0))
    assert list(plain) == list(zero)
    assert all(torch.equal(plain[k], zero[k]) for k in plain)


def test_conditional_layer_widens_only_the_first_linear():
    torch.manual_seed(0)
    plain = N.SplineCouplingLayer(3, 16, torch.tensor([1., 0., 1.]), num_bins=5)
    cond = N.SplineCouplingLayer(3, 16, torch.tensor([1., 0., 1.]), num_bins=5, context_dim=4)
    assert cond.context_dim == 4 and plain.context_dim == 0
    ps, cs = plain.state_dict(), cond.state_dict()
    assert list(ps) == list(cs)
    for k in ps:
        want = (16, 7) if k == "param_net.0.weight" else tuple(ps[k].shape)
        assert tuple(cs[k].shape) == want, k
    m = N.RealNVPSpline(2, 4, 8, context_dim=3)
    assert m.context_dim == 3 and m.flow.context_dim == 3
    assert all(f.context_dim == 3 and f.param_net[0].in_features == 5 for f in m.flow.flows)


def test_bad_context_dim_is_refused():
    for bad in (-1, 1.5):
        with pytest.raises(ValueError):
            N.SplineCouplingLayer(2, 8, torch.tensor([1., 0.]), context_dim=bad)
    a = N.SplineCouplingLayer(2, 8, torch.tensor([1., 0.]), context_dim=2)
    b = N.SplineCouplingLayer(2, 8, torch.tensor([0., 1.]), context_dim=3)
    with pytest.raises(ValueError):
        N.NormalizingFlowModel([a, b])


# Every case raises before a tensor reaches the library, so the models stay on the CPU here.
def _calls(model, x, c):
    return [lambda: model.log_prob(x, context=c), lambda: model.forward(x, context=c),
            lambda: model.inverse(x, context=c)]


def test_context_errors_raise_value_error():
    torch.manual_seed(0)
    cond = N.RealNVPSpline(2, 2, 8, context_dim=3)
    plain = N.RealNVPSpline(2, 2, 8)
    layer = N.SplineCouplingLayer(2, 8, torch.tensor([1., 0.]), context_dim=3)
    x = torch.randn(5, 2)
    good = torch.randn(5, 3)
    bad = {
        "missing": None,
        "width": torch.randn(5, 2),
        "rows": torch.randn(4, 3),
        "one_dim": torch.randn(3),
        "dtype": good.double(),
        "int": torch.ones(5, 3, dtype=torch.int64),
        "device": good.to("meta"),
    }
    for model in (cond, layer, N.SequentialFlow([layer])):
        for name, c in bad.items():
            for call in _calls(model, x, c):
                with pytest.raises(ValueError):
                    call()
    for call in _calls(plain, x, good) + _calls(N.SplineCouplingLayer(2, 8, torch.tensor([1., 0.])), x, good):
        with pytest.raises(ValueError):
            call()
    for model in (cond, layer):
        with pytest.raises(ValueError):
            model.sample_and_log_prob(4, context=torch.randn(2, 2))
        with pytest.raises(ValueError):
            model.sample_and_log_prob(4)
        with pytest.raises(ValueError):
            model.sample(4, context=torch.randn(2, 3, dtype=torch.float64))
        with pytest.raises(ValueError):
            model.sample(4, context=torch.randn(0, 3))
    with pytest.raises(ValueError):
        plain.sample_and_log_prob(4, context=torch.randn(2, 3))


def test_layered_sampling_expands_the_context_once_per_call():
    """n samples per context row: the layered first Linear of every layer reads one [B, C] expansion, made once."""
    from nfb200.flows import _Context
    c = torch.arange(6.0).view(3, 2)
    ctx = _Context(c, 4)
    a, div = ctx.layered(12)
    assert div == 1 and torch.equal(a, c.repeat_interleave(4, 0))
    assert ctx.layered(12)[0] is a
    assert _Context(c, 1).layered(3)[0] is c
    one = c[:1]
    t, div = _Context(one, 12).layered(12)
    assert t is one and div == 12


# ------------------------------------------------------------------------------------------------
# packed bytes of the conditional layout
# ------------------------------------------------------------------------------------------------
def _cond_model(D, H, L, K=8, dt=1, C=4, bn=False, rescale=False, seed=0):
    rng = np.random.default_rng(seed)
    rs = dict(data_min=torch.from_numpy(rng.uniform(-3, -1, D)).float(),
              data_max=torch.from_numpy(rng.uniform(1, 3, D)).float()) if rescale else {}
    layers = [N.SplineCouplingLayer(D, H, m, num_bins=K, bound=3.0, min_bin_width=2e-3, min_bin_height=3e-3,
                                    min_derivative=4e-3, context_dim=C, **rs) for m in _masks(D, L, dt)]
    _fill(layers, rng)
    for l in layers:
        l.eval()
    return layers, (_between(D, L, rng) if bn else None)


PACK_CASES = {
    "ctx_D1_H8_K2_C1": dict(D=1, H=8, L=2, K=2, dt=1, C=1),
    "ctx_D2_H64_K8_C4_bn": dict(D=2, H=64, L=3, K=8, dt=1, C=4, bn=True),
    "ctx_D2_H64_K8_C8": dict(D=2, H=64, L=2, K=8, dt=1, C=8),
    "ctx_D3_H33_K10_C5_rescale": dict(D=3, H=33, L=2, K=10, dt=2, C=5, rescale=True),
    "ctx_D8_H16_K9_C3_bn_rescale": dict(D=8, H=16, L=2, K=9, dt=2, C=3, bn=True, rescale=True),
    "ctx_refuse_C9": dict(D=2, H=64, L=2, K=8, dt=1, C=9),
    "ctx_refuse_H65": dict(D=2, H=65, L=2, K=8, dt=1, C=4),
    "ctx_refuse_K11": dict(D=2, H=64, L=2, K=11, dt=1, C=4),
}


def _digests(pk):
    if pk is None:
        return None
    packed, hdr = pk
    assert hdr.dtype == np.int32 and hdr.shape == (packing.HDR,)
    return (hashlib.sha256(packed.numpy().tobytes()).hexdigest()[:32], hashlib.sha256(hdr.tobytes()).hexdigest()[:32])


# SHA-256 prefixes of (packed, hdr_host); None: the packer refuses the configuration
PACK_DIGESTS = {
    'ctx_D1_H8_K2_C1': ('2abb3a640e5cedda6c121e56afc4b1f4', '243d7bd5b8ee150e7ae9af1c5c1572ae'),
    'ctx_D2_H64_K8_C4_bn': ('c6b573366c6673d0acefd60b8ecbcba1', '4f222a819cf591f4e77c6ff873cb065e'),
    'ctx_D2_H64_K8_C8': ('6ac8d2c3c7b736eddc39f92057b89f18', '0b8c7fadc244514d69540be5e5a0b176'),
    'ctx_D3_H33_K10_C5_rescale': ('31f271c827633d41022d268d36372378', '6e20fc0f7651386932129ec2ef1f5b54'),
    'ctx_D8_H16_K9_C3_bn_rescale': ('68e3c4f12f5eb3f31695f3ed03d3b63f', '5c8bdcbf190ac6a9c34d10263ea16270'),
    'ctx_refuse_C9': None,
    'ctx_refuse_H65': None,
    'ctx_refuse_K11': None,
}


@pytest.mark.parametrize("name", sorted(PACK_CASES))
def test_conditional_packed_bytes_are_pinned(name):
    assert _digests(packing.pack_spline_stack_ctx_tc(*_cond_model(**PACK_CASES[name]))) == PACK_DIGESTS[name]


def test_conditional_layout():
    """Header word 3 holds C; W1k keeps the x columns; the Wc section holds the context columns in unit pairs."""
    layers, _ = _cond_model(D=2, H=64, L=1, K=8, dt=1, C=3)
    packed, hdr = packing.pack_spline_stack_ctx_tc(layers, None)
    assert hdr[0] == packing.MAGIC_SPLINE_CTX_TC and hdr[3] == 3
    block = packed.numpy()[packing.HDR + packing.LAYER_HDR:]
    W1 = layers[0].param_net[0].weight.detach().numpy()
    w1k = block[:64 * 4].reshape(32, 4, 2)          # pair-interleaved: [w0a w0b | w1a w1b | w2a w2b | ba bb]
    assert np.array_equal(w1k[:, 0, :].ravel(), W1[:, 0]) and np.array_equal(w1k[:, 1, :].ravel(), W1[:, 1])
    wc = block[64 * 4 + 64 + 32:][:64 * packing.CTX_MAX].reshape(32, packing.CTX_MAX, 2)
    for c in range(packing.CTX_MAX):
        want = W1[:, 2 + c] if c < 3 else np.zeros(64, dtype=np.float32)
        assert np.array_equal(wc[:, c, :].ravel(), want), c
    assert packing.pack_spline_stack_tc(layers, None) is None
    assert packing.pack_spline_stack(layers, None) is None


# ------------------------------------------------------------------------------------------------
# refusal codes of the three conditional entry points
# ------------------------------------------------------------------------------------------------
P, X, Y, LD, CTX, STATE = 0x10000, 0x20000, 0x30000, 0x40000, 0x60000, 0x50000


def _header(**over):
    packed, hdr = packing.pack_spline_stack_ctx_tc(*_cond_model(**PACK_CASES["ctx_D2_H64_K8_C4_bn"]))
    hdr = hdr.copy()
    for word, v in over.items():
        hdr[int(word[1:])] = v
    return hdr, packed.numel() * 4


def _call(entry, hdr, nbytes, packed=P, x=X, y=Y, ld=LD, ctx=CTX, rows=1000, div=1, B=1000, flags=0, state=STATE):
    h = None if hdr is None else ctypes.c_void_p(hdr.ctypes.data)
    fn = getattr(_lib.lib(), f"nf_spline_stack_ctx_tc_{entry}")
    if entry == "forward":
        return fn(packed, h, nbytes, x, ctx, rows, div, y, ld, B, flags, None)
    if entry == "sample":
        return fn(packed, h, nbytes, ctx, rows, div, 7, 8, y, ld, B, None)
    return fn(packed, h, nbytes, ctx, rows, div, state, y, ld, B, None)


def _unconditional():
    from tests.test_stack_plumbing import _pack
    packed, hdr = _pack("spline_tc_D2_H64_K8_bn")
    return hdr.copy(), packed.numel() * 4


CASES = {
    "context_null": lambda e: _call(e, *_header(), ctx=None),
    "context_null_B0": lambda e: _call(e, *_header(), ctx=None, B=0) if e != "sample_state" else None,
    "div0": lambda e: _call(e, *_header(), div=0),
    "div_negative": lambda e: _call(e, *_header(), div=-3),
    "rows_short": lambda e: _call(e, *_header(), rows=999),
    "rows_short_div": lambda e: _call(e, *_header(), rows=99, div=10),
    "rows_exact_div_refused_after": lambda e: _call(e, *_header(w3=9), rows=100, div=10),
    "rows_broadcast_refused_after": lambda e: _call(e, *_header(w3=0), rows=1, div=1000),
    "C0": lambda e: _call(e, *_header(w3=0)),
    "C9": lambda e: _call(e, *_header(w3=9)),
    "unconditional_pack": lambda e: _call(e, *_unconditional()),
    "context_null_unconditional_pack": lambda e: _call(e, *_unconditional(), ctx=None),
    "context_null_div0": lambda e: _call(e, *_header(), ctx=None, div=0),
    "div0_C9": lambda e: _call(e, *_header(w3=9), div=0),
    "hdr_null": lambda e: _call(e, None, 0),
    "B_negative": lambda e: _call(e, *_header(), B=-1),
    "packed_misaligned": lambda e: _call(e, *_header(), packed=P + 8),
    "H65": lambda e: _call(e, *_header(w2=65)),
    "K11": lambda e: _call(e, *_header(w4=11)),
    "stride_unconditional": lambda e: _call(e, *_header(w8=_unconditional()[0][8])),
    "bytes_one_word_short": lambda e: _call(e, _header()[0], _header()[1] - 4),
    "state_null": lambda e: _call(e, *_header(), state=None) if e == "sample_state" else None,
}
ENTRIES = ("forward", "sample", "sample_state")


def _statuses(case):
    return " ".join("." if rc is None else str(rc) for rc in (CASES[case](e) for e in ENTRIES))


# case -> status of forward, sample, sample_state ("." where the case does not apply)
REFUSALS = {
    'context_null': '-5 -5 -5',
    'context_null_B0': '0 0 .',
    'div0': '-1 -1 -1',
    'div_negative': '-1 -1 -1',
    'rows_short': '-1 -1 -1',
    'rows_short_div': '-1 -1 -1',
    'rows_exact_div_refused_after': '-2 -2 -2',
    'rows_broadcast_refused_after': '-2 -2 -2',
    'C0': '-2 -2 -2',
    'C9': '-2 -2 -2',
    'unconditional_pack': '-1 -1 -1',
    'context_null_unconditional_pack': '-1 -1 -1',
    'context_null_div0': '-5 -5 -5',
    'div0_C9': '-1 -1 -1',
    'hdr_null': '-5 -5 -5',
    'B_negative': '-1 -1 -1',
    'packed_misaligned': '-3 -3 -3',
    'H65': '-2 -2 -2',
    'K11': '-2 -2 -2',
    'stride_unconditional': '-1 -1 -1',
    'bytes_one_word_short': '-6 -6 -6',
    'state_null': '. . -5',
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_conditional_refusal_codes_are_pinned(case):
    assert _statuses(case) == REFUSALS[case]


def test_unconditional_entry_points_refuse_a_conditional_pack():
    hdr, nbytes = _header()
    for stem in ("nf_spline_stack_tc", "nf_spline_stack"):
        fn = getattr(_lib.lib(), stem + "_forward")
        assert fn(P, ctypes.c_void_p(hdr.ctypes.data), nbytes, X, Y, LD, 1000, 0, None) == BAD_SHAPE


def _record():
    print("PACK_DIGESTS = {")
    for name in sorted(PACK_CASES):
        print(f"    {name!r}: {_digests(packing.pack_spline_stack_ctx_tc(*_cond_model(**PACK_CASES[name])))!r},")
    print("}")
    print("REFUSALS = {")
    for case in CASES:
        print(f"    {case!r}: {_statuses(case)!r},")
    print("}")


if __name__ == "__main__":
    _record()
