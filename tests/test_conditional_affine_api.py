"""CPU: the conditional affine-coupling surface (CouplingLayer / RealNVP with context_dim), without launching a kernel.

- context_dim = 0 builds today's modules: same state_dict keys, shapes and seeded initial weights.
- context_dim = C widens s_net[0] and b_net[0] to data_dim + C inputs and keeps every other parameter as it was.
- Every misuse of context raises ValueError before anything runs, as for the conditional spline layers.
- The conditional layout 'NFD2': each net block's Wc section holds the BatchNorm-folded context columns of its first
  Linear in unit pairs, and with zero context columns every other word is the unconditional 'NFA2' pack's word.  A
  conditional layer never reaches the unconditional packers.
- The three conditional entry points' refusal codes for every check they make before a CUDA call.
"""
import ctypes

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
    lambda **kw: N.CouplingLayer(4, 16, torch.tensor([1., 1., 0., 0.]), **kw),
    lambda **kw: N.RealNVP(6, 2, 32, **kw),
    lambda **kw: N.RealNVP(2, 4, 8, batch_norm_between_layers=True, **kw),
])
def test_context_dim_zero_is_todays_module(ctor):
    torch.manual_seed(3)
    plain = _sd(ctor())
    torch.manual_seed(3)
    zero = _sd(ctor(context_dim=0))
    assert list(plain) == list(zero)
    assert all(torch.equal(plain[k], zero[k]) for k in plain)


def test_conditional_layer_widens_only_the_first_linears():
    torch.manual_seed(0)
    plain = N.CouplingLayer(3, 16, torch.tensor([1., 0., 1.]))
    cond = N.CouplingLayer(3, 16, torch.tensor([1., 0., 1.]), context_dim=4)
    assert cond.context_dim == 4 and plain.context_dim == 0
    ps, cs = plain.state_dict(), cond.state_dict()
    assert list(ps) == list(cs)
    for k in ps:
        want = (16, 7) if k in ("s_net.0.weight", "b_net.0.weight") else tuple(ps[k].shape)
        assert tuple(cs[k].shape) == want, k
    m = N.RealNVP(2, 4, 8, context_dim=3)
    assert m.context_dim == 3 and m.flow.context_dim == 3
    assert all(f.context_dim == 3 and f.s_net[0].in_features == 5 and f.b_net[0].in_features == 5 for f in m.flow.flows)


def test_bad_context_dim_is_refused():
    for bad in (-1, 1.5):
        with pytest.raises(ValueError):
            N.CouplingLayer(2, 8, torch.tensor([1., 0.]), context_dim=bad)
        with pytest.raises(ValueError):
            N.RealNVP(2, 2, 8, context_dim=bad)
    a = N.CouplingLayer(2, 8, torch.tensor([1., 0.]), context_dim=2)
    b = N.CouplingLayer(2, 8, torch.tensor([0., 1.]), context_dim=3)
    with pytest.raises(ValueError):
        N.NormalizingFlowModel([a, b])
    s = N.SplineCouplingLayer(2, 8, torch.tensor([0., 1.]), context_dim=3)
    with pytest.raises(ValueError):
        N.NormalizingFlowModel([a, s])
    mixed = N.NormalizingFlowModel([N.CouplingLayer(2, 8, torch.tensor([1., 0.]), context_dim=3), s])
    assert mixed.context_dim == 3


# Every case raises before a tensor reaches the library, so the models stay on the CPU here.
def _calls(model, x, c):
    return [lambda: model.log_prob(x, context=c), lambda: model.forward(x, context=c),
            lambda: model.inverse(x, context=c)]


def test_context_errors_raise_value_error():
    torch.manual_seed(0)
    cond = N.RealNVP(2, 2, 8, context_dim=3)
    plain = N.RealNVP(2, 2, 8)
    layer = N.CouplingLayer(2, 8, torch.tensor([1., 0.]), context_dim=3)
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
    for call in _calls(plain, x, good) + _calls(N.CouplingLayer(2, 8, torch.tensor([1., 0.])), x, good):
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


# ------------------------------------------------------------------------------------------------
# packed layout 'NFD2'
# ------------------------------------------------------------------------------------------------
def _cond_model(D, H, L, dt=1, C=4, bn=False, seed=0):
    """Conditional CouplingLayers with every parameter and every conditioner BatchNorm statistic perturbed."""
    rng = np.random.default_rng(seed)
    layers = [N.CouplingLayer(D, H, m, context_dim=C) for m in _masks(D, L, dt)]
    _fill(layers, rng)
    for l in layers:
        l.eval()
    return layers, (_between(D, L, rng) if bn else None)


def _folded_first(net):
    """The first Linear of one conditioner with its eval-mode BatchNorm folded in, in float64: [H, D + C], [H]."""
    W = net[0].weight.detach().double()
    bn = net[1]
    s = bn.weight.detach().double() / torch.sqrt(bn.running_var.double() + bn.eps)
    return (W * s[:, None]).numpy(), ((net[0].bias.detach().double() - bn.running_mean.double()) * s + bn.bias.detach().double()).numpy()


def _blocks(packed, L, nbw):
    return packed.numpy()[packing.HDR:].reshape(2 * L, nbw)


LAYOUT_CASES = [dict(D=1, H=8, L=2, C=1), dict(D=2, H=64, L=3, C=4, bn=True), dict(D=3, H=100, L=2, dt=2, C=8),
                dict(D=5, H=33, L=2, dt=2, C=3), dict(D=8, H=128, L=2, dt=4, C=5, bn=True)]


@pytest.mark.parametrize("case", LAYOUT_CASES, ids=lambda c: "_".join(f"{k}{v}" for k, v in c.items()))
def test_wc_sections_hold_the_folded_context_columns(case):
    layers, bns = _cond_model(**case)
    D, H, C, L = case["D"], case["H"], case["C"], case["L"]
    HP, W1S = (64 if H <= 64 else 128), (4 if D <= 3 else 12)
    packed, hdr = packing.pack_coupling_stack_ctx_tc(layers, bns)
    nbw = _lib.lib().nf_coupling_stack_ctx_tc_block_words_hidden(D, H)
    assert hdr[0] == packing.MAGIC_AFFINE_CTX_TC and hdr[3] == C and hdr[8] == nbw and hdr[5] == L
    wc_at = packing.LAYER_HDR + HP * W1S + HP + 16
    for i, l in enumerate(layers):
        for j, net in enumerate((l.s_net, l.b_net)):
            blk = _blocks(packed, L, nbw)[2 * i + j]
            W, _ = _folded_first(net)
            wc = blk[wc_at:wc_at + HP * packing.CTX_MAX].reshape(HP // 2, packing.CTX_MAX, 2)
            for c in range(packing.CTX_MAX):
                want = np.zeros(HP, dtype=np.float32)
                if c < C:
                    want[:H] = W[:, D + c]
                assert np.array_equal(wc[:, c, :].ravel(), want), (i, j, c)


@pytest.mark.parametrize("case", LAYOUT_CASES, ids=lambda c: "_".join(f"{k}{v}" for k, v in c.items()))
def test_zero_context_columns_give_the_unconditional_words(case):
    """Every word of 'NFD2' outside the Wc section and its padding is the word of 'NFA2' for the same model without the
    context columns; only the magic, header word 3 (C instead of 2 nets) and the block stride differ in the header."""
    layers, bns = _cond_model(**case)
    D, H, C, L = case["D"], case["H"], case["C"], case["L"]
    HP, W1S = (64 if H <= 64 else 128), (4 if D <= 3 else 12)
    plain = [N.CouplingLayer(D, H, l.mask.clone()) for l in layers]
    with torch.no_grad():
        for l, p in zip(layers, plain):
            for net in (l.s_net, l.b_net):
                net[0].weight[:, D:] = 0
            sd = {k: (v[:, :D] if k.endswith("net.0.weight") else v) for k, v in l.state_dict().items()}
            p.load_state_dict(sd)
            p.eval()
    packed, hdr = packing.pack_coupling_stack_ctx_tc(layers, bns)
    packed0, hdr0 = packing.pack_coupling_stack_tc(plain, bns)
    diff = [w for w in range(packing.HDR) if hdr[w] != hdr0[w]]
    assert diff == [0, 3, 8] and hdr0[3] == 2 and hdr[3] == C
    nbw, nbw0 = int(hdr[8]), int(hdr0[8])
    small = packing.LAYER_HDR + HP * W1S + HP + 16
    images = 2 * HP * HP + 2 * 16 * HP                 # W2 hi / lo, W3 hi / lo
    blocks, blocks0 = _blocks(packed, L, nbw), _blocks(packed0, L, nbw0)
    for b, b0 in zip(blocks, blocks0):
        assert np.array_equal(b[:small], b0[:small])
        assert not b[small:nbw - images].any()
        assert np.array_equal(b[nbw - images:], b0[nbw0 - images:])
    assert nbw == _lib.lib().nf_coupling_stack_ctx_tc_block_words_hidden(D, H)
    assert nbw0 == _lib.lib().nf_coupling_stack_tc_block_words_hidden(D, H)


def test_packers_keep_conditional_and_unconditional_layers_apart():
    layers, bns = _cond_model(D=2, H=64, L=2, C=4)
    assert packing.pack_coupling_stack_tc(layers, bns) is None
    assert packing.pack_coupling_stack(layers, bns) is None
    assert packing.pack_coupling_stack_ctx_tc(layers, bns) is not None
    plain = [N.CouplingLayer(2, 64, m).eval() for m in _masks(2, 2, 1)]
    assert packing.pack_coupling_stack_ctx_tc(plain, None) is None
    assert packing.pack_coupling_stack_ctx_tc(_cond_model(D=2, H=64, L=2, C=9)[0], None) is None
    assert packing.pack_coupling_stack_ctx_tc(_cond_model(D=2, H=129, L=2, C=4)[0], None) is None
    assert packing.pack_coupling_stack_ctx_tc(_cond_model(D=9, H=64, L=2, C=4)[0], None) is None
    mixed = _cond_model(D=2, H=64, L=1, C=4)[0] + _cond_model(D=2, H=64, L=1, C=3)[0]
    assert packing.pack_coupling_stack_ctx_tc(mixed, None) is None


def test_block_words():
    lib = _lib.lib()
    # with the Wc section the weight images move by whole 256-word steps: HP * 8 words, rounded up
    assert lib.nf_coupling_stack_ctx_tc_block_words_hidden(2, 64) - lib.nf_coupling_stack_tc_block_words_hidden(2, 64) == 512
    assert lib.nf_coupling_stack_ctx_tc_block_words_hidden(8, 128) - lib.nf_coupling_stack_tc_block_words_hidden(8, 128) == 1024
    for D, H in ((0, 64), (9, 64), (2, 0), (2, 129)):
        assert lib.nf_coupling_stack_ctx_tc_block_words_hidden(D, H) == -1


# ------------------------------------------------------------------------------------------------
# refusal codes of the three conditional entry points
# ------------------------------------------------------------------------------------------------
P, X, Y, LD, CTX, STATE = 0x10000, 0x20000, 0x30000, 0x40000, 0x60000, 0x50000


def _header(**over):
    packed, hdr = packing.pack_coupling_stack_ctx_tc(*_cond_model(D=2, H=64, L=3, C=4, bn=True))
    hdr = hdr.copy()
    for word, v in over.items():
        hdr[int(word[1:])] = v
    return hdr, packed.numel() * 4


def _unconditional():
    layers, bns = _cond_model(D=2, H=64, L=3, C=0, bn=True)
    packed, hdr = packing.pack_coupling_stack_tc(layers, bns)
    return hdr.copy(), packed.numel() * 4


def _call(entry, hdr, nbytes, packed=P, x=X, y=Y, ld=LD, ctx=CTX, rows=1000, div=1, B=1000, flags=0, state=STATE):
    h = None if hdr is None else ctypes.c_void_p(hdr.ctypes.data)
    fn = getattr(_lib.lib(), f"nf_coupling_stack_ctx_tc_{entry}")
    if entry == "forward":
        return fn(packed, h, nbytes, x, ctx, rows, div, y, ld, B, flags, None)
    if entry == "sample":
        return fn(packed, h, nbytes, ctx, rows, div, 7, 8, y, ld, B, None)
    return fn(packed, h, nbytes, ctx, rows, div, state, y, ld, B, None)


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
    "B_over_32_bits": lambda e: _call(e, *_header(), B=1 << 31, rows=1 << 31),
    "div_over_32_bits": lambda e: _call(e, *_header(), div=1 << 31, rows=1),
    "unconditional_pack": lambda e: _call(e, *_unconditional()),
    "context_null_unconditional_pack": lambda e: _call(e, *_unconditional(), ctx=None),
    "context_null_div0": lambda e: _call(e, *_header(), ctx=None, div=0),
    "div0_C9": lambda e: _call(e, *_header(w3=9), div=0),
    "hdr_null": lambda e: _call(e, None, 0),
    "B_negative": lambda e: _call(e, *_header(), B=-1),
    "packed_misaligned": lambda e: _call(e, *_header(), packed=P + 8),
    "H129": lambda e: _call(e, *_header(w2=129)),
    "D9": lambda e: _call(e, *_header(w1=9)),
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
    'B_over_32_bits': '-2 -2 -2',
    'div_over_32_bits': '-2 -2 -2',
    'unconditional_pack': '-1 -1 -1',
    'context_null_unconditional_pack': '-1 -1 -1',
    'context_null_div0': '-5 -5 -5',
    'div0_C9': '-1 -1 -1',
    'hdr_null': '-5 -5 -5',
    'B_negative': '-1 -1 -1',
    'packed_misaligned': '-3 -3 -3',
    'H129': '-2 -2 -2',
    'D9': '-2 -2 -2',
    'stride_unconditional': '-1 -1 -1',
    'bytes_one_word_short': '-6 -6 -6',
    'state_null': '. . -5',
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_conditional_refusal_codes(case):
    assert _statuses(case) == REFUSALS[case]


def test_unconditional_entry_points_refuse_a_conditional_pack():
    hdr, nbytes = _header()
    for stem in ("nf_coupling_stack_tc", "nf_coupling_stack"):
        fn = getattr(_lib.lib(), stem + "_forward")
        assert fn(P, ctypes.c_void_p(hdr.ctypes.data), nbytes, X, Y, LD, 1000, 0, None) == BAD_SHAPE
