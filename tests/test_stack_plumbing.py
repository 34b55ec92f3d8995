"""Host-side plumbing of the five fused-stack families, pinned without a GPU.

- Packed bytes: every packer (FP32-pipe spline / affine coupling, tcgen05 spline / affine coupling / MADE) is run on CPU
  modules whose weights and statistics come from a seeded numpy generator, and the SHA-256 of the packed buffer and of
  the host header must equal the recorded values.  The between-layer BatchNorm uses eps = 0, running_var = 1 and
  gamma = +-1, so its log-det word is log(1) = 0 on every libm; all other values are random.
- Refusal codes: each of the 15 fused entry points is called with host-side arguments that are refused before any CUDA
  call (the pointers are never dereferenced), and the status must equal the recorded one.  A call that passed every
  check would launch, so every case here fails a check or returns at B == 0 without a device state.
"""
import ctypes
import hashlib

import numpy as np
import pytest
import torch
import torch.nn as nn

import nfb200 as N
from nfb200 import _lib, packing

OK, BAD_SHAPE, UNSUPPORTED, MISALIGNED, NULL, WORKSPACE = 0, -1, -2, -3, -5, -6


# ------------------------------------------------------------------------------------------------
# packed bytes
# ------------------------------------------------------------------------------------------------
def _masks(D, L, dt):
    """Layer i transforms dims (i*dt + j) % D, j < dt (dt = 0: identity layers)."""
    out = []
    for i in range(L):
        m = torch.ones(D)
        for j in range(dt):
            m[(i * dt + j) % D] = 0
        out.append(m)
    return out


def _fill(mods, rng):
    with torch.no_grad():
        for mod in mods:
            for p in mod.parameters():
                p.copy_(torch.from_numpy(rng.uniform(-0.5, 0.5, tuple(p.shape))))
            for m in mod.modules():
                if isinstance(m, nn.BatchNorm1d):
                    m.running_mean.copy_(torch.from_numpy(rng.uniform(-0.5, 0.5, m.num_features)))
                    m.running_var.copy_(torch.from_numpy(rng.uniform(0.5, 2.0, m.num_features)))


def _between(D, L, rng):
    bns = [nn.BatchNorm1d(D, eps=0.0) for _ in range(L)]
    with torch.no_grad():
        for bn in bns:
            bn.running_mean.copy_(torch.from_numpy(rng.uniform(-0.5, 0.5, D)))
            bn.running_var.fill_(1.0)
            bn.weight.copy_(torch.from_numpy(rng.choice([-1.0, 1.0], D)))
            bn.bias.copy_(torch.from_numpy(rng.uniform(-0.5, 0.5, D)))
    return bns


def _model(kind, D, H, L, K=8, dt=1, bn=False, rescale=False, use_bn=False, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "spline":
        rs = dict(data_min=torch.from_numpy(rng.uniform(-3, -1, D)).float(),
                  data_max=torch.from_numpy(rng.uniform(1, 3, D)).float()) if rescale else {}
        layers = [N.SplineCouplingLayer(D, H, m, num_bins=K, bound=3.0, min_bin_width=2e-3, min_bin_height=3e-3,
                                        min_derivative=4e-3, **rs) for m in _masks(D, L, dt)]
    elif kind == "coupling":
        layers = [N.CouplingLayer(D, H, m) for m in _masks(D, L, dt)]
    else:
        layers = [N.MaskedAutoregressiveFlow(D, H, use_batch_norm=use_bn) for _ in range(L)]
    _fill(layers, rng)
    for l in layers:
        l.eval()
    return layers, (_between(D, L, rng) if bn else None)


PACKERS = {"spline": packing.pack_spline_stack, "spline_tc": packing.pack_spline_stack_tc,
           "coupling": packing.pack_coupling_stack, "coupling_tc": packing.pack_coupling_stack_tc,
           "made_tc": packing.pack_made_stack_tc}

# name -> (packer, model kwargs)
PACK_CASES = {
    "spline_D1_H8_K2": ("spline", dict(D=1, H=8, L=2, K=2, dt=1)),
    "spline_D2_H64_K8_bn": ("spline", dict(D=2, H=64, L=3, K=8, dt=1, bn=True)),
    "spline_D3_H65_K10_rescale": ("spline", dict(D=3, H=65, L=2, K=10, dt=2, rescale=True)),
    "spline_D4_H128_K16_bn_rescale": ("spline", dict(D=4, H=128, L=2, K=16, dt=2, bn=True, rescale=True)),
    "spline_D8_H64_K10_dt4_bn": ("spline", dict(D=8, H=64, L=2, K=10, dt=4, bn=True)),
    "spline_D8_H128_K8_dt4_rescale": ("spline", dict(D=8, H=128, L=2, K=8, dt=4, rescale=True)),
    "spline_refuse_K17": ("spline", dict(D=2, H=8, L=2, K=17, dt=1)),
    "spline_tc_D1_H8_K2": ("spline_tc", dict(D=1, H=8, L=2, K=2, dt=1)),
    "spline_tc_D2_H64_K8_bn": ("spline_tc", dict(D=2, H=64, L=3, K=8, dt=1, bn=True)),
    "spline_tc_D3_H33_K10_rescale": ("spline_tc", dict(D=3, H=33, L=2, K=10, dt=2, rescale=True)),
    "spline_tc_D4_H64_K2_bn_rescale": ("spline_tc", dict(D=4, H=64, L=2, K=2, dt=2, bn=True, rescale=True)),
    "spline_tc_D8_H16_K8_dt1": ("spline_tc", dict(D=8, H=16, L=2, K=8, dt=1)),
    "spline_tc_refuse_H65": ("spline_tc", dict(D=2, H=65, L=2, K=8, dt=1)),
    "coupling_D1_H8": ("coupling", dict(D=1, H=8, L=2, dt=1)),
    "coupling_D2_H64_bn": ("coupling", dict(D=2, H=64, L=3, dt=1, bn=True)),
    "coupling_D3_H65": ("coupling", dict(D=3, H=65, L=2, dt=2)),
    "coupling_D4_H128_bn": ("coupling", dict(D=4, H=128, L=2, dt=2, bn=True)),
    "coupling_D8_H64_dt4": ("coupling", dict(D=8, H=64, L=2, dt=4)),
    "coupling_refuse_H129": ("coupling", dict(D=2, H=129, L=2, dt=1)),
    "coupling_tc_D1_H8": ("coupling_tc", dict(D=1, H=8, L=2, dt=1)),
    "coupling_tc_D2_H64_bn": ("coupling_tc", dict(D=2, H=64, L=3, dt=1, bn=True)),
    "coupling_tc_D3_H65_bn": ("coupling_tc", dict(D=3, H=65, L=2, dt=2, bn=True)),
    "coupling_tc_D4_H128": ("coupling_tc", dict(D=4, H=128, L=2, dt=2)),
    "coupling_tc_D8_H64_dt4": ("coupling_tc", dict(D=8, H=64, L=2, dt=4)),
    "coupling_tc_refuse_H129": ("coupling_tc", dict(D=2, H=129, L=2, dt=1)),
    "made_tc_D1_H8": ("made_tc", dict(D=1, H=8, L=2)),
    "made_tc_D2_H64_bn": ("made_tc", dict(D=2, H=64, L=3, bn=True)),
    "made_tc_D2_H64_usebn": ("made_tc", dict(D=2, H=64, L=2, use_bn=True)),
    "made_tc_D3_H33_bn_usebn": ("made_tc", dict(D=3, H=33, L=2, bn=True, use_bn=True)),
    "made_tc_D4_H64": ("made_tc", dict(D=4, H=64, L=2)),
    "made_tc_D8_H48_usebn": ("made_tc", dict(D=8, H=48, L=2, use_bn=True)),
    "made_tc_refuse_H65": ("made_tc", dict(D=2, H=65, L=2)),
}


def _pack(name):
    packer, kw = PACK_CASES[name]
    kind = "made" if packer == "made_tc" else packer.replace("_tc", "")
    layers, bns = _model(kind, **kw)
    return PACKERS[packer](layers, bns)


def _digests(pk):
    if pk is None:
        return None
    packed, hdr = pk
    assert hdr.dtype == np.int32 and hdr.shape == (packing.HDR,)
    return (hashlib.sha256(packed.numpy().tobytes()).hexdigest()[:32], hashlib.sha256(hdr.tobytes()).hexdigest()[:32])


# SHA-256 prefixes of (packed, hdr_host); None: the packer refuses the configuration
PACK_DIGESTS = {
    'coupling_D1_H8': ('5b75c568353eb931852251864c12d3c4', 'c05e14a99f7a6c1a49dbcb1efbdb0c79'),
    'coupling_D2_H64_bn': ('2898a33cd9530faf572c85f174385c41', 'cf344f64f111fcff7e54246796e7ecd5'),
    'coupling_D3_H65': ('1ed8179f3182ab0b86220bfbcfb40907', '5df54c14add72bc2fc376916618bcc9a'),
    'coupling_D4_H128_bn': ('fb7e31dcc37747bfa08f6621f5402672', '5e07a21fa461076eb870390fc4da09c7'),
    'coupling_D8_H64_dt4': ('b6dbf50db8a0d070b585c9a3cb7cc8e7', '45ac52a97ad03c5bf1206628dff9f440'),
    'coupling_refuse_H129': None,
    'coupling_tc_D1_H8': ('a5014c97b0b47e3bb051a30dbe3aa0e6', 'c3ef3031d45e5e9fa9c2ad1886267e26'),
    'coupling_tc_D2_H64_bn': ('2812138f2c49f6d35c1b76ab1ee2cff9', 'cf6e5eae402e7ec73fd93f5454f6aab6'),
    'coupling_tc_D3_H65_bn': ('6571d3f95405d69eadd8a33dbb3ea5de', '2a6ac3ad4ccbe9181677316af667acf4'),
    'coupling_tc_D4_H128': ('38b71ab0488794cd6baa8e78b3bf82f3', 'bf9884ebd899565b280d63ad8df9f499'),
    'coupling_tc_D8_H64_dt4': ('44b6971f15803e1652a29aad7bc13458', '40372c8edd9762cf797da16c831ad149'),
    'coupling_tc_refuse_H129': None,
    'made_tc_D1_H8': ('50fb9a91d7eaf85e8e6375c0f8774988', '25db2224f13c85b617afe70ea8664a30'),
    'made_tc_D2_H64_bn': ('f53baced4ab55aabc23400e0b84ba827', 'f43397dcafe3a4b167bd4d73d54e06b7'),
    'made_tc_D2_H64_usebn': ('868b8d68acedf2494e8d4c01da764982', '7a2d3ad9e1fd7dc6622a7d1daea9d2f5'),
    'made_tc_D3_H33_bn_usebn': ('7713179e8953350f5a6af880e2bf39ea', '113cc1e063a63b257c871c2a030063e6'),
    'made_tc_D4_H64': ('68c83a30b434bd90b5f90630d81bc44b', 'eede9f026bdcd236272de17ba38a5b5b'),
    'made_tc_D8_H48_usebn': ('3e2790c3f35203f19cba8170d53326f0', '5881067e329c58d567665754cbcab58d'),
    'made_tc_refuse_H65': None,
    'spline_D1_H8_K2': ('cc64f2323c259cc0eeb5c75ac66f8d17', '5ed1e00e41c5405b4066fa32590006e7'),
    'spline_D2_H64_K8_bn': ('ec269dc61df60fb99551a3713d446551', '41638ae437548ee1c1d3b5fb601cd8ac'),
    'spline_D3_H65_K10_rescale': ('1aa183569ba259f0ee6cf6a645a75eeb', '1dbf3d552f47b4ea0c053972f4e3a8a3'),
    'spline_D4_H128_K16_bn_rescale': ('0bfc60bed04a201eff176fce4f29a0f0', '001daa0f90efc683e255da9f22733e9e'),
    'spline_D8_H128_K8_dt4_rescale': ('894826a0a90d5fb71aa65ea48a1a0696', '165c8028225549702d9ca8f647411d56'),
    'spline_D8_H64_K10_dt4_bn': ('a06b90a534bb45195149e47d261994c7', '47b3de6a62c3b8483aaedc390e61fb38'),
    'spline_refuse_K17': None,
    'spline_tc_D1_H8_K2': ('2ade7824ae15cc6e9e9cf6fe9922ba10', 'e16ed43ad1297151bb1febbb6f9f6e56'),
    'spline_tc_D2_H64_K8_bn': ('d3a83558c91691daa043dda432811133', '991f9aa68fcd9242df5015700f49b3cc'),
    'spline_tc_D3_H33_K10_rescale': ('8b08e2291d57dbcd82930c1aa661ed2c', 'eb7377a75aa4bd4077336d0dfcfc6d2c'),
    'spline_tc_D4_H64_K2_bn_rescale': ('e52b357334c67f8174e283176e6ded45', 'fd08d5ab2e070a37ac79e228dad46021'),
    'spline_tc_D8_H16_K8_dt1': ('1b1f4dd6fbf8781ff4d911f4e3bd78b0', '7e69b43f2ab2ca81fef5da018eb99465'),
    'spline_tc_refuse_H65': None,
}


@pytest.mark.parametrize("name", sorted(PACK_CASES))
def test_packed_bytes_are_pinned(name):
    assert _digests(_pack(name)) == PACK_DIGESTS[name]


# ------------------------------------------------------------------------------------------------
# refusal codes
# ------------------------------------------------------------------------------------------------
P, X, Y, LD = 0x10000, 0x20000, 0x30000, 0x40000      # 16-byte aligned host addresses, never dereferenced
STATE = 0x50000
MAF_INVERSE, IAF_FORWARD, MAF_FORWARD = _lib.AR_MAF_INVERSE, _lib.AR_IAF_FORWARD, _lib.AR_MAF_FORWARD

# family -> (entry-point stem, pack case of a valid header, sampling mode)
FAMILIES = {"spline": ("nf_spline_stack", "spline_D2_H64_K8_bn", None),
            "spline_tc": ("nf_spline_stack_tc", "spline_tc_D2_H64_K8_bn", None),
            "coupling": ("nf_coupling_stack", "coupling_D2_H64_bn", None),
            "coupling_tc": ("nf_coupling_stack_tc", "coupling_tc_D2_H64_bn", None),
            "made_tc": ("nf_made_stack_tc", "made_tc_D2_H64_bn", IAF_FORWARD)}


def _call(fam, entry, hdr, nbytes, packed=P, x=X, y=Y, ld=LD, B=1000, flags=0, mode="default", state=STATE):
    stem, _, sample_mode = FAMILIES[fam]
    if mode == "default":
        mode = sample_mode if entry != "forward" else MAF_INVERSE
    h = None if hdr is None else ctypes.c_void_p(hdr.ctypes.data)
    m = () if sample_mode is None else (mode,)
    fn = getattr(_lib.lib(), f"{stem}_{entry}")
    if entry == "forward":
        return fn(packed, h, nbytes, x, y, ld, B, flags, *m, None)
    if entry == "sample":
        return fn(packed, h, nbytes, *m, 7, 8, y, ld, B, None)
    return fn(packed, h, nbytes, *m, state, y, ld, B, None)


def _header(fam, **over):
    pk = _pack(FAMILIES[fam][1])
    hdr = pk[1].copy()
    for word, v in over.items():
        hdr[int(word[1:])] = v
    return hdr, pk[0].numel() * 4


def _forged_fp32(fam):
    """FP32-pipe header whose layer block needs more than 227 KB of shared memory."""
    hdr, _ = _header(fam)
    hdr[8] = 60000
    return hdr, 4 * (16 + hdr[5] * 60000)


def _wide_spline():
    pk = _model("spline", D=8, H=128, L=2, K=16, dt=4)
    pk = packing.pack_spline_stack(*pk)
    return pk[1].copy(), pk[0].numel() * 4


# case -> function(fam, entry) returning the status; None: the case does not apply to that entry point
def _cases():
    c = {}
    c["hdr_null"] = lambda f, e: _call(f, e, None, *_header(f)[1:])
    c["packed_null"] = lambda f, e: _call(f, e, *_header(f), packed=None)
    c["ld_null"] = lambda f, e: _call(f, e, *_header(f), ld=None)
    c["x_null"] = lambda f, e: _call(f, e, *_header(f), x=None) if e == "forward" else None
    c["y_null"] = lambda f, e: _call(f, e, *_header(f), y=None) if e == "forward" else None
    c["y_null_skip_y"] = lambda f, e: _call(f, e, *_header(f), y=None, flags=6, packed=P + 8) if e == "forward" else None
    c["B_negative"] = lambda f, e: _call(f, e, *_header(f), B=-1)
    c["B_2pow32"] = lambda f, e: _call(f, e, *_header(f), B=1 << 32) if e != "forward" else None
    c["B_2pow32_forward_short"] = lambda f, e: _call(f, e, _header(f)[0], _header(f)[1] - 4, B=1 << 32) \
        if e == "forward" else None
    c["packed_misaligned"] = lambda f, e: _call(f, e, *_header(f), packed=P + 8)
    c["state_misaligned"] = lambda f, e: _call(f, e, *_header(f), state=STATE + 4) if e == "sample_state" else None
    c["state_null"] = lambda f, e: _call(f, e, *_header(f), state=None) if e == "sample_state" else None
    c["wrong_magic"] = lambda f, e: _call(f, e, *_header(f, w0=0x12345678))
    c["bytes_one_word_short"] = lambda f, e: _call(f, e, _header(f)[0], _header(f)[1] - 4)
    c["B0_no_state"] = lambda f, e: _call(f, e, *_header(f), B=0) if e != "sample_state" else None
    c["B0_packed_null"] = lambda f, e: _call(f, e, *_header(f), B=0, packed=None) if e != "sample_state" else None
    # order of the checks
    c["B_negative_hdr_null"] = lambda f, e: _call(f, e, None, 0, B=-1)
    c["hdr_null_B0"] = lambda f, e: _call(f, e, None, 0, B=0)
    c["packed_null_ld_null"] = lambda f, e: _call(f, e, *_header(f), packed=None, ld=None)
    c["misaligned_wrong_magic"] = lambda f, e: _call(f, e, *_header(f, w0=0), packed=P + 4)
    c["wrong_magic_short"] = lambda f, e: _call(f, e, _header(f, w0=0)[0], 0)
    c["state_misaligned_B_negative"] = lambda f, e: _call(f, e, None, 0, B=-1, state=STATE + 4) \
        if e == "sample_state" else None
    # envelopes
    c["D0"] = lambda f, e: _call(f, e, *_header(f, w1=0))
    c["D9"] = lambda f, e: _call(f, e, *_header(f, w1=9))
    c["L0"] = lambda f, e: _call(f, e, *_header(f, w5=0))
    c["K11"] = lambda f, e: _call(f, e, *_header(f, w4=11)) if f == "spline_tc" else None
    c["K17"] = lambda f, e: _call(f, e, *_header(f, w4=17)) if f.startswith("spline") else None
    c["H65"] = lambda f, e: _call(f, e, *_header(f, w2=65)) if f.endswith("_tc") else None
    c["H129"] = lambda f, e: _call(f, e, *_header(f, w2=129)) if f.endswith("_tc") else None
    c["HP96"] = lambda f, e: _call(f, e, *_header(f, w3=96)) if f in ("spline", "coupling") else None
    c["NO_wrong"] = lambda f, e: _call(f, e, *_header(f, w7=10)) if f != "made_tc" else None
    c["stride_unaligned"] = lambda f, e: _call(f, e, *_header(f, w8=_header(f)[0][8] + 2))
    c["W1S_wrong"] = lambda f, e: _call(f, e, *_header(f, w6=12)) if f.endswith("_tc") else None
    c["smem_over_227KB"] = lambda f, e: (_call(f, e, *_wide_spline()) if f == "spline" else
                                         _call(f, e, *_forged_fp32(f)) if f == "coupling" else None)
    c["sequential_mode_D3"] = lambda f, e: _call(f, e, *_header(f, w1=3), mode=MAF_FORWARD) \
        if f == "made_tc" and e == "forward" else None
    c["mode_out_of_range_short"] = lambda f, e: _call(f, e, _header(f)[0], 0, mode=7) if f == "made_tc" else None
    c["density_mode_sample"] = lambda f, e: _call(f, e, None, 0, B=-1, mode=MAF_INVERSE, state=None) \
        if f == "made_tc" and e != "forward" else None
    return c


CASES = _cases()
ENTRIES = ("forward", "sample", "sample_state")
COLUMNS = [(fam, entry) for fam in sorted(FAMILIES) for entry in ENTRIES]


def _statuses(case):
    rcs = [CASES[case](fam, entry) for fam, entry in COLUMNS]
    return " ".join("." if rc is None else str(rc) for rc in rcs)


# case -> status of every entry point, in COLUMNS order ("." where the case does not apply)
REFUSALS = {
    'hdr_null': '-5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5',
    'packed_null': '-5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5',
    'ld_null': '-5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5',
    'x_null': '-5 . . -5 . . -5 . . -5 . . -5 . .',
    'y_null': '-5 . . -5 . . -5 . . -5 . . -5 . .',
    'y_null_skip_y': '-3 . . -3 . . -3 . . -3 . . -3 . .',
    'B_negative': '-1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1',
    'B_2pow32': '. -1 -1 . -1 -1 . -1 -1 . -1 -1 . -1 -1',
    'B_2pow32_forward_short': '-6 . . -6 . . -6 . . -6 . . -6 . .',
    'packed_misaligned': '-3 -3 -3 -3 -3 -3 -3 -3 -3 -3 -3 -3 -3 -3 -3',
    'state_misaligned': '. . -3 . . -3 . . -3 . . -3 . . -3',
    'state_null': '. . -5 . . -5 . . -5 . . -5 . . -5',
    'wrong_magic': '-1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1',
    'bytes_one_word_short': '-6 -6 -6 -6 -6 -6 -6 -6 -6 -6 -6 -6 -6 -6 -6',
    'B0_no_state': '0 0 . 0 0 . 0 0 . 0 0 . 0 0 .',
    'B0_packed_null': '0 0 . 0 0 . 0 0 . 0 0 . 0 0 .',
    'B_negative_hdr_null': '-1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1',
    'hdr_null_B0': '-5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5',
    'packed_null_ld_null': '-5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5 -5',
    'misaligned_wrong_magic': '-3 -3 -3 -3 -3 -3 -3 -3 -3 -3 -3 -3 -3 -3 -3',
    'wrong_magic_short': '-1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1 -1',
    'state_misaligned_B_negative': '. . -3 . . -3 . . -3 . . -3 . . -3',
    'D0': '-1 -1 -1 -2 -2 -2 -2 -2 -2 -1 -1 -1 -2 -2 -2',
    'D9': '-1 -1 -1 -2 -2 -2 -2 -2 -2 -1 -1 -1 -2 -2 -2',
    'L0': '-1 -1 -1 -2 -2 -2 -2 -2 -2 -1 -1 -1 -2 -2 -2',
    'K11': '. . . . . . . . . . . . -2 -2 -2',
    'K17': '. . . . . . . . . -1 -1 -1 -2 -2 -2',
    'H65': '. . . -1 -1 -1 -2 -2 -2 . . . -2 -2 -2',
    'H129': '. . . -2 -2 -2 -2 -2 -2 . . . -2 -2 -2',
    'HP96': '-1 -1 -1 . . . . . . -1 -1 -1 . . .',
    'NO_wrong': '-1 -1 -1 -2 -2 -2 . . . -1 -1 -1 -2 -2 -2',
    'stride_unaligned': '-3 -3 -3 -1 -1 -1 -1 -1 -1 -3 -3 -3 -1 -1 -1',
    'W1S_wrong': '. . . -1 -1 -1 -1 -1 -1 . . . -1 -1 -1',
    'smem_over_227KB': '-2 -2 -2 . . . . . . -2 -2 -2 . . .',
    'sequential_mode_D3': '. . . . . . -2 . . . . . . . .',
    'mode_out_of_range_short': '. . . . . . -2 -2 -2 . . . . . .',
    'density_mode_sample': '. . . . . . . -2 -2 . . . . . .',
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_refusal_codes_are_pinned(case):
    assert _statuses(case) == REFUSALS[case]


def _record():
    """Print both tables (run at the commit whose behaviour is pinned)."""
    print("PACK_DIGESTS = {")
    for name in sorted(PACK_CASES):
        print(f"    {name!r}: {_digests(_pack(name))!r},")
    print("}")
    print("REFUSALS = {")
    for case in CASES:
        print(f"    {case!r}: {_statuses(case)!r},")
    print("}")


if __name__ == "__main__":
    _record()
