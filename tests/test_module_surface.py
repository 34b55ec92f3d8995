"""CPU: the drop-in nn.Module surface (names, constructor arguments, state_dict layout, shims) and the
C-ABI library's exported symbols.  No kernel is launched here."""
import ctypes
import os
import re

import pytest
import torch

import nfb200 as N
from tests import golden_util as G
from tests.build_util import MODULE_KINDS, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "nfb200.h")).read()
    declared = set(re.findall(r"NF_API\s+[\w\s\*]+?\b(nf_\w+)\s*\(", hdr))
    assert len(declared) >= 30
    lib = ctypes.CDLL(N._lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/nfb200.h but not exported"
    assert declared == set(N._lib.EXPORTED_SYMBOLS), declared ^ set(N._lib.EXPORTED_SYMBOLS)
    assert N._lib.lib().nf_abi_version() == 1
    assert N._lib.lib().nf_status_string(-2).decode().startswith("unsupported")


@pytest.mark.parametrize("name", [n for n in G.golden_names() if G.load(n)["kind"] in MODULE_KINDS])
def test_reference_state_dict_loads_strictly(name):
    g = G.load(name)
    m = build(g)                      # load_state_dict(strict=True) inside
    ours = {k: (tuple(v.shape), v.dtype) for k, v in m.state_dict().items()}
    ref = {k: (tuple(v.shape), v.dtype) for k, v in g["sd"].items()}
    assert ours == ref
    assert list(m.state_dict().keys()) == list(g["sd"].keys())


def test_made_masks_match_reference():
    for name in G.golden_names("maf_") + G.golden_names("iaf_"):
        g = G.load(name)
        made = N.MADE(g["D"], g["H"])
        assert torch.equal(torch.as_tensor(made.m[0]), g["degrees"])
        for idx in (0, 2, 4, 6):
            assert torch.equal(made.net[idx].mask, g["sd"][f"conditioner.net.{idx}.mask"])


def test_initialisation_draws_match_reference():
    """Same seed => same initial weights as the reference constructors (tests/golden/init_parity.pt)."""
    g = G.load("init_parity")
    ctors = {
        "coupling": lambda: N.CouplingLayer(4, 16, torch.tensor([1., 0., 1., 0.])),
        "spline": lambda: N.SplineCouplingLayer(4, 16, torch.tensor([1., 1., 0., 0.]), num_bins=6),
        "maf": lambda: N.MaskedAutoregressiveFlow(5, 32),
        "iaf": lambda: N.InverseAutoregressiveFlow(5, 32),
        "made_bn": lambda: N.MADE(3, 8, 2, use_batch_norm=True),
        "realnvp_bn": lambda: N.RealNVP(4, 4, 16, batch_norm_between_layers=True),
        "realnvpspline": lambda: N.RealNVPSpline(6, 2, 32),
    }
    for key, ctor in ctors.items():
        torch.manual_seed(g["seed"])
        sd = ctor().state_dict()
        assert list(sd.keys()) == list(g[key].keys()), key
        for k, v in g[key].items():
            assert torch.equal(sd[k], v), f"{key}.{k}"


def test_constructor_contracts():
    with pytest.raises(AssertionError):
        N.RealNVP(2, 3, 8)
    with pytest.raises(AssertionError):
        N.RealNVPSpline(2, 3, 8)
    with pytest.raises(ValueError):
        N.SequentialFlow(tuple())
    with pytest.raises(ValueError):
        N.NormalizingFlowModel([torch.nn.Identity()], batch_norm_between_layers=True)
    m = N.RealNVP(6, 4, 8)
    masks = [f.mask.tolist() for f in m.flow.flows]
    assert masks[0] == [1, 1, 1, 0, 0, 0] and masks[1] == [0, 0, 0, 1, 1, 1] and masks[2] == masks[0]
    s = N.SplineCouplingLayer(4, 8, torch.tensor([1., 0., 1., 0.]))
    assert (s.num_bins, s.bound, s.data_dim) == (10, 5.0, 4)
    assert s.param_net[-1].out_features == 4 * 29
    f = N.MaskedAutoregressiveFlow(3)
    assert (f.dim, f.data_dim, f.conditioner.hidden_dim) == (3, 3, 64)
    assert isinstance(f.conditioner.net[-1], N.MaskedLinear)
    with pytest.raises(NotImplementedError):
        N.Flow().forward(torch.zeros(1, 1))


def test_src_shims_resolve_to_product():
    import src.flows as SF
    import src.models as SM
    assert SF.CouplingLayer is N.CouplingLayer and SM.RealNVP is N.RealNVP
    assert SF.rational_quadratic_spline is N.rational_quadratic_spline


def test_no_cpu_route():
    layer = N.CouplingLayer(2, 8, torch.tensor([1., 0.]))
    with pytest.raises(RuntimeError, match="no CPU path"):
        layer.forward(torch.zeros(4, 2))


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "normalizing-flows-study_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src.replace("flows_oracle", "oracle") or fn == "build.py" or "import oracle" not in src
            assert "import oracle" not in src and "from oracle" not in src


def test_library_options_from_the_environment():
    """NFB200_OPTIONS="key:value,..." (the A/B knob of the measurement scripts) is applied through nf_set_option when the
    library is loaded; a refused value fails the load loudly.  Only keys 7, 10 and 11 exist: the keys of the retired
    kernel variants (1, 2, 3, 5, 6, 9) are refused, so a script that still sets one fails instead of measuring the default."""
    import subprocess, sys
    code = "import nfb200; l = nfb200._lib.lib(); print(l.nf_set_option(11, 1), l.nf_set_option(7, 2))"
    env = dict(os.environ, NFB200_OPTIONS="11:0,7:3")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT)
    out = r.stdout.split()
    assert r.returncode == 0 and out[0] == "0" and out[1] != "0", r.stderr[-400:]
    for key in (1, 2, 3, 5, 6, 9):
        for value in (0, 1, 2, 3, 64):
            assert N._lib.lib().nf_set_option(key, value) != 0, (key, value)
    for opts in ("7:2", "3:3"):
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=dict(os.environ, NFB200_OPTIONS=opts), cwd=ROOT)
        assert r.returncode != 0 and "refused" in r.stderr, opts


def test_gemm_precision_switch_is_host_only_and_validated():
    """set_gemm_precision maps onto nf_set_option(7, passes); no device is needed to flip it, unknown modes and pass
    counts are rejected, and the default is the fp32-parity mode."""
    assert N.get_gemm_precision() == "fp32"
    try:
        N.set_gemm_precision("tf32")
        assert N.get_gemm_precision() == "tf32"
    finally:
        N.set_gemm_precision("fp32")
    assert N.get_gemm_precision() == "fp32"
    try:
        N.set_gemm_precision("bf16")                      # round 2: the fused bf16 MADE-chain mode
        assert N.get_gemm_precision() == "bf16" and N.ops.MADE_CHAIN_BF16
    finally:
        N.set_gemm_precision("fp32")
    assert not N.ops.MADE_CHAIN_BF16
    with pytest.raises(ValueError):
        N.set_gemm_precision("fp8")
    assert N._lib.lib().nf_set_option(7, 2) != 0          # only 1 and 3 passes exist
    assert N._lib.lib().nf_set_option(7, 3) == 0
    assert N._lib.lib().nf_set_option(99, 0) != 0         # unknown key


@pytest.mark.parametrize("D,H,gb", [(64, 512, 8), (16, 128, 8), (12, 100, 4), (784, 1024, 8), (8, 16, 8)])
def test_blocked_sampler_layout_pads_blocks_to_aligned_starts(D, H, gb):
    """packing.blocked_layout (host logic of the blocked sequential direction, csrc/ar_blocked.cu): every block of `gb`
    degrees starts at a multiple of 4 units (8 in the per-degree layout), the sorted order of the live units is kept, the
    dead units sit behind the live units of their degree, and the padded boundaries delimit exactly the live units of each
    degree plus its dead ones."""
    import numpy as np
    from nfb200 import packing
    deg = np.sort(np.arange(H) % (D - 1) + 1)                      # made.py:31-33 hidden degrees, sorted
    gstart = np.searchsorted(deg, np.arange(D + 1), side="left").astype(np.int32)
    pos, pg, Hp = packing.blocked_layout(gstart, gb)
    assert Hp % 4 == 0 and pg[D] == Hp and len(pos) == H
    assert np.all(np.diff(pos) > 0) and pos[-1] < Hp
    assert Hp <= 1.10 * H + 4 * ((D + gb - 1) // gb)              # per-degree padding only when it is cheap
    for g in range(D):
        n = gstart[g + 1] - gstart[g]
        assert np.array_equal(pos[gstart[g]:gstart[g + 1]], pg[g] + np.arange(n))
        assert 0 <= pg[g + 1] - pg[g] - n < 8                     # dead units behind the degree's live ones
        if g % gb == 0:
            assert pg[g] % 4 == 0
    # per-degree layout (every degree 4-aligned): blocks are padded to multiples of 8 units, so no slice GEMM of the route
    # contracts over K = 4 (mod 32) and every output slice is 32-byte aligned
    if all(pg[g] % 4 == 0 for g in range(D)):
        assert all(pg[g] % 8 == 0 for g in range(0, D, gb)) and Hp % 8 == 0
