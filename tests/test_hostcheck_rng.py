"""CPU: the N(0, I) base stream of sample_and_log_prob (csrc/nf_rng.cuh, compiled for the host from
tests/hostcheck/rng_check.cpp): Philox4x32-10 against published known answers and a pure-Python Philox, the normals
against a float64 Box-Muller of the same 32-bit words, and the row / prefix layout of the stream."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "normalizing-flows-study_b200", "csrc")
SRC = os.path.join(ROOT, "tests", "hostcheck", "rng_check.cpp")
LIB = os.path.join(ROOT, "tests", "hostcheck", "_rng_check.so")

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF
KEY_XOR = 0x6E666232


@pytest.fixture(scope="module")
def hc():
    deps = [SRC, os.path.join(CSRC, "nf_rng.cuh")]
    if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps):
        subprocess.check_call(["g++", "-O1", "-ffp-contract=off", "-shared", "-fPIC", "-x", "c++", "-I", CSRC, SRC,
                               "-o", LIB])
    lib = ctypes.CDLL(LIB)
    lib.hc_philox.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_long]
    lib.hc_box_muller.argtypes = [ctypes.c_void_p] * 2 + [ctypes.c_long]
    lib.hc_std_normal_rows.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_long, ctypes.c_int,
                                       ctypes.c_void_p, ctypes.c_void_p]
    return lib


def py_philox(ctr, key):
    c0, c1, c2, c3 = ctr
    k0, k1 = key
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & MASK, p1 & MASK, ((p0 >> 32) ^ c3 ^ k1) & MASK, p0 & MASK
        k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
    return [c0, c1, c2, c3]


def philox(hc, ctr, key):
    ctr = np.ascontiguousarray(ctr, dtype=np.uint32).reshape(-1, 4)
    key = np.ascontiguousarray(key, dtype=np.uint32).reshape(-1, 2)
    out = np.empty_like(ctr)
    hc.hc_philox(ctr.ctypes.data, key.ctypes.data, out.ctypes.data, len(ctr))
    return out


def unit_f32(u):
    """curand's uniform in fp32 arithmetic: u * 2^-32 + 2^-33."""
    return (u.astype(np.float32) * np.float32(2.0 ** -32) + np.float32(2.0 ** -33)).astype(np.float32)


def box_muller64(ua, ub):
    a, b = unit_f32(ua).astype(np.float64), unit_f32(ub).astype(np.float64)
    r = np.sqrt(-2.0 * np.log(a))
    t = np.pi * (2.0 * b.astype(np.float32)).astype(np.float64)
    return r * np.cos(t), r * np.sin(t)


def ulp_err(z32, z64):
    ref = z64.astype(np.float32)
    ulp = np.spacing(np.abs(ref)).astype(np.float64)
    return np.abs(z32.astype(np.float64) - z64) / np.maximum(ulp, np.spacing(np.float32(1e-30)))


@pytest.mark.parametrize("key,ctr,want", [
    ((0, 0), (0, 0, 0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((MASK, MASK), (MASK, MASK, MASK, MASK), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0xA4093822, 0x299F31D0), (0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(hc, key, ctr, want):
    assert py_philox(ctr, key) == list(want)
    assert philox(hc, ctr, key)[0].tolist() == list(want)


def test_philox_matches_python_on_random_keys(hc):
    rng = np.random.default_rng(7)
    ctr = rng.integers(0, 2 ** 32, size=(500, 4), dtype=np.uint64).astype(np.uint32)
    key = rng.integers(0, 2 ** 32, size=(500, 2), dtype=np.uint64).astype(np.uint32)
    got = philox(hc, ctr, key)
    for i in range(len(ctr)):
        assert got[i].tolist() == py_philox(ctr[i].tolist(), key[i].tolist())


def test_box_muller_within_4_ulp_of_float64(hc):
    rng = np.random.default_rng(11)
    u = rng.integers(0, 2 ** 32, size=(200000, 2), dtype=np.uint64).astype(np.uint32)
    # the extremes of the uniform: a = 2^-33 (largest radius) and a -> 1 (radius 0), angles at the quadrant edges
    edges = np.array([[0, 0], [MASK, MASK], [0, 2 ** 30], [MASK, 2 ** 31], [1, 3 * 2 ** 30], [2 ** 31, 1]], dtype=np.uint32)
    u = np.ascontiguousarray(np.concatenate([u, edges]))
    z = np.empty(u.shape, dtype=np.float32)
    hc.hc_box_muller(u.ctypes.data, z.ctypes.data, len(u))
    z0, z1 = box_muller64(u[:, 0], u[:, 1])
    assert ulp_err(z[:, 0], z0).max() <= 4
    assert ulp_err(z[:, 1], z1).max() <= 4


def rows(hc, seed, offset, B, D):
    z = np.empty((B, D), dtype=np.float32)
    lp = np.empty(B, dtype=np.float32)
    hc.hc_std_normal_rows(seed, offset, B, D, z.ctypes.data, lp.ctypes.data)
    return z, lp


@pytest.mark.parametrize("D", [1, 2, 3, 5, 8])
def test_row_layout_key_and_counter(hc, D):
    seed, offset = 0x0123456789ABCDEF, 4 * 0x1_0000_0003
    z, lp = rows(hc, seed, offset, 37, D)
    key = ((seed & MASK) ^ KEY_XOR, seed >> 32)
    o4 = offset // 4
    for r in (0, 1, 36):
        words = []
        for j in range((D + 3) // 4):
            words += py_philox([j, r, o4 & MASK, o4 >> 32], key)
        w = np.array(words, dtype=np.uint32).reshape(-1, 2)
        c, s = box_muller64(w[:, 0], w[:, 1])
        ref = np.stack([c, s], axis=1).reshape(-1)[:D]
        assert ulp_err(z[r], ref).max() <= 4
        lp64 = -0.5 * (z[r].astype(np.float64) ** 2).sum() - 0.5 * D * np.log(2 * np.pi)
        assert abs(lp[r] - lp64) <= 1e-5 * (1 + abs(lp64))


def test_prefix_offsets_and_seeds(hc):
    z1, _ = rows(hc, 5, 8, 10, 3)
    z2, _ = rows(hc, 5, 8, 100, 3)
    assert np.array_equal(z1, z2[:10])                     # a row does not depend on the row count
    assert not np.array_equal(rows(hc, 5, 12, 10, 3)[0], z1)    # the next offset step is a new stream
    assert not np.array_equal(rows(hc, 6, 8, 10, 3)[0], z1)
    za, _ = rows(hc, 5, 8, 10, 8)
    assert np.array_equal(za[:, :3], z1)                   # dims >= D are discarded, not re-drawn
