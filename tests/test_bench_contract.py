"""Host-side pieces of bench.py that need no GPU: the roofline block of the JSON line (algorithmic FLOPs over the measured
launch time against the measured peak, traffic read from the committed cold-cache capture of the same precision mode),
the bounded CPU sample sizes and the writer of --dump-outputs."""
import importlib.util
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    argv = sys.argv
    sys.argv = ["bench.py"]
    try:
        spec = importlib.util.spec_from_file_location("nfb200_bench_under_test", os.path.join(ROOT, "bench.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.argv = argv
    return mod


def test_roofline_block_uses_the_capture_of_its_own_precision_mode():
    b = _bench()
    r = {"ms_log_prob": 1.25, "ms_sample": 3.7}
    fp32 = b.roofline_for("c3", r, "fp32")
    bf16 = b.roofline_for("c3", {"ms_log_prob": 0.26, "ms_sample": 3.6}, "bf16")
    rows = b.WORKLOADS["c3"]["rows"]
    # achieved = dense FLOPs of one MADE evaluation per row x rows / the log_prob pass
    assert abs(fp32["achieved"] - b.FLOPS_DENSE["c3"] * rows / 1.25e-3 / 1e12) < 1e-6
    assert fp32["bound"] == "tensor" and abs(fp32["frac"] - fp32["achieved"] / fp32["peak"]) < 1e-12
    # the fp32 chain's cold-cache traffic is committed; it must not leak into the bf16 block (another kernel)
    assert fp32["traffic"] == b.load_traffic("c3")[0] and fp32["traffic"] > rows * 516
    assert bf16["traffic"] == b.load_traffic("c3", "bf16")[0]
    assert not os.path.exists(os.path.join(ROOT, "profiles", "r02_c3_bf16_traffic.json")) or bf16["traffic"] is not None
    c2 = b.roofline_for("c2", {"ms_log_prob": 0.56, "ms_sample": 0.55}, "fp32")
    assert c2["traffic"] == b.load_traffic("c2")[0] and c2["unit"] == "TFLOP/s"


def test_cpu_sample_is_bounded():
    b = _bench()
    for wl in b.WORKLOADS:
        assert 0 < b.cpu_sample_rows(wl) <= b.WORKLOADS[wl]["rows"]


def test_dump_outputs_writes_whole_small_arrays_and_a_fixed_sample_of_large_ones(tmp_path):
    b = _bench()
    rows, D = b.WORKLOADS["c3"]["rows"], b.WORKLOADS["c3"]["D"]
    g = torch.Generator().manual_seed(3)
    sample = torch.randn(rows, D, generator=g)
    sample[:, 0] = torch.arange(rows)                   # each row carries its index
    outputs = {"log_prob": torch.randn(rows, generator=g), "sample": sample}
    for d in ("a", "b"):
        b.dump_outputs(str(tmp_path / d), "c3", outputs)
    lp = np.load(tmp_path / "a" / "c3_log_prob.npy")
    assert lp.dtype == np.float32 and np.array_equal(lp, outputs["log_prob"].numpy())
    xs = np.load(tmp_path / "a" / "c3_sample.npy")
    assert xs.dtype == np.float32 and xs.nbytes == b.DUMP_ARRAY_BYTES and xs.shape[1] == D
    assert np.array_equal(xs, np.load(tmp_path / "b" / "c3_sample.npy"))
    # the sample is whole rows of the output, in order
    src = xs[:, 0].astype(np.int64)
    assert np.all(np.diff(src) > 0) and np.array_equal(xs, sample.numpy()[src])
