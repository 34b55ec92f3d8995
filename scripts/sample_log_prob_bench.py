"""Three ways to get samples and their log-density (x, log_q) from a flow, timed on the GPU:
  (a) model.sample_and_log_prob(n)                                   N(0, I) drawn on the device, fused where possible;
  (b) z = torch.randn; x, ld = model(z); base.log_prob(z).sum(1) - ld     the torch composition;
  (c) x = model.sample(n); model.log_prob(x)                           both directions;
  (d) model.sample_and_log_prob(n, generator=nfb200.DeviceGenerator())  (a) with the key read from and advanced in
                                                                         device memory (the CUDA-graph-safe draw).
(d) is timed in rounds alternated with (a) ("round" field), so that the difference can be read against the run-to-run
spread of (a) itself.
Per way: median / min / max ms per call over 7 timed regions of CUDA events (warmed up; the L2 cache is overwritten with
a 256 MB buffer before each region, outside the timed window, since the outputs of a 2^20-row call fit in L2) and the
library launch count of one call.  The card name and power limit are read in the same run.

usage: sample_log_prob_bench.py [--out FILE.jsonl] [--regions 7] [--rounds 3] [--quick]"""
import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from torch import distributions as td

import nfb200 as N

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
ap.add_argument("--regions", type=int, default=7)
ap.add_argument("--rounds", type=int, default=3, help="alternated (a) / (d) rounds per configuration")
ap.add_argument("--quick", action="store_true", help="small sizes only (a rehearsal of the script, not a measurement)")
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("sample_log_prob_bench.py measures on the GPU: no CUDA device")
DEV = torch.device("cuda:0")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def perturbed(m, sigma, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in m.parameters():
            p.add_(sigma * torch.randn(p.shape, generator=g))
    return m.to(DEV).eval()


def spline_c2():
    masks = [torch.tensor([1., 0.]) if i % 2 == 0 else torch.tensor([0., 1.]) for i in range(8)]
    return N.NormalizingFlowModel([N.SplineCouplingLayer(2, 64, m, num_bins=8) for m in masks])


CONFIGS = [       # name, factory, D, rows, gemm precision
    ("RealNVPSpline-C2 8x spline(2,64,K=8)", spline_c2, 2, 1 << 20, "fp32"),
    ("RealNVP(2,10,128)", lambda: N.RealNVP(2, 10, 128), 2, 1 << 20, "fp32"),
    ("6xIAF(2,64)", lambda: N.NormalizingFlowModel([N.InverseAutoregressiveFlow(2, 64) for _ in range(6)]), 2, 1 << 20, "fp32"),
    ("6xMAF(2,64)", lambda: N.NormalizingFlowModel([N.MaskedAutoregressiveFlow(2, 64) for _ in range(6)]), 2, 1 << 20, "fp32"),
    ("IAF(64,512)", lambda: N.InverseAutoregressiveFlow(64, 512), 64, 262144, "fp32"),
    ("IAF(64,512)", lambda: N.InverseAutoregressiveFlow(64, 512), 64, 262144, "bf16"),
    ("MAF(64,512)", lambda: N.MaskedAutoregressiveFlow(64, 512), 64, 262144, "fp32"),
]

flush_buf = torch.empty(64 << 20, dtype=torch.float32, device=DEV)       # 256 MB > 126 MB of L2


def time_way(fn):
    with torch.no_grad():
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        c0 = N._lib.launch_count()
        fn()
        torch.cuda.synchronize()
        launches = N._lib.launch_count() - c0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        reps = max(1, min(200, math.ceil(10.0 / max(e0.elapsed_time(e1), 1e-3))))      # >= ~10 ms per region
        ms = []
        for _ in range(a.regions):
            flush_buf.fill_(1.0)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1) / reps)
    ms.sort()
    return {"ms_median": ms[len(ms) // 2], "ms_min": ms[0], "ms_max": ms[-1], "reps_per_region": reps,
            "library_launches": launches}


def main():
    info = gpu_info()
    lines = [dict(kind="device", **info, l2="overwritten before each timed region")]
    print(json.dumps(lines[0]), flush=True)
    for name, make, D, rows, prec in CONFIGS:
        N.set_gemm_precision(prec)
        model = perturbed(make(), 0.02 if D == 64 else 0.05, 1)
        base = td.Normal(torch.zeros(D, device=DEV), torch.ones(D, device=DEV))
        for n in ([4000] if a.quick else [rows, 4000]):
            if a.quick and D == 64:
                n = 2048

            def way_a():
                return model.sample_and_log_prob(n)

            def way_b():
                z = torch.randn(n, D, device=DEV)
                x, ld = model(z)
                return x, base.log_prob(z).sum(1) - ld

            def way_c():
                x = model.sample(n, device=DEV)
                return x, model.log_prob(x)

            gen = N.DeviceGenerator(DEV)

            def way_d():
                return model.sample_and_log_prob(n, generator=gen)

            timed = [(None, "a", way_a), (None, "b", way_b), (None, "c", way_c)]
            timed += [(r, w, f) for r in range(a.rounds) for w, f in (("a", way_a), ("d", way_d))]
            for rnd, way, fn in timed:
                rec = dict(kind="timing", config=name, precision=prec, n=n, way=way, **time_way(fn),
                           gpu=info["gpu"], nvidia_smi=info["nvidia_smi"])
                if rnd is not None:
                    rec["round"] = rnd
                lines.append(rec)
                print(json.dumps(rec), flush=True)
    N.set_gemm_precision("fp32")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
