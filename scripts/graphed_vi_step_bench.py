"""Reverse-KL (variational) training step and a no-grad sampling call, eager against CUDA-graph replay, on the GPU.

The step draws its own samples with a DeviceGenerator, whose seed and offset live in device memory, so the whole step
-- draw, forward, log-q head, the target's log-density, backward, Adam -- is captured once by graphs.GraphedTrainStep
and every replay draws new samples:

    x, lq = model.sample_and_log_prob(n, generator=g); loss = (lq - target_log_prob(x)).mean()

Adam is fused in both legs (capturable=True only in the graphed one), as in scripts/train_step_bench.py.
target: a fixed 2-D mixture of two unit Gaussians at (-2, 0) and (2, 0), in torch ops.  Models: the reference's four
published configs (plots/_common.py:158-170), in train mode, at n = 4000 and 65 536 rows.  Also timed: a replayed
no-grad model.sample_and_log_prob(4000) against the eager call (eval mode).  Per case: median / min / max ms per step
over --regions timed regions of CUDA events (warmed up), each region >= ~20 ms of work.  The card name and power limit
are read in the same run.

usage: graphed_vi_step_bench.py [--out FILE.jsonl] [--regions 7] [--quick]"""
import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import nfb200 as N  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
ap.add_argument("--regions", type=int, default=7)
ap.add_argument("--quick", action="store_true", help="one config, few steps (a rehearsal of the script, not a measurement)")
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("graphed_vi_step_bench.py measures on the GPU: no CUDA device")
DEV = torch.device("cuda:0")

CONFIGS = {
    "RealNVP(2,10,128)": lambda: N.RealNVP(2, 10, 128),
    "RealNVPSpline(2,8,64)": lambda: N.RealNVPSpline(2, 8, 64),
    "6xMAF(2,64)": lambda: N.NormalizingFlowModel([N.MaskedAutoregressiveFlow(2, 64) for _ in range(6)]),
    "6xIAF(2,64)": lambda: N.NormalizingFlowModel([N.InverseAutoregressiveFlow(2, 64) for _ in range(6)]),
}
MEANS = torch.tensor([[-2.0, 0.0], [2.0, 0.0]], device=DEV)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def target_log_prob(x):
    d = x[:, None, :] - MEANS[None]
    return torch.logsumexp(-0.5 * (d * d).sum(-1) - math.log(2 * math.pi), dim=1) - math.log(2.0)


def time_fn(fn):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    reps = max(1, min(500, math.ceil(20.0 / max(e0.elapsed_time(e1), 1e-3))))
    ms = []
    for _ in range(a.regions):
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1) / reps)
    ms.sort()
    return {"ms_median": ms[len(ms) // 2], "ms_min": ms[0], "ms_max": ms[-1], "reps_per_region": reps}


def vi_step_cases(name, make, n):
    torch.manual_seed(0)
    out = {}
    for mode in ("eager", "graphed"):
        model = make().to(DEV).train()
        # as scripts/train_step_bench.py: fused Adam, capturable only where the step is captured
        opt = torch.optim.Adam(model.parameters(), lr=1e-4, fused=True, capturable=(mode == "graphed"))
        g = N.DeviceGenerator(DEV, seed=1)

        def loss_fn(m, _):
            x, lq = m.sample_and_log_prob(n, generator=g)
            return (lq - target_log_prob(x)).mean()

        if mode == "eager":
            def step():
                opt.zero_grad(set_to_none=True)
                loss = loss_fn(model, None)
                loss.backward()
                opt.step()
                return loss
        else:
            step = N.graphs.GraphedTrainStep(model, opt, loss_fn, torch.empty(1, device=DEV))
        out[mode] = time_fn(step)
    return out


def sample_cases(name, make, n):
    model = make().to(DEV).eval()
    g = N.DeviceGenerator(DEV, seed=2)
    out = {}
    with torch.no_grad():
        out["eager"] = time_fn(lambda: model.sample_and_log_prob(n, generator=g))
        model.sample_and_log_prob(n, generator=g)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            model.sample_and_log_prob(n, generator=g)
        out["graphed"] = time_fn(graph.replay)
    return out


def main():
    info = gpu_info()
    lines = [dict(kind="device", **info)]
    print(json.dumps(lines[0]), flush=True)
    configs = list(CONFIGS.items())[:1] if a.quick else list(CONFIGS.items())
    for name, make in configs:
        for what, fn, sizes in (("reverse_kl_train_step", vi_step_cases, [4000] if a.quick else [4000, 65536]),
                                ("sample_and_log_prob_no_grad", sample_cases, [4000])):
            for n in sizes:
                res = fn(name, make, n)
                for mode, t in res.items():
                    rec = dict(kind="timing", what=what, config=name, n=n, mode=mode, **t, gpu=info["gpu"],
                               nvidia_smi=info["nvidia_smi"])
                    lines.append(rec)
                    print(json.dumps(rec), flush=True)
                rec = dict(kind="speedup", what=what, config=name, n=n,
                           eager_over_graphed=res["eager"]["ms_median"] / res["graphed"]["ms_median"])
                lines.append(rec)
                print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
