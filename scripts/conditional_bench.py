"""Cost of the context in the conditional spline stack, timed on the GPU.

Variants, on the C2 shape 8 x SplineCouplingLayer(2, 64, K=8) with alternating half masks:
  (a) the unconditional model                                             (one launch of spline_stack_tc2_kernel);
  (b) the same model with context_dim 4 and 8                             (one launch of spline_stack_ctx_tc2_kernel);
  (c) the same conditional model in eager PyTorch: the reference's layer with [x*mask, c] concatenated in front of its
      conditioner (tests/conditional_oracle.py on CUDA tensors) -- what a user has without the conditional kernel.
Calls: log_prob(x, context=c) with one context row per row (and, for (b), with one row broadcast to all), and
sample_and_log_prob(n, context=c) with m = 1024 context rows of n = rows / m samples each.  Then one conditional
training step (NLL, backward, Adam) at 65 536 rows, which takes the layered route.
Per variant: median / min / max ms per call over 7 timed regions of CUDA events (warmed up; the L2 cache is overwritten
with a 256 MB buffer before each region, outside the timed window) and the library launch count of one call.  The
variants are alternated within each of 3 rounds, so that a difference can be read against the round-to-round spread.
The card name and power limit are read in the same run.

--model realnvp times the conditional affine stack instead, on the unconditional RealNVP(2, 8, 64) and the published
RealNVP(2, 10, 128), and on the same models with context_dim 4 and 8: (a) unconditional (coupling_stack_tc_kernel),
(b) conditional fused (coupling_stack_ctx_tc_kernel), (c) conditional eager PyTorch (tests/conditional_affine_oracle.py
on CUDA tensors), (d) the conditional model's layered route (flows.USE_TENSOR_CORES = False: no stack kernel), with the
same calls, method and training step (RealNVP(2, 8, 64), context_dim 4).

usage: conditional_bench.py [--model spline|realnvp] [--out FILE.jsonl] [--regions 7] [--rounds 3] [--rows 1048576] [--quick]"""
import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import nfb200 as N
from oracle import flows_oracle as O
from tests import conditional_affine_oracle as CAO
from tests import conditional_oracle as CO

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
ap.add_argument("--regions", type=int, default=7)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--rows", type=int, default=1 << 20)
ap.add_argument("--train-rows", type=int, default=65536)
ap.add_argument("--quick", action="store_true", help="small sizes, one round (a rehearsal of the script)")
ap.add_argument("--model", choices=("spline", "realnvp"), default="spline")
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("conditional_bench.py measures on the GPU: no CUDA device")
DEV = torch.device("cuda:0")
if a.quick:
    a.rows, a.train_rows, a.rounds, a.regions = 8192, 4096, 1, 3
M_CTX = 1024


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def c2(context_dim, seed=1):
    torch.manual_seed(seed)
    masks = [torch.tensor([1., 0.]) if i % 2 == 0 else torch.tensor([0., 1.]) for i in range(8)]
    model = N.NormalizingFlowModel([N.SplineCouplingLayer(2, 64, m, num_bins=8, context_dim=context_dim) for m in masks])
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in model.parameters():
            p.add_(0.05 * torch.randn(p.shape, generator=g))
    return model.to(DEV).eval()


flush_buf = torch.empty(64 << 20, dtype=torch.float32, device=DEV)       # 256 MB > 126 MB of L2


def time_fn(fn, grad=False):
    with torch.set_grad_enabled(grad):
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
    lines = [dict(kind="device", **info, l2="overwritten before each timed region", rows=a.rows)]
    print(json.dumps(lines[0]), flush=True)
    n = a.rows
    g = torch.Generator(device=DEV).manual_seed(0)
    x = 1.5 * torch.randn(n, 2, device=DEV, generator=g)
    specs = [dict(kind="spline", num_bins=8)] * 8
    models = {0: c2(0), 4: c2(4), 8: c2(8)}
    ctx = {C: torch.randn(n, C, device=DEV, generator=g) for C in (4, 8)}
    cs = {C: torch.randn(M_CTX, C, device=DEV, generator=g) for C in (4, 8)}
    sds = {C: {k: v.detach() for k, v in models[C].state_dict().items()} for C in (4, 8)}
    per = n // M_CTX

    def eager_log_prob(C):
        z, ld = CO.flow_model(sds[C], "", specs, x, ctx[C], True)
        return O.std_normal_log_prob(z) + ld

    def eager_sample(C):
        z = torch.randn(M_CTX * per, 2, device=DEV)
        xs, ld = CO.flow_model(sds[C], "", specs, z, cs[C].repeat_interleave(per, 0), False)
        return xs, O.std_normal_log_prob(z) - ld

    variants = [
        ("a_unconditional", "log_prob", lambda: models[0].log_prob(x)),
        ("a_unconditional", "sample_and_log_prob", lambda: models[0].sample_and_log_prob(n)),
    ]
    for C in (4, 8):
        variants += [
            (f"b_fused_C{C}", "log_prob", lambda C=C: models[C].log_prob(x, context=ctx[C])),
            (f"b_fused_C{C}", "sample_and_log_prob", lambda C=C: models[C].sample_and_log_prob(per, context=cs[C])),
            (f"b_fused_C{C}_broadcast", "log_prob", lambda C=C: models[C].log_prob(x, context=ctx[C][:1])),
            (f"c_eager_C{C}", "log_prob", lambda C=C: eager_log_prob(C)),
            (f"c_eager_C{C}", "sample_and_log_prob", lambda C=C: eager_sample(C)),
        ]
    # outputs of the fused route against the eager reference, on the timed inputs (float32 both)
    with torch.no_grad():
        for C in (4, 8):
            lp, lr = models[C].log_prob(x, context=ctx[C]), eager_log_prob(C)
            err = (lp - lr).abs().nan_to_num(0.0).max().item()
            rec = dict(kind="agreement", variant=f"C{C}", call="log_prob", max_abs_diff_vs_eager=err)
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    for rnd in range(a.rounds):
        for variant, call, fn in variants:
            rec = dict(kind="timing", variant=variant, call=call, rows=n, round=rnd, **time_fn(fn), gpu=info["gpu"],
                       nvidia_smi=info["nvidia_smi"])
            lines.append(rec)
            print(json.dumps(rec), flush=True)

    # conditional training step on the layered route
    tm = c2(4, seed=3).train()
    opt = torch.optim.Adam(tm.parameters(), lr=1e-4)
    xt = 1.5 * torch.randn(a.train_rows, 2, device=DEV, generator=g)
    ct = torch.randn(a.train_rows, 4, device=DEV, generator=g)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = -tm.log_prob(xt, context=ct).mean()
        loss.backward()
        opt.step()
        return loss
    rec = dict(kind="timing", variant="train_C4", call="nll+backward+adam", rows=a.train_rows, **time_fn(step, grad=True),
               gpu=info["gpu"], nvidia_smi=info["nvidia_smi"])
    lines.append(rec)
    print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


def realnvp(n_layers, hidden, context_dim, seed=1):
    torch.manual_seed(seed)
    model = N.RealNVP(2, n_layers, hidden, context_dim=context_dim)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in model.parameters():
            p.add_(0.05 * torch.randn(p.shape, generator=g))
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.running_mean.add_(0.1 * torch.randn(m.running_mean.shape, generator=g))
                m.running_var.add_(0.2 * torch.rand(m.running_var.shape, generator=g))
    return model.to(DEV).eval()


def layered(fn):
    """fn() on the layered route: no tcgen05 stack kernel, and no FP32-pipe one for a conditional layer."""
    def run():
        N.flows.USE_TENSOR_CORES = False
        try:
            return fn()
        finally:
            N.flows.USE_TENSOR_CORES = True
    return run


def main_realnvp():
    info = gpu_info()
    lines = [dict(kind="device", **info, l2="overwritten before each timed region", rows=a.rows)]
    print(json.dumps(lines[0]), flush=True)
    n = a.rows
    g = torch.Generator(device=DEV).manual_seed(0)
    x = 1.5 * torch.randn(n, 2, device=DEV, generator=g)
    ctx = {C: torch.randn(n, C, device=DEV, generator=g) for C in (4, 8)}
    cs = {C: torch.randn(M_CTX, C, device=DEV, generator=g) for C in (4, 8)}
    per = n // M_CTX
    variants, agree = [], []
    for L_, H in ((8, 64), (10, 128)):
        shape = f"L{L_}_H{H}"
        specs = [dict(kind="affine")] * L_
        models = {C: realnvp(L_, H, C) for C in (0, 4, 8)}
        sds = {C: {k: v.detach() for k, v in models[C].state_dict().items()} for C in (4, 8)}

        def eager_log_prob(C, sds=sds, specs=specs):
            z, ld = CAO.flow_model(sds[C], "flow.", specs, x, ctx[C], True)
            return O.std_normal_log_prob(z) + ld

        def eager_sample(C, sds=sds, specs=specs):
            z = torch.randn(M_CTX * per, 2, device=DEV)
            xs, ld = CAO.flow_model(sds[C], "flow.", specs, z, cs[C].repeat_interleave(per, 0), False)
            return xs, O.std_normal_log_prob(z) - ld

        m0 = models[0]
        variants += [(f"a_unconditional_{shape}", "log_prob", lambda m0=m0: m0.log_prob(x)),
                     (f"a_unconditional_{shape}", "sample_and_log_prob", lambda m0=m0: m0.sample_and_log_prob(n))]
        for C in (4, 8):
            m = models[C]
            variants += [
                (f"b_fused_{shape}_C{C}", "log_prob", lambda m=m, C=C: m.log_prob(x, context=ctx[C])),
                (f"b_fused_{shape}_C{C}", "sample_and_log_prob", lambda m=m, C=C: m.sample_and_log_prob(per, context=cs[C])),
                (f"c_eager_{shape}_C{C}", "log_prob", lambda C=C, f=eager_log_prob: f(C)),
                (f"c_eager_{shape}_C{C}", "sample_and_log_prob", lambda C=C, f=eager_sample: f(C)),
                (f"d_layered_{shape}_C{C}", "log_prob", layered(lambda m=m, C=C: m.log_prob(x, context=ctx[C]))),
                (f"d_layered_{shape}_C{C}", "sample_and_log_prob",
                 layered(lambda m=m, C=C: m.sample_and_log_prob(per, context=cs[C]))),
            ]
            with torch.no_grad():
                lp, lr = m.log_prob(x, context=ctx[C]), eager_log_prob(C)
                ll = layered(lambda: m.log_prob(x, context=ctx[C]))()
            agree.append(dict(kind="agreement", variant=f"{shape}_C{C}", call="log_prob",
                              max_abs_diff_vs_eager=(lp - lr).abs().nan_to_num(0.0).max().item(),
                              max_abs_diff_vs_layered=(lp - ll).abs().nan_to_num(0.0).max().item()))
    for rec in agree:
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    for rnd in range(a.rounds):
        for variant, call, fn in variants:
            rec = dict(kind="timing", variant=variant, call=call, rows=n, round=rnd, **time_fn(fn), gpu=info["gpu"],
                       nvidia_smi=info["nvidia_smi"])
            lines.append(rec)
            print(json.dumps(rec), flush=True)

    # conditional training step on the layered route (train mode: conditioner BatchNorm on batch statistics)
    tm = realnvp(8, 64, 4, seed=3).train()
    opt = torch.optim.Adam(tm.parameters(), lr=1e-4)
    xt = 1.5 * torch.randn(a.train_rows, 2, device=DEV, generator=g)
    ct = torch.randn(a.train_rows, 4, device=DEV, generator=g)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = -tm.log_prob(xt, context=ct).mean()
        loss.backward()
        opt.step()
        return loss
    rec = dict(kind="timing", variant="train_L8_H64_C4", call="nll+backward+adam", rows=a.train_rows,
               **time_fn(step, grad=True), gpu=info["gpu"], nvidia_smi=info["nvidia_smi"])
    lines.append(rec)
    print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main_realnvp() if a.model == "realnvp" else main()
