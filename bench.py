#!/usr/bin/env python
"""Headline benchmark: log_prob + sample throughput (samples/s, inverse/forward + log-det) of the flow hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl product|reference] [--workload c2|c3] [--no-also]
                    [--dump-outputs DIR]

Workload at every N (weak scaling: fixed rows per GPU, no data-path collective -- rows are independent):
  c2 (default, BASELINE.json configs[1]): 8 SplineCouplingLayers, data_dim=2, hidden 64, 8 RQ-spline bins,
      synthetic checkerboard, 2^20 rows per GPU; one step = one log_prob pass (inverse + log-det + N(0,I) head, ONE
      launch: the head is the last layer's epilogue) + one sample pass (forward + log-det of a N(0,I) batch).
  c3 (configs[2]): MaskedAutoregressiveFlow(64, 512), 262144 rows, log_prob + sequential-direction sampling.  The
      default (c2) run also measures c3 and carries it in the same JSON line under "also" (fp32-parity mode and the
      bf16 fused-chain mode), so that the tensor-pipe half of the path is driver-observed too.
`value` counts rows through either pass (2 x batch per step), inputs resident in HBM; `e2e` is the same step
through the public nn.Module API from pinned HOST buffers with H2D/D2H copies inside the timed region.
One JSON line on stdout (rank 0).  The product arm never touches oracle/ on its measured path; three legs do, as the
checker/baseline only: `cpu_baseline` and `--impl reference` (the unmodified reference staged in oracle/_ref -- kind
"reference" -- or, when that is absent, the oracle port) on the host cores, and `eager_cuda` (the same reference
modules on CUDA tensors: what a user of the reference gets on this GPU today).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "log_prob+sample samples/sec (inverse/forward + log-det)"
UNIT = "samples/s"
WORKLOADS = {
    "c2": dict(name="RealNVPSpline-style stack: 8 x SplineCouplingLayer(2, 64, num_bins=8), checkerboard, 2^20 rows/GPU, "
                    "log_prob + sample",
               rows=1 << 20, D=2, H=64, K=8, L=8),
    "c3": dict(name="MaskedAutoregressiveFlow(64, 512), 8-component Gaussian mixture, 262144 rows/GPU, "
                    "log_prob + sequential-direction sample",
               rows=262144, D=64, H=512),
}
# dense GEMM FLOPs per row of one direction (SURVEY 8d): c2 8 layers x 2*(D*H + H*H + H*D*(3K-1)); c3 one MADE pass
FLOPS_DENSE = {"c2": 8 * 2 * (2 * 64 + 64 * 64 + 64 * 2 * 23), "c3": 2 * (64 * 512 + 2 * 512 * 512 + 512 * 128)}
# executed by the fused kernels: c2 drops the provably-unused half of the last GEMM (SURVEY D9);
# c3 skips the masked-out weight tiles
FLOPS_EXEC = {"c2": 8 * 2 * (2 * 64 + 64 * 64 + 64 * 23), "c3": None}


def config_for(wl):
    """The `config` object: identical for the product and the reference arm (same workload, same rows per step)."""
    cfg = WORKLOADS[wl]
    step_bytes = cfg["rows"] * cfg["D"] * 4 * 2
    ring = max(2, min(32, math.ceil(3 * 126e6 / step_bytes)))
    return {"workload": cfg["name"], "rows_per_gpu": cfg["rows"], "passes_per_step": "log_prob(inverse)+sample(forward)",
            "l2": f"ring of {ring} distinct input sets ({ring * step_bytes / 1e6:.0f} MB) cycled between steps",
            "sharding": "rows sharded across ranks, no data-path collective"}, ring


# ------------------------------------------------------------------------------------------------
# synthetic data + weights (no oracle imports here)
# ------------------------------------------------------------------------------------------------
def checkerboard(n, seed):
    """plots/_common.py:121-128 recipe: uniform(-2,2)^2, keep (floor(x)+floor(y)) even, standardise."""
    rng = np.random.default_rng(seed)
    out = np.empty((0, 2), dtype=np.float32)
    while out.shape[0] < n:
        p = rng.uniform(-2, 2, size=(2 * n, 2))
        keep = (np.floor(p[:, 0]) + np.floor(p[:, 1])) % 2 == 0
        out = np.concatenate([out, p[keep].astype(np.float32)])
    out = out[:n]
    return (out - out.mean(0)) / out.std(0)


def gaussian_mixture(n, D, seed):
    rng = np.random.default_rng(seed)
    means = 3.0 * np.random.default_rng(0).standard_normal((8, D))
    comp = rng.integers(0, 8, size=n)
    return (means[comp] + 0.5 * rng.standard_normal((n, D))).astype(np.float32)


def build_model(wl, N):
    """Reference-layout module with reference init + N(0, sigma^2) perturbation so no layer is the identity.  `N` is
    a namespace with the reference's class names: the product package, or the staged reference itself (the
    constructors draw the same random numbers, tests/test_module_surface.py pins that)."""
    cfg = WORKLOADS[wl]
    torch.manual_seed(0)
    if wl == "c2":
        masks = []
        for i in range(cfg["L"]):
            m = torch.zeros(cfg["D"])
            if i % 2 == 0:
                m[: cfg["D"] // 2] = 1
            else:
                m[cfg["D"] // 2:] = 1
            masks.append(m)
        model = N.NormalizingFlowModel([N.SplineCouplingLayer(cfg["D"], cfg["H"], m, num_bins=cfg["K"]) for m in masks])
        sigma = 0.05
    else:
        model = N.MaskedAutoregressiveFlow(cfg["D"], cfg["H"])
        sigma = 0.02
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for p in model.parameters():
            p.add_(sigma * torch.randn(p.shape, generator=g))
    model.eval()
    return model


def make_inputs(wl, rows, seed):
    cfg = WORKLOADS[wl]
    x = checkerboard(rows, seed) if wl == "c2" else gaussian_mixture(rows, cfg["D"], seed)
    z = np.random.default_rng(seed + 7919).standard_normal((rows, cfg["D"])).astype(np.float32)
    return torch.from_numpy(x), torch.from_numpy(z)


# ------------------------------------------------------------------------------------------------
# clocks, affinity
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        rows = [l for (t, l) in self.lines if t0 - 0.05 <= t <= t1 + 0.15] or [l for (_, l) in self.lines]
        for l in rows:
            f = [c.strip() for c in l.split(",")]
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(f) > col and f[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def bind_to_gpu_numa_node(local):
    """Pin this rank (and the pinned host buffers it allocates afterwards: first touch) to the NUMA node of its GPU.
    Round 1's end-to-end number moved between 1.17 and 1.51 G samples/s from box to box with 8 ranks sharing node 0."""
    try:
        p = torch.cuda.get_device_properties(local)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return {"numa_node": None, "note": "no NUMA affinity reported for the GPU"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as e:          # best effort: containers may hide sysfs
        return {"numa_node": None, "note": f"{type(e).__name__}"}


# ------------------------------------------------------------------------------------------------
# reference legs (the only place bench.py touches oracle/): host cores, and eager on CUDA
# ------------------------------------------------------------------------------------------------
def reference_step_fn(wl, device):
    """(step(x, z), kind): one log_prob + sample step with the UNMODIFIED reference staged in oracle/_ref (kind
    "reference"), else with the oracle port (kind "port": same ATen op sequence).  Modules live on `device`."""
    from oracle import ref_loader
    cfg = WORKLOADS[wl]
    if ref_loader.available():
        R = ref_loader.reference_modules()
        model = build_model(wl, R).to(device).eval()
        D = cfg["D"]
        base = torch.distributions.MultivariateNormal(torch.zeros(D, device=device), torch.eye(D, device=device))

        def step(x, z):
            with torch.no_grad():
                zz, ld = model.inverse(x)
                lp = base.log_prob(zz) + ld               # Flow.log_prob (flow.py:56-73) / plots/_common.py:201-202
                xs, _ = model.forward(z)
            return lp, xs
        return step, "reference"
    from oracle import flows_oracle as O
    import nfb200 as N
    sd = {k: v.detach().clone().to(device) for k, v in build_model(wl, N).state_dict().items()}
    if wl == "c2":
        specs = [dict(kind="spline", num_bins=cfg["K"])] * cfg["L"]

        def step(x, z):
            with torch.no_grad():
                zz, ld = O.flow_model(sd, "", specs, x, True)
                lp = O.std_normal_log_prob(zz) + ld
                xs, _ = O.flow_model(sd, "", specs, z, False)
            return lp, xs
    else:
        def step(x, z):
            with torch.no_grad():
                zz, ld = O.maf_inverse(sd, "", x)
                lp = O.std_normal_log_prob(zz) + ld
                xs, _ = O.maf_forward(sd, "", z)
            return lp, xs
    return step, "port"


def cpu_sample_rows(wl):
    # bounded sample of the workload: ~10-30 s of host work in total
    return 262144 if wl == "c2" else 2048


def time_cpu(wl, sample_rows, reps):
    torch.set_num_threads(os.cpu_count() or 1)
    step, kind = reference_step_fn(wl, "cpu")
    x, z = make_inputs(wl, sample_rows, 123)
    step(x[:1024], z[:1024])
    ts = []
    while len(ts) < reps or (sum(ts) < 10.0 and len(ts) < 40):      # at least `reps` passes and ~10 s of host work
        t = time.perf_counter()
        step(x, z)
        ts.append(time.perf_counter() - t)
    return 2 * sample_rows / (sum(ts) / len(ts)), sum(ts) / len(ts), len(ts), kind


def time_eager_cuda(wl, dev, x, z, reps=3):
    """The reference's modules (eager PyTorch, its stock code path) on CUDA tensors at the workload's full size."""
    try:
        step, kind = reference_step_fn(wl, dev)
        n = x.shape[0]
        if wl == "c3":
            n = 32768          # the reference's sampler re-evaluates MADE 64 times: bounded sample, rows are independent
        xs, zs = x[:n], z[:n]
        step(xs, zs)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            step(xs, zs)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        return {"value": 2 * n / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "rows_per_step": n, "kind": kind,
                "what": "reference nn.Modules, PyTorch eager on this GPU (cuBLAS/ATen kernels), resident inputs"}
    except Exception as e:       # an out-of-memory in the reference's eager path must not kill the product line
        torch.cuda.empty_cache()
        return {"unavailable": f"{type(e).__name__}: {str(e)[:120]}"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload
    rows = WORKLOADS[wl]["rows"] if wl == "c2" else 16384      # c3's reference sampler: 64 MADE passes per step
    torch.set_num_threads(os.cpu_count() or 1)
    step, kind = reference_step_fn(wl, "cpu")
    x, z = make_inputs(wl, rows, 123)
    for _ in range(max(args.warmup, 1)):
        step(x, z)
    t = time.perf_counter()
    for _ in range(args.steps):
        step(x, z)
    dt = (time.perf_counter() - t) / args.steps
    val = 2 * rows / dt
    config, _ = config_for(wl)
    sample = (f"{rows} rows per step" + (" = the full workload" if rows == WORKLOADS[wl]["rows"] else
                                        f" of the {WORKLOADS[wl]['rows']}-row workload") +
              ", log_prob + sample, fp32 PyTorch eager on the host cores, " +
              ("unmodified reference modules (oracle/_ref)" if kind == "reference" else "oracle port"))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------
# product arm
# ------------------------------------------------------------------------------------------------
def load_traffic(wl, precision="fp32"):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed cold-cache
    (`--cache-control all`) ncu capture, read at run time; None when no capture of this round is committed (the file is
    per workload and precision mode: `r02_<workload>_traffic.json` / `r02_<workload>_<mode>_traffic.json`)."""
    path = os.path.join(ROOT, "profiles", f"r02_{wl}_traffic.json" if precision == "fp32" else f"r02_{wl}_{precision}_traffic.json")
    try:
        t = json.load(open(path))
        return float(t["dram_bytes_read"]) + float(t["dram_bytes_write"]), t.get("source")
    except Exception:
        return None, None


def measure(wl, args, N, dev, world, rank, barrier, steps, warmup, precision="fp32", with_clocks=True):
    """Resident + end-to-end timing of one workload in one precision mode; returns a dict of results."""
    import copy
    ops = N.ops
    cfg = WORKLOADS[wl]
    rows, D = cfg["rows"], cfg["D"]
    config, ring = config_for(wl)
    N.set_gemm_precision(precision)
    model = copy.deepcopy(build_model(wl, N)).to(dev).eval()

    host_sets = []
    for i in range(ring):
        x, z = make_inputs(wl, rows, seed=1000 * rank + i)
        host_sets.append((x.pin_memory(), z.pin_memory()))
    dev_sets = [(x.to(dev), z.to(dev)) for x, z in host_sets]

    def step_resident(i, ev=None):
        x, z = dev_sets[i % ring]
        if ev:
            ev[0].record()
        lp = model.log_prob(x)              # standard-normal base: head fused into the last layer where the route allows
        if ev:
            ev[1].record()
        xs, ld2 = model.forward(z)
        if ev:
            ev[2].record()
        return lp, xs, ld2

    # end-to-end arm: the same step through the public modules from pinned HOST buffers.  Three input/output buffer
    # sets and three streams (H2D, compute, D2H) let the copy engines run under the kernels, as a serving loop would;
    # every byte still crosses PCIe inside the timed region.
    NB = 3
    lp_host = [torch.empty(rows, dtype=torch.float32).pin_memory() for _ in range(NB)]
    xs_host = [torch.empty(rows, D, dtype=torch.float32).pin_memory() for _ in range(NB)]
    x_in = [torch.empty(rows, D, dtype=torch.float32, device=dev) for _ in range(NB)]
    z_in = [torch.empty(rows, D, dtype=torch.float32, device=dev) for _ in range(NB)]
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    ev_in = [torch.cuda.Event() for _ in range(NB)]
    ev_done = [torch.cuda.Event() for _ in range(NB)]
    ev_free = [torch.cuda.Event() for _ in range(NB)]
    keep = [None] * NB

    def step_e2e(i):
        b = i % NB
        xh, zh = host_sets[i % ring]
        cur = torch.cuda.current_stream()
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_free[b])                 # the previous user of this buffer set has read it
            x_in[b].copy_(xh, non_blocking=True)
            z_in[b].copy_(zh, non_blocking=True)
            ev_in[b].record(s_in)
        cur.wait_event(ev_in[b])
        lp = model.log_prob(x_in[b])
        xs, _ = model.forward(z_in[b])
        ev_done[b].record(cur)
        lp.record_stream(s_out)
        xs.record_stream(s_out)
        keep[b] = (lp, xs)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_done[b])
            lp_host[b].copy_(lp, non_blocking=True)
            xs_host[b].copy_(xs, non_blocking=True)
            ev_free[b].record(s_out)

    with torch.no_grad():
        for i in range(max(warmup, 3)):
            step_resident(i)
        barrier()
        clocks = ClockSampler(dev.index) if with_clocks else None
        if clocks:
            clocks.start()
            time.sleep(0.3)
        # ---- timed region: exactly K steps ------------------------------------------------------
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
        launches0 = N._lib.launch_count()
        barrier()
        t0 = time.time()
        e_start, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e_start.record()
        # only the last step's outputs are kept (for --dump-outputs): holding every step's outputs into the next step
        # changes what the caching allocator has to map inside the timed window
        for i in range(steps - 1):
            step_resident(i, evs[i])
        last = step_resident(steps - 1, evs[steps - 1])
        e_end.record()
        barrier()
        t1 = time.time()
        launches = N._lib.launch_count() - launches0
        outputs = dict(zip(("log_prob", "sample", "sample_log_det"), (t.float().cpu() for t in last)))
        del last
        ms_total = e_start.elapsed_time(e_end)
        clk = clocks.stop(t0, t1) if clocks else None
        # ---- end-to-end through the public API from pinned host buffers ----------------------
        # warm the copy path as well: a PCIe link that idled trains back up over the first transfers
        for i in range(max(warmup, 3) + 12):
            step_e2e(i)
        # seven timed regions of K steps each; the MEDIAN is reported (all seven are in the line).  Host<->device copies
        # on a shared box see transients the kernels do not: one r02 run measured 0.33 G samples/s end to end between
        # two runs at 1.44 and 1.66 G on the same box, with nvidia-smi unresponsive during that window; another had
        # regions of 1.12 / 4.78 / 1.76 ms per step back to back (a median of three does not survive two bad regions).
        e2e_runs = []
        for _ in range(7):
            barrier()
            s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s2.record()
            for i in range(steps):
                step_e2e(i)
            torch.cuda.current_stream().wait_stream(s_out)      # the last device->host copies close the timed region
            e2.record()
            barrier()
            e2e_runs.append(s2.elapsed_time(e2))
        ms_e2e = sorted(e2e_runs)[len(e2e_runs) // 2]

    t = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = t.tolist()
    ms_step = ms_total / steps
    ms_lp = float(np.mean([e[0].elapsed_time(e[1]) for e in evs]))
    ms_fwd = float(np.mean([e[1].elapsed_time(e[2]) for e in evs]))
    res = {
        "value": 2.0 * rows * world / (ms_step * 1e-3), "ms_per_step": ms_step,
        "e2e": {"value": 2.0 * rows * world / (ms_e2e / steps * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": 2 * rows * D * 4, "d2h_bytes_per_step": rows * 4 + rows * D * 4,
                "ms_per_step_runs": [t / steps for t in e2e_runs], "reported": "median of 7 regions of K steps (this rank)"},
        "gpu_launches": int(launches), "ms_log_prob": ms_lp, "ms_sample": ms_fwd, "clocks": clk, "config": config,
        "precision": precision, "dev_sets": dev_sets, "outputs": outputs,
    }
    N.set_gemm_precision("fp32")
    return res


DUMP_ARRAY_BYTES = 8 << 20


def dump_outputs(out_dir, prefix, outputs):
    """Write the outputs of the last timed step as <out_dir>/<prefix>_<name>.npy (float32).  An array larger than 8 MB
    keeps a fixed, seeded sample of its rows (the same rows in every run), so a default run writes at most 36 MB."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        if t.numel() * t.element_size() > DUMP_ARRAY_BYTES:
            keep = DUMP_ARRAY_BYTES // (t[0].numel() * t.element_size())
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t[rows]
        np.save(os.path.join(out_dir, f"{prefix}_{name}.npy"), t.numpy())


def roofline_for(wl, r, precision):
    cfg = WORKLOADS[wl]
    rows, D = cfg["rows"], cfg["D"]
    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
    peak_tf = peaks.get("bf16_tflops", 1590.0)
    which = "measured (MEASURED_PEAKS.json bf16 burst)" if peaks else "fallback 1.59 PFLOP/s"
    ms_dom = 0.5 * (r["ms_log_prob"] + r["ms_sample"]) if wl == "c2" else r["ms_log_prob"]
    achieved = FLOPS_DENSE[wl] * rows / (ms_dom * 1e-3) / 1e12
    traffic, traffic_src = load_traffic(wl, precision)
    if wl == "c2":
        kernel = ("spline_stack_tc2_kernel: one launch = all 8 layers of one direction (+ the N(0,I) log-prob head in the "
                  "log_prob pass); layer-2 and head GEMMs on tcgen05 (3xTF32, A operand in TMEM), layer 1 + spline on the "
                  "FP32 pipe")
        note = ("GEMM FLOPs on the dense accounting of SURVEY 8d (what the reference's F.linear calls execute); the kernel "
                "skips the unused half of the head (D9) and runs the remaining GEMM FLOPs 3x on the tensor pipe for fp32 "
                "parity (tensor_flops_per_row_executed); it is bound by the per-row spline / split work on the FP32 pipe, "
                "not by the tensor pipe or HBM (20 B per row)")
        tensor_exec = 8 * 3 * 2 * (64 * 64 + 64 * 32)
    elif precision == "bf16":
        kernel = ("made_chain_bf16_kernel: ONE persistent launch per MAF.inverse -- x -> bf16, four masked linears as "
                  "tcgen05 kind::f16 MMAs (weights streamed by TMA, activations never leave the SM: TMEM -> registers -> "
                  "bias/ReLU -> bf16 -> shared-memory A operand of the next layer), affine-AR transform + log-det (+ "
                  "N(0,I) head) in the last epilogue")
        note = ("dense GEMM FLOPs of one MADE evaluation (SURVEY 8d) over the time of the whole MAF.inverse launch; "
                "masked-out K tiles are skipped; bf16 operands, fp32 accumulation (documented bounds: DESIGN.md)")
        tensor_exec = None
    else:
        kernel = ("gemm_tc2_kernel x4 (persistent, tcgen05 3xTF32, TMA-fed, masked-out K tiles skipped; K > 128: chains of "
                  "24 MMAs folded into registers with round-to-nearest adds; K = 64 input layer: direct variant) + "
                  "affine_ar_fwd_kernel + std_normal_log_prob")
        note = ("dense GEMM FLOPs of one MADE evaluation (SURVEY 8d) over the time of the whole MAF.inverse chain; the "
                "tensor pipe executes 3x the unskipped FLOPs (3xTF32 keeps fp32 parity)")
        tensor_exec = None
    return {
        "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
        "traffic": traffic, "traffic_source": traffic_src, "kernel": kernel,
        "flops_per_row": FLOPS_DENSE[wl], "flops_per_row_executed": FLOPS_EXEC[wl],
        "tensor_flops_per_row_executed": tensor_exec, "peak_source": which,
        "ms_per_launch": {"log_prob": r["ms_log_prob"], "sample": r["ms_sample"]},
        "hbm_gbs_algorithmic": (rows * (2 * D + 1) * 4) / (ms_dom * 1e-3) / 1e9,
        "note": note,
    }


def run_product(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (product arm) needs a CUDA device: libnfb200 has no CPU path")
    torch.cuda.set_device(local)
    affinity = bind_to_gpu_numa_node(local)
    import nfb200 as N
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    wl = args.workload
    steps, warmup = args.steps, max(args.warmup, 3)
    r = measure(wl, args, N, dev, world, rank, barrier, steps, warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, wl, r["outputs"])
    out = {
        "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": r["config"], "clocks": r["clocks"], "e2e": r["e2e"],
        "gpu_launches": r["gpu_launches"], "roofline": roofline_for(wl, r, "fp32"), "host_affinity": affinity,
    }
    if rank == 0 and world == 1 and not args.no_cpu:
        x, z = r["dev_sets"][0]
        out["eager_cuda"] = time_eager_cuda(wl, dev, x, z)
    del r
    torch.cuda.empty_cache()

    # the other log_prob+sample config of BASELINE.json (the tensor-pipe one) in the same line
    if wl == "c2" and not args.no_also:
        also = {}
        modes = ["fp32"] + (["bf16"] if "bf16" in getattr(N, "GEMM_PRECISIONS", ()) and not os.environ.get("NF_SKIP_BF16") else [])
        for mode in modes:
            try:
                a = measure("c3", args, N, dev, world, rank, barrier, steps, 3, precision=mode, with_clocks=False)
            except Exception as e:
                also["c3_" + mode] = {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}
                continue
            if args.dump_outputs and rank == 0:
                dump_outputs(args.dump_outputs, "c3" if mode == "fp32" else "c3_" + mode, a["outputs"])
            blk = {"workload": WORKLOADS["c3"]["name"], "gemm_precision": mode, "value": a["value"], "unit": UNIT,
                   "steps": steps, "ms_per_step": a["ms_per_step"], "e2e": a["e2e"], "gpu_launches": a["gpu_launches"],
                   "ms_per_launch": {"log_prob": a["ms_log_prob"], "sample": a["ms_sample"]},
                   "roofline": roofline_for("c3", a, mode)}
            if mode == "fp32" and rank == 0 and world == 1 and not args.no_cpu:
                x, z = a["dev_sets"][0]
                blk["eager_cuda"] = time_eager_cuda("c3", dev, x, z, reps=1)
            also["c3" if mode == "fp32" else "c3_" + mode] = blk
            del a
            torch.cuda.empty_cache()
        out["also"] = also

    if rank == 0 and world == 1 and not args.no_cpu:
        n = cpu_sample_rows(wl)
        v, secs, nrep, kind = time_cpu(wl, n, reps=3)
        out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                               "sample": f"{n} rows of the workload, log_prob + sample, {nrep} x {secs:.2f} s per pass pair, "
                                         + ("unmodified reference modules (oracle/_ref)" if kind == "reference" else
                                            "oracle port (fp32 ATen eager, same op sequence as the reference)")}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="product", choices=["product", "reference"])
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline and eager_cuda legs")
    ap.add_argument("--no-also", action="store_true", help="skip the c3 block of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the log_prob, sample and sample log-det of the last timed step of each product "
                         "workload as DIR/<workload>[_<mode>]_<name>.npy, float32")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1 and args.gpus > 1 and args.impl == "product":
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_product(args)


if __name__ == "__main__":
    main()
