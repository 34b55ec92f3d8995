"""C3 sequential direction (MaskedAutoregressiveFlow(64, 512).forward, 262144 rows): timing of the blocked route and a
fixed target for ncu (--reps 1: three forward passes, nothing else).  usage: sampler_target.py [--reps N] [--rows B]"""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import nfb200 as N

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--rows", type=int, default=262144)
ap.add_argument("--precision", default="fp32")
a = ap.parse_args()
torch.manual_seed(0)
N.set_gemm_precision(a.precision)
m = N.MaskedAutoregressiveFlow(64, 512).cuda().eval()
with torch.no_grad():
    for p in m.parameters():
        p.add_(0.02 * torch.randn_like(p))
    z = torch.randn(a.rows, 64, device="cuda")
    for _ in range(2):
        x, ld = m.forward(z)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    before = N._lib.launch_count()
    e0.record()
    for _ in range(a.reps):
        x, ld = m.forward(z)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.reps
    zz, ld2 = m.inverse(x)
    print(json.dumps({"what": "MAF(64,512).forward", "rows": a.rows, "precision": a.precision, "ms": ms,
                      "launches_per_pass": (N._lib.launch_count() - before) / a.reps,
                      "roundtrip_max_abs": float((zz - z).abs().max()), "ld_sum_abs": float((ld + ld2).abs().max())}))
