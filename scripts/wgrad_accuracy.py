"""Error of the tcgen05 weight gradient (TMEM accumulation chains of at most 64 K blocks) vs float64, beside cuBLAS fp32
and the FP32-pipe GEMM."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import nfb200 as N
torch.backends.cuda.matmul.allow_tf32 = False
def t(fn, n=5):
    for _ in range(2): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n
for B, Nn, K in [(262144, 512, 512), (65536, 1024, 1024), (4096, 2844, 1024)]:
    for kind in ("randn", "positive"):
        gen = torch.Generator(device="cuda").manual_seed(1)
        g = torch.randn(B, Nn, device="cuda", generator=gen); x = torch.randn(B, K, device="cuda", generator=gen)
        if kind == "positive":
            g, x = g.abs(), x.abs()
        ref = (g.double().T @ x.double())
        rms = ref.pow(2).mean().sqrt()
        def report(name, d, ms=None):
            e = (d.double() - ref)
            print(f"  {name:28s} max|err|/rms {e.abs().max().item() / rms.item():.2e}   mean err/rms {e.mean().item() / rms.item():+.2e}   rms err/rms {e.pow(2).mean().sqrt().item() / rms.item():.2e}" + (f"   {ms:.3f} ms" if ms else ""), flush=True)
        print(f"B={B} N={Nn} K={K} {kind}: rms(dW)={rms.item():.3g}")
        report("torch fp32 (cuBLAS, no tf32)", g.T @ x)
        report("FP32-pipe nf_gemm", N.ops.gemm(g, x, Nn, K, B, 1, Nn, K, 1))
        ms = t(lambda: N.ops.linear_wgrad_tc(g, x))
        report("tcgen05 nf_linear_wgrad_tc", N.ops.linear_wgrad_tc(g, x), ms)
