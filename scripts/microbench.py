#!/usr/bin/env python
"""Per-kernel roofline microbenchmark (B200): times every stand-alone kernel of libnfb200 with CUDA events on
inputs larger than L2 and prints achieved GB/s (algorithmic bytes) or TFLOP/s against MEASURED_PEAKS.json.

    python scripts/microbench.py [--only rqs,spline_tf,...] [--json gpurun_out/microbench.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import nfb200 as N  # noqa: E402

ops = N.ops
DEV = torch.device("cuda:0")
PEAKS = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
HBM = PEAKS.get("hbm_gbs", 6650.0)
TF = PEAKS.get("bf16_tflops", 1590.0)


def timeit(fn, reps=5, warm=2, inner=8):
    """median over `reps` of (CUDA-event time of `inner` back-to-back calls) / inner: the launch queue stays full, so
    host-side call overhead (~20-50 us per op through Python) does not leak into sub-millisecond kernels"""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(inner):
            fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / inner)
    ts.sort()
    return ts[len(ts) // 2]


RESULTS = []


def report(name, ms, nbytes=None, flops=None, note=""):
    r = {"kernel": name, "ms": ms, "note": note}
    if nbytes is not None:
        r.update(gbs=nbytes / ms / 1e6, hbm_frac=nbytes / ms / 1e6 / HBM, bytes=nbytes)
    if flops is not None:
        r.update(tflops=flops / ms / 1e9, tensor_frac=flops / ms / 1e9 / TF, flops=flops)
    RESULTS.append(r)
    s = f"{name:58s} {ms:9.3f} ms"
    if nbytes is not None:
        s += f"  {r['gbs']:8.1f} GB/s ({100 * r['hbm_frac']:5.1f}% of measured {HBM:.0f})"
    if flops is not None:
        s += f"  {r['tflops']:8.2f} TFLOP/s ({100 * r['tensor_frac']:5.2f}% of bf16 {TF:.0f})"
    print(s + ("  " + note if note else ""), flush=True)


def bench_rqs():
    for K in (8, 10):
        n = 1 << 24
        x = torch.rand(n, device=DEV)
        w, h = torch.randn(n, K, device=DEV), torch.randn(n, K, device=DEV)
        d = torch.randn(n, K - 1, device=DEV)
        nbytes = n * 4 * (1 + 3 * K - 1 + 2)
        for inv in (False, True):
            with torch.no_grad():
                ms = timeit(lambda: ops.rqs_unit(x, w, h, d, inv, (1e-3, 1e-3, 1e-3)))
            report(f"rqs_unit K={K} {'inv' if inv else 'fwd'} n=2^24", ms, nbytes)
        gy, gl = torch.randn(n, device=DEV), torch.randn(n, device=DEV)
        y, ld, gx, gw, gh, gd = (torch.empty_like(t) for t in (x, x, x, w, h, d))

        def bwd():
            N._lib.call("nf_rqs_unit_backward", x.data_ptr(), w.data_ptr(), h.data_ptr(), d.data_ptr(), gy.data_ptr(),
                        gl.data_ptr(), gx.data_ptr(), gw.data_ptr(), gh.data_ptr(), gd.data_ptr(), n, K, 0, 1e-3, 1e-3,
                        1e-3, 0, N._lib.stream())
        report(f"rqs_unit K={K} backward n=2^24", timeit(bwd), n * 4 * (1 + 2 * (3 * K - 1) + 3))
        del x, w, h, d, gy, gl, y, ld, gx, gw, gh, gd


def bench_spline_tf():
    for (B, D, K) in ((1 << 22, 2, 8), (8192, 784, 10), (1 << 18, 16, 10)):
        P = 3 * K - 1
        mask = torch.zeros(D)
        mask[: D // 2] = 1
        Dt = int((mask == 0).sum())
        tidx = torch.nonzero(mask == 0).flatten().to(torch.int32).to(DEV)
        x = torch.randn(B, D, device=DEV) * 2
        maskd = mask.to(DEV)
        for compact in (True, False):
            params = torch.randn(B, (Dt if compact else D) * P, device=DEV)
            tag = "compact" if compact else "full  "
            nbytes = B * 4 * (2 * D + 1 + (Dt if compact else D) * P)
            for inv in (False, True):
                with torch.no_grad():
                    ms = timeit(lambda: ops.spline_transform(x, params, maskd, tidx, K, inv, 5.0, (1e-3, 1e-3, 1e-3),
                                                            None, compact))
                report(f"spline_transform {tag} B={B} D={D} K={K} {'inv' if inv else 'fwd'}", ms, nbytes,
                       note="bytes = x + y + ld + the params tensor as laid out")
            gy, gl = torch.randn(B, D, device=DEV), torch.randn(B, device=DEV)
            gx, gp = torch.empty_like(x), torch.zeros_like(params)

            def bwd():
                N._lib.call("nf_spline_transform_backward", x.data_ptr(), params.data_ptr(), maskd.data_ptr(),
                            tidx.data_ptr(), gy.data_ptr(), gl.data_ptr(), gx.data_ptr(), gp.data_ptr(), B, D, Dt, K, 0,
                            5.0, 1e-3, 1e-3, 1e-3, None, None, None, int(compact), 0, N._lib.stream())
            report(f"spline_transform {tag} B={B} D={D} K={K} backward", timeit(bwd, reps=3, inner=2),
                   B * 4 * (3 * D + 1 + 2 * (Dt if compact else D) * P))
            del params, gy, gl, gx, gp
        del x


def bench_affine():
    for (B, D) in ((1 << 24, 2), (1 << 18, 256), (1 << 20, 64)):
        x, s, b = (torch.randn(B, D, device=DEV) for _ in range(3))
        mask = torch.zeros(D, device=DEV)
        mask[: D // 2] = 1
        with torch.no_grad():
            ms = timeit(lambda: ops.affine_coupling(x, s, b, mask, False))
        report(f"affine_coupling fwd B={B} D={D}", ms, B * 4 * (4 * D + 1))
        gy, gl = torch.randn(B, D, device=DEV), torch.randn(B, device=DEV)
        gx, gs, gb = (torch.empty_like(x) for _ in range(3))

        def bwd():
            N._lib.call("nf_affine_coupling_backward", x.data_ptr(), s.data_ptr(), b.data_ptr(), mask.data_ptr(),
                        gy.data_ptr(), gl.data_ptr(), gx.data_ptr(), gs.data_ptr(), gb.data_ptr(), B, D, 0, 0,
                        N._lib.stream())
        report(f"affine_coupling bwd B={B} D={D}", timeit(bwd), B * 4 * (7 * D + 1))
        params = torch.randn(B, 2 * D, device=DEV)
        with torch.no_grad():
            ms = timeit(lambda: ops.affine_ar(x, params, 0))
        report(f"affine_ar (MAF.inverse) fwd B={B} D={D}", ms, B * 4 * (4 * D + 1))
        with torch.no_grad():
            ms = timeit(lambda: ops.std_normal_log_prob(x, gl))
        report(f"std_normal_log_prob B={B} D={D}", ms, B * 4 * (D + 2))
        sub, div, mul, add = (torch.rand(D, device=DEV) + 0.5 for _ in range(4))
        with torch.no_grad():
            ms = timeit(lambda: ops.feature_affine(x, sub, div, mul, add))
        report(f"feature_affine fwd B={B} D={D}", ms, B * 4 * 2 * D)
        ms = timeit(lambda: ops.col_stats(x))
        report(f"col_stats B={B} D={D}", ms, B * 4 * D)
        ms = timeit(lambda: ops.col_sum(x))
        report(f"col_sum (bias gradient) B={B} D={D}", ms, B * 4 * D)
        del x, s, b, gy, gl, gx, gs, gb, params


def bench_bn():
    for (B, H) in ((1 << 20, 64), (1 << 18, 512)):
        x = torch.randn(B, H, device=DEV)
        bn = torch.nn.BatchNorm1d(H).to(DEV)
        bn.train()
        with torch.no_grad():
            ms = timeit(lambda: ops.batchnorm_relu(x, bn))
        report(f"batchnorm+relu train fwd B={B} H={H}", ms, B * H * 4 * 3, note="2 reads (stats, apply) + 1 write")
        bn.eval()
        with torch.no_grad():
            ms = timeit(lambda: ops.batchnorm_relu(x, bn))
        report(f"batchnorm+relu eval fwd B={B} H={H}", ms, B * H * 4 * 2)
        del x


def bench_peaks():
    """Library throughput of the pipes the dense layers run on (SURVEY 8d: TF32 and FP32 peaks are not in
    MEASURED_PEAKS.json): torch.matmul (cuBLAS) 8192^3 in bf16, TF32 and plain fp32."""
    n = 8192
    flops = 2.0 * n ** 3
    a32, b32 = torch.randn(n, n, device=DEV), torch.randn(n, n, device=DEV)
    a16, b16 = a32.bfloat16(), b32.bfloat16()
    old = torch.backends.cuda.matmul.allow_tf32
    try:
        report("cuBLAS bf16 matmul 8192^3", timeit(lambda: torch.matmul(a16, b16), reps=3, inner=4), None, flops)
        torch.backends.cuda.matmul.allow_tf32 = True
        report("cuBLAS TF32 matmul 8192^3 (the pipe rate of the 3xTF32 kernels)", timeit(lambda: torch.matmul(a32, b32), reps=3, inner=4), None, flops)
        torch.backends.cuda.matmul.allow_tf32 = False
        report("cuBLAS fp32 matmul 8192^3 (FP32 pipe)", timeit(lambda: torch.matmul(a32, b32), reps=3, inner=2), None, flops)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def bench_gemm():
    shapes = [("MADE(64,512) in->H", 262144, 512, 64), ("MADE(64,512) H->H", 262144, 512, 512),
              ("MADE(64,512) H->2D", 262144, 128, 512), ("coupling(256,512) H->H", 262144, 512, 512),
              ("spline(784,1024) H->H", 4096, 1024, 1024), ("spline(784,1024) H->D*P", 4096, 22736, 1024),
              ("dW = dY^T X (512x512, B=262144)", 512, 512, 262144), ("dW = dY^T X (1024x1024, B=65536)", 1024, 1024, 65536),
              ("dW = dY^T X (11368x1024, B=4096)", 11368, 1024, 4096)]
    for name, M, Nn, K in shapes:
        if name.startswith("dW"):
            g = torch.randn(K, M, device=DEV)
            x = torch.randn(K, Nn, device=DEV)
            ms = timeit(lambda: ops.gemm(g, x, M, Nn, K, 1, M, Nn, 1), reps=3, inner=2)
            ms_tc = timeit(lambda: ops.linear_wgrad_tc(g, x), reps=3, inner=4)
            report(f"nf_linear_wgrad_tc 3xTF32 {name} [{M}x{Nn}x{K}]", ms_tc, None, 2.0 * M * Nn * K,
                   note="tensor pipe executes 3x these FLOPs")
            N.set_gemm_precision("tf32")
            ms_tc = timeit(lambda: ops.linear_wgrad_tc(g, x), reps=3, inner=4)
            N.set_gemm_precision("fp32")
            report(f"nf_linear_wgrad_tc 1xTF32 (reduced precision) {name} [{M}x{Nn}x{K}]", ms_tc, None, 2.0 * M * Nn * K)
        else:
            a = torch.randn(M, K, device=DEV)
            w = torch.randn(Nn, K, device=DEV)
            bias = torch.randn(Nn, device=DEV)
            ms = timeit(lambda: ops.linear_raw(a, w, bias, relu=True), reps=3, inner=2)
        report(f"nf_gemm fp32 {name} [{M}x{Nn}x{K}]", ms, None, 2.0 * M * Nn * K)
        if not name.startswith("dW"):
            hi, lo = ops.split_tf32(w)
            if ops.linear_tc(a, hi, lo, bias, relu=True) is not None:
                ms = timeit(lambda: ops.linear_tc(a, hi, lo, bias, relu=True), reps=3, inner=4)
                report(f"nf_linear_tc 3xTF32 {name} [{M}x{Nn}x{K}]", ms, None, 2.0 * M * Nn * K,
                       note="tensor pipe executes 3x these FLOPs")
                N.set_gemm_precision("tf32")
                ms = timeit(lambda: ops.linear_tc(a, hi, lo, bias, relu=True), reps=3, inner=4)
                N.set_gemm_precision("fp32")
                report(f"nf_linear_tc 1xTF32 (reduced precision) {name} [{M}x{Nn}x{K}]", ms, None, 2.0 * M * Nn * K)


def bench_stacks():
    torch.manual_seed(0)
    B = 1 << 20
    x = torch.randn(B, 2, device=DEV)
    m = N.RealNVP(2, 8, 64).to(DEV).eval()
    with torch.no_grad():
        for p in m.parameters():
            p.add_(0.05 * torch.randn_like(p))
        ms = timeit(lambda: m.inverse(x))
    report("coupling_stack RealNVP(2,8,64) inverse B=2^20", ms, B * 20, 8 * 2 * 2 * (2 * 64 + 64 * 64 + 64 * 2) * B)
    m = N.RealNVPSpline(2, 8, 64).to(DEV).eval()
    with torch.no_grad():
        for p in m.parameters():
            p.add_(0.05 * torch.randn_like(p))
        ms = timeit(lambda: m.inverse(x))
    report("spline_stack RealNVPSpline(2,8,64) K=10 inverse B=2^20", ms, B * 20, 8 * 2 * (2 * 64 + 64 * 64 + 64 * 58) * B)
    import time
    xs = torch.randn(128, 2, device=DEV)
    with torch.no_grad():
        for _ in range(20):
            m.inverse(xs)
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(200):
            m.inverse(xs)
        host_us = (time.perf_counter() - t) / 200 * 1e6
        torch.cuda.synchronize()
    print(f"host-side cost of one fused model.inverse call (B=128, launch queue not full): {host_us:.1f} us")
    maf = N.MaskedAutoregressiveFlow(64, 512).to(DEV).eval()
    xm = torch.randn(262144, 64, device=DEV)
    with torch.no_grad():
        ms = timeit(lambda: maf.inverse(xm), reps=3, inner=2)
        report("MAF(64,512).inverse B=262144 (4 GEMMs + transform)", ms, 262144 * 516, 1245184 * 262144)
        ms = timeit(lambda: maf.forward(xm), reps=3, warm=1, inner=1)
        report("MAF(64,512).forward sequential B=262144", ms, 262144 * 516, 1245184 * 262144)


def bench_spline_tf_ncu():
    """one launch of each compact spline transform kernel (forward, inverse, backward) on two shapes + rqs_unit:
    the target of the ncu --set full capture (scripts/gpu_r02p.sh)"""
    for (B, D, K) in ((1 << 22, 2, 8), (8192, 784, 10), (1 << 18, 16, 10)):
        P = 3 * K - 1
        mask = torch.zeros(D)
        mask[: D // 2] = 1
        Dt = int((mask == 0).sum())
        tidx = torch.nonzero(mask == 0).flatten().to(torch.int32).to(DEV)
        x = torch.randn(B, D, device=DEV) * 2
        maskd = mask.to(DEV)
        params = torch.randn(B, Dt * P, device=DEV)
        gy, gl = torch.randn(B, D, device=DEV), torch.randn(B, device=DEV)
        gx, gp = torch.empty_like(x), torch.zeros_like(params)
        with torch.no_grad():
            for inv in (False, True):
                ops.spline_transform(x, params, maskd, tidx, K, inv, 5.0, (1e-3, 1e-3, 1e-3), None, True)
        N._lib.call("nf_spline_transform_backward", x.data_ptr(), params.data_ptr(), maskd.data_ptr(), tidx.data_ptr(),
                    gy.data_ptr(), gl.data_ptr(), gx.data_ptr(), gp.data_ptr(), B, D, Dt, K, 0, 5.0, 1e-3, 1e-3, 1e-3,
                    None, None, None, 1, 0, N._lib.stream())
        torch.cuda.synchronize()
    n, K = 1 << 22, 8
    xx = torch.rand(n, device=DEV)
    w, h, d = torch.randn(n, K, device=DEV), torch.randn(n, K, device=DEV), torch.randn(n, K - 1, device=DEV)
    with torch.no_grad():
        ops.rqs_unit(xx, w, h, d, False, (1e-3, 1e-3, 1e-3))
    torch.cuda.synchronize()
    print("spline_tf_ncu: done")


def bench_skinny():
    """first / last Linear of a 2-D conditioner (RealNVP(2, 8, 256), RealNVP(2, 10, 128), MADE(2, 64)): streaming kernels"""
    for (B, H, D) in ((1 << 20, 256, 2), (1 << 20, 128, 2), (1 << 20, 64, 2)):
        x = torch.randn(B, D, device=DEV)
        h = torch.randn(B, H, device=DEV)
        w1, b1 = torch.randn(H, D, device=DEV), torch.randn(H, device=DEV)
        w3, b3 = torch.randn(2 * D, H, device=DEV), torch.randn(2 * D, device=DEV)
        with torch.no_grad():
            report(f"skinny first Linear [{B} x {D}] -> {H} (+bias, ReLU)", timeit(lambda: ops.linear_raw(x, w1, b1, relu=True)),
                   B * 4 * (D + H))
            report(f"skinny last Linear [{B} x {H}] -> {2 * D} (+bias)", timeit(lambda: ops.linear_raw(h, w3, b3)),
                   B * 4 * (H + 2 * D))
        del x, h
    # training-side skinny products of a 2-D spline / coupling conditioner (2^20 rows, hidden 64)
    B, H = 1 << 20, 64
    gy = torch.randn(B, 23, device=DEV)
    w = torch.randn(23, H, device=DEV)
    report(f"skinny input gradient of the spline head dX[{B} x {H}] = dY[. x 23] W", timeit(lambda: ops.gemm(gy, w, B, H, 23, 23, 1, H, 1)),
           B * 4 * (23 + H))
    g1, x2 = torch.randn(B, H, device=DEV), torch.randn(B, 2, device=DEV)
    report(f"skinny weight gradient dW[{H} x 2] = dY[{B} x {H}]^T x", timeit(lambda: ops.gemm(g1, x2, H, 2, B, 1, H, 2, 1)),
           B * 4 * (H + 2))
    del gy, g1, x2


ALL = {"peaks": bench_peaks, "rqs": bench_rqs, "spline_tf": bench_spline_tf, "affine": bench_affine, "bn": bench_bn, "gemm": bench_gemm,
       "stacks": bench_stacks, "skinny": bench_skinny, "spline_tf_ncu": bench_spline_tf_ncu}

if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    ap.add_argument("--json", default="")
    a = ap.parse_args()
    names = [n for n in a.only.split(",") if n] or [n for n in ALL if not n.endswith("_ncu")]
    print(f"peaks: HBM {HBM} GB/s, bf16 {TF} TFLOP/s ({'measured' if PEAKS else 'fallback'})")
    for n in names:
        ALL[n]()
        torch.cuda.empty_cache()
    if a.json:
        json.dump({"peaks": {"hbm_gbs": HBM, "bf16_tflops": TF}, "results": RESULTS}, open(a.json, "w"), indent=1)
