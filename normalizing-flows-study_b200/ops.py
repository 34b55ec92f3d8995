"""Tensor-level wrappers and autograd Functions over the C ABI (include/nfb200.h).

Two families:
  * layer-wise ops with hand-written backward kernels (training / general path):
      linear (F.linear incl. MaskedLinear's W*mask, masked_linear.py:14-18), batchnorm_relu
      (nn.BatchNorm1d+ReLU of coupling_layer.py:18-35), affine_coupling, spline_transform,
      affine_ar, rqs_unit;
  * fused inference launches (no autograd): stack, made_affine,
    ar_sequential.
Every op allocates its outputs with torch (device memory plumbing) and launches on the
current CUDA stream.  Nothing here has a CPU implementation.
"""
from __future__ import annotations

import weakref

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib as L

ptr, call, stream = L.ptr, L.call, L.stream

USE_TENSOR_CORE_GEMM = True      # tcgen05 3xTF32 GEMMs for float32 layers; False forces the FP32-pipe GEMM
USE_MASK_PLANS = True            # skip the exactly-zero K ranges / tiles of 2-D weight masks (MADE) in the training GEMMs


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


def _same_dtype(ref, *ts):
    return [None if t is None else (t if t.dtype == ref.dtype else t.to(ref.dtype)) for t in ts]


# --------------------------------------------------------------------------------------------
# raw kernels (no autograd)
# --------------------------------------------------------------------------------------------
def gemm(A, Bm, M, N, K, sam, sak, sbk, sbn, bias=None, relu=False, out=None, accumulate=False, k_extent=None):
    """C[M,N] (+)= A[M,K]*B[K,N] with element strides; see nf_gemm in include/nfb200.h."""
    if out is None:
        out = torch.empty((M, N), dtype=A.dtype, device=A.device)
    call("nf_gemm", ptr(A), ptr(Bm), ptr(out), ptr(bias), M, N, K, sam, sak, sbk, sbn, N, int(relu), int(accumulate),
         ptr(k_extent), L.dtype_code(A), stream())
    return out


def linear_raw(x, w, bias=None, relu=False, k_extent=None):
    """y = relu?(x @ w.T + bias) for contiguous x [M,K], w [N,K]."""
    M, K = x.shape
    N = w.shape[0]
    return gemm(x, w, M, N, K, K, 1, 1, K, bias=bias, relu=relu, k_extent=k_extent)


def split_tf32(w):
    """(hi, lo) operands of the 3xTF32 tensor-core GEMM for a contiguous fp32 weight."""
    w = _c(w)
    hi, lo = torch.empty_like(w), torch.empty_like(w)
    call("nf_split_tf32", ptr(w), ptr(hi), ptr(lo), w.numel(), stream())
    return hi, lo


def linear_tc(x, w_hi, w_lo, bias=None, relu=False, k_extent=None, out=None, k_begin=None):
    """y = relu?(x @ W.T + bias) on tcgen05 (3xTF32, fp32-accurate); returns None when the shape / alignment is not
    taken by the tensor-core kernel (caller uses linear_raw).  k_extent / k_begin: int32 per 64 output columns, the
    K range outside of which W is exactly zero for those outputs (mask-folded MADE weights)."""
    M, K = x.shape
    N = w_hi.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=x.dtype, device=x.device)
    if K % 4 != 0:
        return None
    if k_begin is None:
        ok = L.try_call("nf_linear_tc", ptr(x), ptr(w_hi), ptr(w_lo), ptr(bias), ptr(out), M, N, K, K, K, N, int(relu),
                        ptr(k_extent), stream())
    else:
        ok = L.try_call("nf_linear_tc_range", ptr(x), ptr(w_hi), ptr(w_lo), ptr(bias), ptr(out), M, N, K, K, K, N,
                        int(relu), ptr(k_begin), ptr(k_extent), stream())
    return out if ok else None


class MaskPlan:
    """Zero structure of a 2-D weight mask [N, K] (MaskedLinear.mask, masked_linear.py:10): the K ranges / tiles the
    tensor-core GEMMs of the layer may skip.  MADE masks are block lower-triangular once the hidden units are sorted
    by degree (they are for data_dim > 2, made.py:36), so ~44 % of the 128 x 128 tiles are exactly zero."""
    __slots__ = ("k_extent", "k_begin_t", "tile_live", "live_fraction", "owner")


_MASK_PLANS = {}


def mask_plan(mask):
    if mask is None or mask.dim() != 2 or mask.shape[0] < 256 or mask.shape[1] < 256:
        return None
    from . import packing
    key = (id(mask), packing.tensors_key([mask]), tuple(mask.shape))
    plan = _MASK_PLANS.get(key)
    # the entry pins its mask through a weak reference: a freed mask's address (and id) may be handed to a new mask
    # of the same shape with different degrees, whose zero structure must not be taken from the stale plan
    if plan is not None and plan.owner() is not mask:
        plan = None
    if plan is None:
        if len(_MASK_PLANS) > 256:
            _MASK_PLANS.clear()
        nz = mask != 0
        N, K = nz.shape
        dev = mask.device
        last = torch.where(nz, torch.arange(1, K + 1, device=dev)[None, :], 0).amax(dim=1)        # per output row n
        first = torch.where(nz, torch.arange(N, device=dev)[:, None], N).amin(dim=0)              # per input column k

        def grouped(v, g, fill, red):
            pad = (-v.numel()) % g
            if pad:
                v = torch.cat([v, torch.full((pad,), fill, dtype=v.dtype, device=dev)])
            return red(v.view(-1, g), dim=1).to(torch.int32).contiguous()
        plan = MaskPlan()
        plan.k_extent = grouped(last, 64, 0, torch.amax)
        plan.k_begin_t = grouped(first, 64, N, torch.amin)
        tn, tk = (N + 127) // 128, (K + 127) // 128
        padded = torch.zeros(tn * 128, tk * 128, dtype=torch.bool, device=dev)
        padded[:N, :K] = nz
        live = padded.view(tn, 128, tk, 128).any(dim=3).any(dim=1)
        plan.tile_live = live.to(torch.uint8).contiguous().view(-1)
        plan.live_fraction = float(live.float().mean())
        plan.owner = weakref.ref(mask)
        _MASK_PLANS[key] = plan
    return plan if plan.live_fraction < 0.95 else None


def linear_wgrad_tc(gy, x, out=None, tile_live=None):
    """dW[N,K] = gy[B,N]^T x[B,K] on tcgen05 (3xTF32, deterministic split over the batch); None when the shape /
    alignment is not taken by the tensor-core kernel (caller uses gemm).  tile_live: MaskPlan.tile_live (128 x 128
    tiles on which the weight mask is all zero are written as zeros without being computed)."""
    B, N = gy.shape
    K = x.shape[1]
    if K % 4 != 0:
        return None
    if out is None:
        out = torch.empty((N, K), dtype=gy.dtype, device=gy.device)
    ws_bytes = int(L.lib().nf_linear_wgrad_tc_workspace(B, N, K))
    ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=gy.device) if ws_bytes else None
    if tile_live is None:
        ok = L.try_call("nf_linear_wgrad_tc", ptr(gy), ptr(x), ptr(out), B, N, K, N, K, K, ptr(ws), ws_bytes, stream())
    else:
        ok = L.try_call("nf_linear_wgrad_tc_masked", ptr(gy), ptr(x), ptr(out), B, N, K, N, K, K, ptr(ws), ws_bytes,
                        ptr(tile_live), stream())
    return out if ok else None


def mul_rows(a, b):
    """a * b where b has a's shape or is a single row broadcast over a's rows."""
    a2 = a.view(-1, a.shape[-1])
    out = torch.empty_like(a2)
    b_rows = 1 if b.dim() == 1 else a2.shape[0]
    call("nf_mul_rows", ptr(a2), ptr(_c(b)), ptr(out), a2.shape[0], a2.shape[1], b_rows, L.dtype_code(a), stream())
    return out.view_as(a)


def col_sum(a):
    out = torch.empty(a.shape[1], dtype=a.dtype, device=a.device)
    call("nf_col_sum", ptr(a), ptr(out), a.shape[0], a.shape[1], L.dtype_code(a), stream())
    return out


def relu_backward(y, gy):
    gx = torch.empty_like(gy)
    call("nf_relu_backward", ptr(y), ptr(gy), ptr(gx), gy.numel(), L.dtype_code(gy), stream())
    return gx


def relu_backward_colsum(y, gy):
    """(gy * (y > 0), its column sums) in one pass: the ReLU backward of a Linear(+ReLU) and that Linear's bias gradient."""
    gx = torch.empty_like(gy)
    cs = torch.empty(gy.shape[1], dtype=gy.dtype, device=gy.device)
    call("nf_relu_backward_colsum", ptr(y), ptr(gy), ptr(gx), ptr(cs), gy.shape[0], gy.shape[1], L.dtype_code(gy), stream())
    return gx, cs


# --------------------------------------------------------------------------------------------
# Linear (+ optional weight mask, + optional fused ReLU)
# --------------------------------------------------------------------------------------------
def _tc_ok(x, K):
    return USE_TENSOR_CORE_GEMM and x.dtype == torch.float32 and x.shape[0] >= 256 and K % 4 == 0


class _LinearFn(Function):
    """F.linear(x, W*mask, b) (+ReLU).  float32 with >= 256 rows: forward and the input gradient run on tcgen05
    (3xTF32, fp32-accurate; the weight is split hi/lo per call -- weights are small next to the activations);
    so does the weight gradient (reduction over the batch, both operands in their row-major layout, wgrad_tc.cu);
    float64 and tiny / unaligned shapes use the FP32/FP64-pipe GEMM."""

    @staticmethod
    def forward(ctx, x, weight, bias, mask, relu):
        x = _c(x)
        w_eff = _c(weight) if mask is None else mul_rows(_c(weight), mask)
        b = None if bias is None else _c(bias)
        y = None
        plan = mask_plan(mask) if USE_MASK_PLANS else None
        if _tc_ok(x, x.shape[1]):
            hi, lo = split_tf32(w_eff)
            y = linear_tc(x, hi, lo, b, relu, k_extent=None if plan is None else plan.k_extent)
        if y is None:
            y = linear_raw(x, w_eff, b, relu)
        ctx.relu = relu
        ctx.has_bias = bias is not None
        ctx.save_for_backward(x, w_eff, mask, y if relu else None)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, w_eff, mask, y = ctx.saved_tensors
        g = _c(gy)
        gb_fused = None
        if ctx.relu:
            if ctx.has_bias and ctx.needs_input_grad[2] and g.dim() == 2:
                g, gb_fused = relu_backward_colsum(y, g)      # the bias gradient comes out of the same pass
            else:
                g = relu_backward(y, g)
        M, K = x.shape
        N = w_eff.shape[0]
        gx = gw = gb = None
        plan = mask_plan(mask) if USE_MASK_PLANS else None
        if ctx.needs_input_grad[0]:
            if _tc_ok(g, N):
                hi, lo = split_tf32(w_eff.t().contiguous())             # [K, N]: dX = dY (W^T)^T
                gx = linear_tc(g, hi, lo, k_begin=None if plan is None else plan.k_begin_t)
            if gx is None:
                gx = gemm(g, w_eff, M, K, N, N, 1, K, 1)                 # dX = dY W
        if ctx.needs_input_grad[1]:
            gw = linear_wgrad_tc(g, x, tile_live=None if plan is None else plan.tile_live) if _tc_ok(g, K) else None   # dW = dY^T X
            if gw is None:
                gw = gemm(g, x, N, K, M, 1, N, K, 1)
            if mask is not None:
                gw = mul_rows(gw, mask)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = gb_fused if gb_fused is not None else col_sum(g)
        return gx, gw, gb, None, None


def linear(x, weight, bias=None, mask=None, relu=False):
    """F.linear(x, weight*mask, bias) (+ReLU).  mask: None, [in] (column mask, broadcast) or [out,in]."""
    weight, bias, mask = _same_dtype(x, weight, bias, mask)
    return _LinearFn.apply(x, weight, bias, mask, relu)


def _product(a, w):
    """a [M, K] @ w[N, K]^T without bias, on the route _LinearFn takes for that shape: tcgen05 (3xTF32) for float32 with
    >= 256 rows and K % 4 == 0, the FP32 / FP64-pipe nf_gemm otherwise."""
    M, K = a.shape
    N = w.shape[0]
    if _tc_ok(a, K):
        hi, lo = split_tf32(w)
        y = linear_tc(a, hi, lo)
        if y is not None:
            return y
    return gemm(a, w, M, N, K, K, 1, 1, K)


def _wgrad(g, a):
    """dW[N, K] = g[B, N]^T a[B, K], on the route _LinearFn.backward takes."""
    B, N = g.shape
    K = a.shape[1]
    gw = linear_wgrad_tc(g, a) if _tc_ok(g, K) else None
    return gw if gw is not None else gemm(g, a, N, K, B, 1, N, K, 1)


class _LinearCtxFn(Function):
    """relu(W[:, :D] (x*mask) + W[:, D:] c + b): the first Linear of a conditional coupling conditioner, whose input is
    [x*mask, c] (context columns last), without concatenating x and c.  Two products into one output: the context one
    without bias, then the masked x one with bias and ReLU accumulated onto it (nf_gemm computes relu(acc + bias + C_old)
    on every path).  `div`: row r of x uses context row r // div; 1 (one context row per row) or, with a single context
    row, anything (that row is read with row stride 0).  relu=False (the affine conditioner, whose BatchNorm follows the
    Linear): the same products without the ReLU."""

    @staticmethod
    def forward(ctx, x, c, weight, bias, mask, div, relu=True):
        x, c = _c(x), _c(c)
        B, D = x.shape
        H, C = weight.shape[0], c.shape[1]
        wx = mul_rows(_c(weight[:, :D]), mask)                      # x*mask folded into the x columns, as linear()
        wc = _c(weight[:, D:])
        per_row = c.shape[0] == B and div == 1
        y = _product(c, wc) if per_row else gemm(c, wc, B, H, C, 0, 1, 1, C)
        gemm(x, wx, B, H, D, D, 1, 1, D, bias=_c(bias), relu=relu, out=y, accumulate=True)
        ctx.per_row, ctx.relu = per_row, relu
        ctx.save_for_backward(x, c, wx, wc, mask, y)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, c, wx, wc, mask, y = ctx.saved_tensors
        B, D = x.shape
        H, C = wc.shape
        if ctx.relu:
            g, gb = relu_backward_colsum(y, _c(gy))                 # the bias gradient comes out of the same pass
        else:
            g = _c(gy)
            gb = col_sum(g)
        gx = gc = gw = None
        if ctx.needs_input_grad[0]:
            gx = _product(g, _c(wx.t()))                            # dX = dY Wx
        if ctx.needs_input_grad[1]:                                 # one shared row: (column sums of dY) Wc
            gc = _product(g, _c(wc.t())) if ctx.per_row else gemm(gb.view(1, H), wc, 1, C, H, H, 1, C, 1)
        if ctx.needs_input_grad[2]:
            gw = torch.empty((H, D + C), dtype=g.dtype, device=g.device)
            gw[:, :D] = mul_rows(_wgrad(g, x), mask)
            gw[:, D:] = _wgrad(g, c) if ctx.per_row else gemm(gb.view(H, 1), c, H, C, 1, 1, 1, C, 1)
        return gx, gc, gw, (gb if ctx.needs_input_grad[3] else None), None, None, None


def linear_ctx(x, c, weight, bias, mask, div, relu=True):
    """relu(F.linear(cat([x*mask, c[r // div]]), weight, bias)) with x [B, D], c [rows, C], weight [H, D+C] (see
    _LinearCtxFn); relu=False: without the ReLU."""
    weight, bias, mask, c = _same_dtype(x, weight, bias, mask, c)
    return _LinearCtxFn.apply(x, c, weight, bias, mask, int(div), bool(relu))


# --------------------------------------------------------------------------------------------
# BatchNorm1d (+ReLU)
# --------------------------------------------------------------------------------------------
class _BatchNormFn(Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, training, momentum, eps, relu):
        x = _c(x)
        B, H = x.shape
        y = torch.empty_like(x)
        sm = torch.empty(H, dtype=x.dtype, device=x.device)
        sr = torch.empty(H, dtype=x.dtype, device=x.device)
        ws = torch.empty(2 * H, dtype=torch.float64, device=x.device) if training else None
        call("nf_batchnorm_forward", ptr(x), ptr(_c(gamma)), ptr(_c(beta)), ptr(running_mean), ptr(running_var),
             ptr(y), ptr(sm), ptr(sr), ptr(ws), B, H, int(training), float(momentum), float(eps), int(relu),
             L.dtype_code(x), stream())
        ctx.relu, ctx.training = relu, training
        ctx.save_for_backward(x, y, gamma, sm, sr, beta)
        ctx.mark_non_differentiable(sm, sr)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, y, gamma, sm, sr, beta = ctx.saved_tensors
        B, H = x.shape
        gx = torch.empty_like(x)
        gg = torch.empty_like(sm)
        gb = torch.empty_like(sm)
        ws = torch.empty(2 * H, dtype=torch.float64, device=x.device)
        call("nf_batchnorm_backward", ptr(x), ptr(y), ptr(_c(gamma)), ptr(sm), ptr(sr), ptr(_c(gy)), ptr(gx), ptr(gg),
             ptr(gb), ptr(ws), B, H, int(ctx.relu), int(ctx.training), L.dtype_code(x), ptr(_c(beta)), stream())
        return gx, gg, gb, None, None, None, None, None, None


# Synchronised batch statistics (SURVEY 8e).  CouplingLayer's train-mode BatchNorm (coupling_layer.py:18-35) is the one
# cross-row reduction of the path: with per-shard statistics an N-GPU data-parallel step differs from the 1-GPU step on
# the same global batch.  When a process group is registered here (parallel.DataParallelFlow(sync_batchnorm=True) or
# parallel.enable_sync_batchnorm()), every train-mode BatchNorm all-reduces its [2H + 1] triple (sum x, sum x^2, n)
# between the statistics pass and the normalisation, and the two batch sums of its backward.
_SYNC_BN = {"group": None, "enabled": False}


def set_sync_batchnorm(enabled: bool, group=None):
    _SYNC_BN["enabled"], _SYNC_BN["group"] = bool(enabled), group


def _sync_bn_world():
    if not _SYNC_BN["enabled"]:
        return 1
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return 1
    return dist.get_world_size(_SYNC_BN["group"])


def allreduce_bn_sums(ws, count, group=None):
    """ws: float64 [2H] local sums; count: local row count.  Returns (global sums in ws, global count); one collective."""
    import torch.distributed as dist
    packed = torch.cat([ws, ws.new_tensor([float(count)])])
    dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
    ws.copy_(packed[:-1])
    return ws, int(round(float(packed[-1])))


class _SyncBatchNormFn(Function):
    """Train-mode BatchNorm1d (+ReLU) with statistics over all ranks' rows.  One all-reduce of [2H + 1] doubles in the
    forward (sum x, sum x^2, row count) and one of [2H] in the backward; the global row count stays on the device
    (`count = -1`: the kernels read it from workspace[2H]), so the pass has no host synchronisation."""

    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, momentum, eps, relu, group):
        import torch.distributed as dist
        x = _c(x)
        B, H = x.shape
        y = torch.empty_like(x)
        sm = torch.empty(H, dtype=x.dtype, device=x.device)
        sr = torch.empty(H, dtype=x.dtype, device=x.device)
        packed = torch.empty(2 * H + 1, dtype=torch.float64, device=x.device)
        code = L.dtype_code(x)
        call("nf_batchnorm_forward_staged", ptr(x), None, None, None, None, None, None, None, ptr(packed), B, H, 0.0, float(eps),
             int(relu), 1, 0, code, stream())
        packed[2 * H:].fill_(float(B))
        dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
        call("nf_batchnorm_forward_staged", ptr(x), ptr(_c(gamma)), ptr(_c(beta)), ptr(running_mean), ptr(running_var),
             ptr(y), ptr(sm), ptr(sr), ptr(packed), B, H, float(momentum), float(eps), int(relu), 2, -1, code, stream())
        ctx.relu, ctx.group = relu, group
        ctx.save_for_backward(x, y, gamma, sm, sr, packed[2 * H:], beta)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        import torch.distributed as dist
        x, y, gamma, sm, sr, count, beta = ctx.saved_tensors
        B, H = x.shape
        code = L.dtype_code(x)
        gy = _c(gy)
        gx = torch.empty_like(x)
        glob = torch.empty(2 * H + 1, dtype=torch.float64, device=x.device)
        call("nf_batchnorm_backward_staged", ptr(x), ptr(y), ptr(_c(gamma)), ptr(sm), ptr(sr), ptr(gy), None, None, None, ptr(glob),
             B, H, int(ctx.relu), 1, 0, code, ptr(_c(beta)), stream())
        gg = glob[:H].to(x.dtype)                         # this shard's ggamma / gbeta: the gradient all-reduce sums them
        gb = glob[H:2 * H].to(x.dtype)
        dist.all_reduce(glob[:2 * H], op=dist.ReduceOp.SUM, group=ctx.group)
        glob[2 * H:].copy_(count)
        gg_g = torch.empty(H, dtype=x.dtype, device=x.device)
        gb_g = torch.empty(H, dtype=x.dtype, device=x.device)
        call("nf_batchnorm_backward_staged", ptr(x), ptr(y), ptr(_c(gamma)), ptr(sm), ptr(sr), ptr(gy), ptr(gx), ptr(gg_g),
             ptr(gb_g), ptr(glob), B, H, int(ctx.relu), 2, -1, code, ptr(_c(beta)), stream())
        return gx, gg, gb, None, None, None, None, None, None


def batchnorm_relu(x, bn: torch.nn.BatchNorm1d, relu=True):
    """nn.BatchNorm1d forward (train: batch stats + running-stat update, eval: running stats) fused with ReLU."""
    training = bn.training or bn.running_mean is None
    if training and _sync_bn_world() > 1 and x.dtype in (torch.float32, torch.float64):
        momentum = 0.0
        if bn.track_running_stats and bn.running_mean is not None:
            if bn.num_batches_tracked is not None:
                bn.num_batches_tracked.add_(1)
            momentum = (1.0 / float(bn.num_batches_tracked)) if bn.momentum is None else bn.momentum
        rm, rv = bn.running_mean, bn.running_var
        if rm is not None and rm.dtype != x.dtype:
            rm32, rv32 = rm.to(x.dtype), rv.to(x.dtype)
            y = _SyncBatchNormFn.apply(x, bn.weight.to(x.dtype), bn.bias.to(x.dtype), rm32, rv32, momentum, bn.eps, relu,
                                       _SYNC_BN["group"])
            rm.copy_(rm32)
            rv.copy_(rv32)
            return y
        return _SyncBatchNormFn.apply(x, bn.weight, bn.bias, rm, rv, momentum, bn.eps, relu, _SYNC_BN["group"])
    momentum = 0.0
    if training and bn.track_running_stats and bn.running_mean is not None:
        if bn.num_batches_tracked is not None:
            bn.num_batches_tracked.add_(1)
        momentum = (1.0 / float(bn.num_batches_tracked)) if bn.momentum is None else bn.momentum
    rm, rv = bn.running_mean, bn.running_var
    if rm is not None and rm.dtype != x.dtype:       # mixed dtypes: keep the module's buffers authoritative
        rm32, rv32 = rm.to(x.dtype), rv.to(x.dtype)
        y = _BatchNormFn.apply(x, bn.weight.to(x.dtype), bn.bias.to(x.dtype), rm32, rv32, training, momentum, bn.eps, relu)
        if training:
            rm.copy_(rm32)
            rv.copy_(rv32)
        return y
    return _BatchNormFn.apply(x, bn.weight, bn.bias, rm, rv, training, momentum, bn.eps, relu)


# --------------------------------------------------------------------------------------------
# transforms
# --------------------------------------------------------------------------------------------
class _AffineCouplingFn(Function):
    @staticmethod
    def forward(ctx, x, s_raw, b_raw, mask, inverse):
        x, s_raw, b_raw = _c(x), _c(s_raw), _c(b_raw)
        B, D = x.shape
        y = torch.empty_like(x)
        ld = torch.empty(B, dtype=x.dtype, device=x.device)
        call("nf_affine_coupling_forward", ptr(x), ptr(s_raw), ptr(b_raw), ptr(mask), ptr(y), ptr(ld), B, D,
             int(inverse), L.dtype_code(x), stream())
        ctx.inverse = inverse
        ctx.save_for_backward(x, s_raw, b_raw, mask)
        return y, ld

    @staticmethod
    @once_differentiable
    def backward(ctx, gy, gld):
        x, s_raw, b_raw, mask = ctx.saved_tensors
        B, D = x.shape
        gx, gs, gb = torch.empty_like(x), torch.empty_like(x), torch.empty_like(x)
        call("nf_affine_coupling_backward", ptr(x), ptr(s_raw), ptr(b_raw), ptr(mask), ptr(_c(gy)), ptr(_c(gld)),
             ptr(gx), ptr(gs), ptr(gb), B, D, int(ctx.inverse), L.dtype_code(x), stream())
        return gx, gs, gb, None, None


def affine_coupling(x, s_raw, b_raw, mask, inverse):
    return _AffineCouplingFn.apply(x, s_raw, b_raw, _c(mask.to(x.dtype)), inverse)


class _SplineTransformFn(Function):
    @staticmethod
    def forward(ctx, x, params, mask, tidx, K, inverse, bound, mins, rescale, compact):
        x, params = _c(x), _c(params)
        B, D = x.shape
        y = torch.empty_like(x)
        ld = torch.empty(B, dtype=x.dtype, device=x.device)
        r = rescale if rescale is not None else (None, None, None)
        call("nf_spline_transform_forward", ptr(x), ptr(params), ptr(mask), ptr(tidx), ptr(y), ptr(ld), B, D,
             tidx.numel(), K, int(inverse), bound, mins[0], mins[1], mins[2], ptr(r[0]), ptr(r[1]), ptr(r[2]),
             int(compact), L.dtype_code(x), stream())
        ctx.cfg = (K, inverse, bound, mins, compact)
        ctx.rescale = rescale
        ctx.save_for_backward(x, params, mask, tidx)
        return y, ld

    @staticmethod
    @once_differentiable
    def backward(ctx, gy, gld):
        x, params, mask, tidx = ctx.saved_tensors
        K, inverse, bound, mins, compact = ctx.cfg
        B, D = x.shape
        r = ctx.rescale if ctx.rescale is not None else (None, None, None)
        gx = torch.empty_like(x)
        gp = torch.empty_like(params) if compact else torch.zeros_like(params)
        call("nf_spline_transform_backward", ptr(x), ptr(params), ptr(mask), ptr(tidx), ptr(_c(gy)), ptr(_c(gld)),
             ptr(gx), ptr(gp), B, D, tidx.numel(), K, int(inverse), bound, mins[0], mins[1], mins[2], ptr(r[0]),
             ptr(r[1]), ptr(r[2]), int(compact), L.dtype_code(x), stream())
        return gx, gp, None, None, None, None, None, None, None, None


def spline_transform(x, params, mask, tidx, K, inverse, bound, mins, rescale=None, compact=False):
    """params: [B, D*(3K-1)] (reference layout) or, with compact=True, [B, Dt*(3K-1)] (transformed dims only)."""
    return _SplineTransformFn.apply(x, params, _c(mask.to(x.dtype)), tidx, K, inverse, float(bound),
                                    tuple(float(m) for m in mins), rescale, bool(compact))


class _AffineARFn(Function):
    @staticmethod
    def forward(ctx, v, params, mode):
        v, params = _c(v), _c(params)
        B, D = v.shape
        out = torch.empty_like(v)
        ld = torch.empty(B, dtype=v.dtype, device=v.device)
        call("nf_affine_ar_forward", ptr(v), ptr(params), ptr(out), ptr(ld), B, D, mode, L.dtype_code(v), stream())
        ctx.mode = mode
        ctx.save_for_backward(v, params, ld)
        return out, ld

    @staticmethod
    @once_differentiable
    def backward(ctx, gout, gld):
        v, params, ld = ctx.saved_tensors
        B, D = v.shape
        gv, gp = torch.empty_like(v), torch.empty_like(params)
        call("nf_affine_ar_backward", ptr(v), ptr(params), ptr(ld), ptr(_c(gout)), ptr(_c(gld)), ptr(gv), ptr(gp), B, D,
             ctx.mode, L.dtype_code(v), stream())
        return gv, gp, None


def affine_ar(v, params, mode):
    return _AffineARFn.apply(v, params, mode)


class _RqsUnitFn(Function):
    @staticmethod
    def forward(ctx, x, w, h, d, inverse, mins):
        x, w, h, d = _c(x), _c(w), _c(h), _c(d)
        n, K = x.numel(), w.shape[-1]
        y, ld = torch.empty_like(x), torch.empty_like(x)
        call("nf_rqs_unit_forward", ptr(x), ptr(w), ptr(h), ptr(d), ptr(y), ptr(ld), n, K, int(inverse), mins[0],
             mins[1], mins[2], L.dtype_code(x), stream())
        ctx.cfg = (inverse, mins)
        ctx.save_for_backward(x, w, h, d)
        return y, ld

    @staticmethod
    @once_differentiable
    def backward(ctx, gy, gld):
        x, w, h, d = ctx.saved_tensors
        inverse, mins = ctx.cfg
        n, K = x.numel(), w.shape[-1]
        gx, gw, gh, gd = torch.empty_like(x), torch.empty_like(w), torch.empty_like(h), torch.empty_like(d)
        call("nf_rqs_unit_backward", ptr(x), ptr(w), ptr(h), ptr(d), ptr(_c(gy)), ptr(_c(gld)), ptr(gx), ptr(gw),
             ptr(gh), ptr(gd), n, K, int(inverse), mins[0], mins[1], mins[2], L.dtype_code(x), stream())
        return gx, gw, gh, gd, None, None


def rqs_unit(x, w, h, d, inverse, mins):
    return _RqsUnitFn.apply(x, w, h, d, bool(inverse), tuple(float(m) for m in mins))


class _FeatureAffineFn(Function):
    """y = (x - sub) / div * mul + add, per feature; any of sub/div/mul/add may be None (add: python float ok)."""

    @staticmethod
    def forward(ctx, x, sub, div, mul, add):
        x = _c(x)
        B, D = x.shape
        y = torch.empty_like(x)
        add_t = add if isinstance(add, torch.Tensor) else None
        add_s = 0.0 if add is None or add_t is not None else float(add)
        call("nf_feature_affine_forward", ptr(x), ptr(sub), ptr(div), ptr(mul), ptr(add_t), add_s, ptr(y), B, D,
             L.dtype_code(x), stream())
        ctx.save_for_backward(x, sub, div, mul)
        ctx.add_is_tensor = add_t is not None
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        x, sub, div, mul = ctx.saved_tensors
        B, D = x.shape
        need = [sub is not None and ctx.needs_input_grad[1], div is not None and ctx.needs_input_grad[2],
                mul is not None and ctx.needs_input_grad[3], ctx.add_is_tensor and ctx.needs_input_grad[4]]
        outs = [torch.empty(D, dtype=x.dtype, device=x.device) if n else None for n in need]
        ws = torch.empty(2 * D, dtype=torch.float64, device=x.device) if any(need) else None
        gx = torch.empty_like(x)
        call("nf_feature_affine_backward", ptr(x), ptr(sub), ptr(div), ptr(mul), ptr(_c(gy)), ptr(gx), ptr(outs[0]),
             ptr(outs[1]), ptr(outs[2]), ptr(outs[3]), ptr(ws), B, D, L.dtype_code(x), stream())
        return gx, outs[0], outs[1], outs[2], outs[3]


def feature_affine(x, sub=None, div=None, mul=None, add=None):
    sub, div, mul = _same_dtype(x, sub, div, mul)
    if isinstance(add, torch.Tensor):
        add, = _same_dtype(x, add)
    return _FeatureAffineFn.apply(x, sub, div, mul, add)


def col_stats(x):
    """Per-feature batch mean and biased variance of x [B,D] (no autograd)."""
    x = _c(x.detach())
    B, D = x.shape
    mean = torch.empty(D, dtype=x.dtype, device=x.device)
    var = torch.empty(D, dtype=x.dtype, device=x.device)
    ws = torch.empty(2 * D, dtype=torch.float64, device=x.device)
    call("nf_col_stats", ptr(x), ptr(mean), ptr(var), ptr(ws), B, D, L.dtype_code(x), stream())
    return mean, var


class _ArStepFn(Function):
    @staticmethod
    def forward(ctx, cur, v, params, ld_in, col, mode):
        cur, v, params = _c(cur), _c(v), _c(params)
        B, D = v.shape
        out = torch.empty_like(v)
        ld = torch.empty(B, dtype=v.dtype, device=v.device)
        call("nf_ar_step_forward", ptr(cur), ptr(v), ptr(params), ptr(None if ld_in is None else _c(ld_in)), ptr(out),
             ptr(ld), B, D, col, mode, L.dtype_code(v), stream())
        ctx.cfg = (col, mode, ld_in is not None)
        ctx.save_for_backward(v, params)
        return out, ld

    @staticmethod
    @once_differentiable
    def backward(ctx, gout, gld):
        v, params = ctx.saved_tensors
        col, mode, has_ld = ctx.cfg
        B, D = v.shape
        gcur, gv, gp = torch.empty_like(v), torch.empty_like(v), torch.empty_like(params)
        gld = _c(gld)
        call("nf_ar_step_backward", ptr(v), ptr(params), ptr(_c(gout)), ptr(gld), ptr(gcur), ptr(gv), ptr(gp), B, D,
             col, mode, L.dtype_code(v), stream())
        return gcur, gv, gp, (gld if has_ld else None), None, None


def ar_step(cur, v, params, ld_in, col, mode):
    return _ArStepFn.apply(cur, v, params, ld_in, col, mode)


class _ArqsStepFn(Function):
    """One step of ARQS's sequential loops (arqs.py:53-76 / :93-116): column `col` of `cur` is replaced by the public
    [0,1] spline of v[:, col] under the [B, 3K-1] parameter block `params`; the float32 log-det vector accumulates."""

    @staticmethod
    def forward(ctx, cur, v, params, ld_in, col, K, inverse, mins):
        cur, v, params = _c(cur), _c(v), _c(params)
        B, D = v.shape
        out = torch.empty_like(v)
        ld = torch.empty(B, dtype=torch.float32, device=v.device)
        call("nf_arqs_step_forward", ptr(cur), ptr(v), ptr(params), params.shape[1], ptr(None if ld_in is None else _c(ld_in)),
             ptr(out), ptr(ld), B, D, col, K, int(inverse), mins[0], mins[1], mins[2], L.dtype_code(v), stream())
        ctx.cfg = (col, K, inverse, mins, ld_in is not None)
        ctx.save_for_backward(v, params)
        return out, ld

    @staticmethod
    @once_differentiable
    def backward(ctx, gout, gld):
        v, params = ctx.saved_tensors
        col, K, inverse, mins, has_ld = ctx.cfg
        B, D = v.shape
        gcur, gv, gp = torch.empty_like(v), torch.empty_like(v), torch.empty_like(params)
        gld = _c(gld.to(torch.float32))
        call("nf_arqs_step_backward", ptr(v), ptr(params), params.shape[1], ptr(_c(gout)), ptr(gld), ptr(gcur), ptr(gv),
             ptr(gp), B, D, col, K, int(inverse), mins[0], mins[1], mins[2], L.dtype_code(v), stream())
        return gcur, gv, gp, (gld if has_ld else None), None, None, None, None


def arqs_step(cur, v, params, ld_in, col, K, inverse, mins=(1e-3, 1e-3, 1e-3)):
    return _ArqsStepFn.apply(cur, v, params, ld_in, col, K, bool(inverse), tuple(float(m) for m in mins))


class _ArFinishFn(Function):
    @staticmethod
    def forward(ctx, cur, v, ld_sum, mode):
        cur, v, ld_sum = _c(cur), _c(v), _c(ld_sum)
        B, D = v.shape
        out = torch.empty_like(v)
        ld = torch.empty_like(ld_sum)
        call("nf_ar_finish_forward", ptr(cur), ptr(v), ptr(ld_sum), ptr(out), ptr(ld), B, D, mode, L.dtype_code(v),
             stream())
        ctx.mode = mode
        ctx.save_for_backward(cur, ld_sum)
        return out, ld

    @staticmethod
    @once_differentiable
    def backward(ctx, gout, gld):
        cur, ld_sum = ctx.saved_tensors
        B, D = cur.shape
        gcur, gv, gls = torch.empty_like(cur), torch.empty_like(cur), torch.empty_like(ld_sum)
        call("nf_ar_finish_backward", ptr(cur), ptr(ld_sum), ptr(_c(gout)), ptr(_c(gld)), ptr(gcur), ptr(gv), ptr(gls),
             B, D, ctx.mode, L.dtype_code(cur), stream())
        return gcur, gv, gls, None


def ar_finish(cur, v, ld_sum, mode):
    return _ArFinishFn.apply(cur, v, ld_sum, mode)


class _StdNormalLogProbFn(Function):
    @staticmethod
    def forward(ctx, z, ld):
        z = _c(z)
        B, D = z.shape
        lp = torch.empty(B, dtype=z.dtype, device=z.device)
        call("nf_std_normal_log_prob_forward", ptr(z), ptr(None if ld is None else _c(ld)), ptr(lp), B, D,
             L.dtype_code(z), stream())
        ctx.has_ld = ld is not None
        ctx.save_for_backward(z)
        return lp

    @staticmethod
    @once_differentiable
    def backward(ctx, glp):
        z, = ctx.saved_tensors
        B, D = z.shape
        glp = _c(glp)
        gz = torch.empty_like(z)
        call("nf_std_normal_log_prob_backward", ptr(z), ptr(glp), ptr(gz), B, D, L.dtype_code(z), stream())
        return gz, (glp if ctx.has_ld else None)


def std_normal_log_prob(z, log_det=None):
    """log N(z; 0, I) + log_det per row: the Flow.log_prob head (flow.py:56-73) for a standard-normal base."""
    if log_det is not None and log_det.dtype != z.dtype:
        log_det = log_det.to(z.dtype)
    return _StdNormalLogProbFn.apply(z, log_det)


def std_normal_draw(seed, offset, B, D, dtype, device):
    """z [B, D] ~ N(0, I) from the counter-based stream of csrc/nf_rng.cuh at (seed, offset): the same bits as the
    in-kernel draw of the fused stacks.  float64 widens the float32 normals.
    seed may instead be the int64 [4] state tensor of a DeviceGenerator (offset None): the kernel reads the key from it
    and advances it by 4 in the same launch (nf_std_normal_draw_state), so the call can be captured in a CUDA graph."""
    z = torch.empty((B, D), dtype=dtype, device=device)
    if isinstance(seed, torch.Tensor):
        call("nf_std_normal_draw_state", ptr(seed), ptr(z), B, D, L.dtype_code(z), stream())
    else:
        call("nf_std_normal_draw", seed, offset, ptr(z), B, D, L.dtype_code(z), stream())
    return z


def _draw_key(draw):
    """The (seed, offset) argument pair of std_normal_draw for a `draw`: a host key (seed, offset) or a state tensor."""
    return (draw, None) if isinstance(draw, torch.Tensor) else draw


class _StdNormalLogQFn(Function):
    @staticmethod
    def forward(ctx, z, ld):
        z, ld = _c(z), _c(ld)
        B, D = z.shape
        lq = torch.empty(B, dtype=z.dtype, device=z.device)
        call("nf_std_normal_log_q_forward", ptr(z), ptr(ld), ptr(lq), B, D, L.dtype_code(z), stream())
        ctx.save_for_backward(z)
        return lq

    @staticmethod
    @once_differentiable
    def backward(ctx, glq):
        z, = ctx.saved_tensors
        B, D = z.shape
        gz = torch.empty_like(z) if ctx.needs_input_grad[0] else None
        gld = torch.empty(B, dtype=z.dtype, device=z.device) if ctx.needs_input_grad[1] else None
        call("nf_std_normal_log_q_backward", ptr(z), ptr(_c(glq)), ptr(gz), ptr(gld), B, D, L.dtype_code(z), stream())
        return gz, gld


def std_normal_log_q(z, log_det):
    """log N(z; 0, I) - log_det per row: the sample_and_log_prob head for a standard-normal base."""
    if log_det.dtype != z.dtype:
        log_det = log_det.to(z.dtype)
    return _StdNormalLogQFn.apply(z, log_det)


# --------------------------------------------------------------------------------------------
# fused inference launches
# --------------------------------------------------------------------------------------------
STACK_INVERSE, STACK_LOG_PROB_HEAD, STACK_SKIP_Y, STACK_SAMPLE_LOG_Q = 1, 2, 4, 8      # csrc/stack_small.cuh


def _stack_flags(inverse, head):
    """Flag word of the fused stack entry points.  head=True: the per-row output is the Flow.log_prob value
    log N(z; 0, I) + log_det (flow.py:56-73) computed in the last layer's epilogue, and z is not stored."""
    return (STACK_INVERSE if inverse else 0) | ((STACK_LOG_PROB_HEAD | STACK_SKIP_Y) if head else 0)


def stack(entry, packed, hdr_host, x, inverse, head=False, sample=None, mode=(), context=None):
    """One launch of the fused-stack entry point `entry` (nf_spline_stack, nf_spline_stack_tc, nf_coupling_stack,
    nf_coupling_stack_tc; nf_made_stack_tc with mode=(mode,)) on the (packed, hdr_host) pair of its packer; returns None if
    the configuration is unsupported.  sample=(seed, offset): the `_sample` entry point instead -- x is the output buffer of the rows, drawn from N(0, I) in the kernel and run forward, and the
    per-row output is log N(z) - log_det (sample_and_log_prob).  sample=<DeviceGenerator state tensor>: `_sample_state`,
    the same draw with the key read from, and advanced in, device memory (a refused call leaves the state as it was).
    context=(c, div) (nf_spline_stack_ctx_tc, nf_coupling_stack_ctx_tc): the float32 [rows, C] context, row r of the
    batch reading row r // div."""
    x = _c(x)
    B = x.shape[0]
    ld = torch.empty(B, dtype=x.dtype, device=x.device)
    hdr, nbytes = hdr_host.ctypes.data, packed.numel() * 4
    cargs = () if context is None else (ptr(_c(context[0])), context[0].shape[0], int(context[1]))
    if isinstance(sample, torch.Tensor):
        ok = L.try_call(entry + "_sample_state", ptr(packed), hdr, nbytes, *mode, *cargs, ptr(sample), ptr(x), ptr(ld), B,
                        stream())
        return (x, ld) if ok else None
    if sample is not None:
        ok = L.try_call(entry + "_sample", ptr(packed), hdr, nbytes, *mode, *cargs, sample[0], sample[1], ptr(x), ptr(ld),
                        B, stream())
        return (x, ld) if ok else None
    y = None if head else torch.empty_like(x)
    ok = L.try_call(entry + "_forward", ptr(packed), hdr, nbytes, ptr(x), *cargs, ptr(y), ptr(ld), B,
                    _stack_flags(inverse, head), *mode, stream())
    return (y, ld) if ok else None


MADE_CHAIN_BF16 = False          # set by nfb200.set_gemm_precision("bf16"): the fused bf16 chain kernel for MAF / IAF


def made_chain_bf16(v, folded, mode, head=False, draw=None):
    """Whole parallel direction in ONE launch on bf16 tensor cores (csrc/made_chain_bf16.cu); None when the shape is
    outside the kernel's envelope (data_dim <= 64 and a multiple of 4, hidden_dim a multiple of 128 and <= 512).
    head=True: returns (None, log N(z;0,I) + log_det) without storing z.
    draw=(seed, offset) or a DeviceGenerator state tensor (IAF.forward): v only gives the shape; the input is the N(0, I)
    draw of std_normal_draw, made once the shape is known to fit, and the result is (x, log N(z) - log_det).  Should the
    chain refuse after the draw, the drawn z [B, D] is returned instead of None: the caller must go on with that z, since
    drawing again would advance a device-resident state a second time."""
    from . import packing
    if v.dtype != torch.float32:
        return None
    if folded.bf16 is None:
        folded.bf16 = packing.made_bf16_pack(folded)
    pk = folded.bf16
    if pk is False:
        return None
    B, D = v.shape
    flags = (STACK_LOG_PROB_HEAD | STACK_SKIP_Y) if head else 0
    if draw is not None:
        v = std_normal_draw(*_draw_key(draw), B, D, v.dtype, v.device)
        flags = STACK_SAMPLE_LOG_Q
    v = _c(v)
    out = None if head else torch.empty_like(v)
    ld = torch.empty(B, dtype=v.dtype, device=v.device)
    ok = L.try_call("nf_made_chain_bf16_forward", ptr(v), ptr(pk.w[0]), ptr(pk.w[1]), ptr(pk.w[2]), ptr(pk.w[3]),
                    ptr(pk.b[0]), ptr(pk.b[1]), ptr(pk.b[2]), ptr(pk.b[3]), pk.kext16_host.ctypes.data, ptr(out), ptr(ld),
                    B, D, folded.H, mode, flags, stream())
    if ok:
        return out, ld
    return v if draw is not None else None


def made_params_tc(v, folded):
    """Raw MADE outputs [B, 2D] = [mu | alpha] from the folded weights, layer by layer: the tensor-core GEMM where the
    shape has a TMA row pitch and a tile's worth of columns, the streaming FP32 kernels of nf_gemm for the skinny first /
    last layer of a low-dimensional MADE."""
    h = v
    for i in range(4):
        hi, lo = folded.w_split[i]
        N_, K_ = folded.w[i].shape
        y = None
        if K_ % 4 == 0 and K_ >= 16 and N_ >= 16:
            y = linear_tc(h, hi, lo, folded.b[i], relu=(i < 3), k_extent=(folded.kext[i - 1] if i > 0 else None))
        h = y if y is not None else linear_raw(h, folded.w[i], folded.b[i], relu=(i < 3))
    return h


AR_TWO_DIM_CHAIN_MIN_ROWS = 16384


def ar_sequential_two_dim(v, folded, mode):
    """MAF.forward / IAF.inverse for data_dim == 2 at large batch: the reference's loop (masked_autoregressive_flow.py:
    55-67 / inverse_autoregressive_flow.py:76-91) with its two conditioner evaluations -- the first one, on zeros, yields
    exactly the output biases for dim 0 (its masked output rows are all zero), the second one runs as the tensor-core
    chain of the parallel direction.  6 x MAF(2, 64) sampling at 2^20 rows: 5.3 -> 3.3 ms; 8 x MAF(2, 128): 20 -> 9 ms
    (the incremental one-launch kernel keeps a [D + 3H][32] tile per warp: few warps per SM at hidden 128)."""
    B, D = v.shape
    v = _c(v)
    cur = torch.zeros_like(v)
    p0 = folded.b[3].to(v.dtype).unsqueeze(0).expand(B, 2 * D).contiguous()      # made(0)[:, (0, D)] == (b_mu0, b_alpha0)
    cur, ld = ar_step(cur, v, p0, None, 0, mode)
    cur, ld = ar_step(cur, v, made_params_tc(cur, folded), ld, 1, mode)
    return ar_finish(cur, v, ld, mode)


def made_affine(v, folded, mode):
    """MADE chain + MAF.inverse / IAF.forward.  folded: packing.FoldedMade.  float32: four tcgen05 GEMMs (3xTF32,
    bias/ReLU epilogues, masked-out K tiles skipped) + the transform kernel; float64 or tiny shapes: FP32/FP64-pipe chain.
    In the bf16 mode (set_gemm_precision("bf16")) the whole direction is one fused launch."""
    v = _c(v)
    B, D = v.shape
    H = folded.H
    if MADE_CHAIN_BF16 and USE_TENSOR_CORE_GEMM and B >= 128:
        res = made_chain_bf16(v, folded, mode)
        if res is not None:
            return res
    if USE_TENSOR_CORE_GEMM and folded.w_split is not None and v.dtype == torch.float32 and B >= 128:
        # layer by layer: the tensor-core GEMM where the shape has a TMA row pitch and a tile's worth of columns, the
        # streaming FP32 kernels of nf_gemm for the skinny first / last layer of a low-dimensional MADE (MADE(2, 64):
        # K = 2 in, 4 out) -- refusing the whole chain for them sent the two 64 x 64 layers to the FP32-pipe GEMM too
        h = made_params_tc(v, folded)
        out = torch.empty_like(v)
        ld = torch.empty(B, dtype=v.dtype, device=v.device)
        call("nf_affine_ar_forward", ptr(v), ptr(h), ptr(out), ptr(ld), B, D, mode, L.dtype_code(v), stream())
        return out, ld
    ws = torch.empty(2 * B * max(H, 2 * D), dtype=v.dtype, device=v.device)
    out = torch.empty_like(v)
    ld = torch.empty(B, dtype=v.dtype, device=v.device)
    w, b = folded.w, folded.b
    call("nf_made_affine_forward", ptr(v), ptr(w[0]), ptr(b[0]), ptr(w[1]), ptr(b[1]), ptr(w[2]), ptr(b[2]),
         ptr(w[3]), ptr(b[3]), ptr(folded.kext[0]), ptr(folded.kext[1]), ptr(folded.kext[2]), ptr(ws), ptr(out),
         ptr(ld), B, D, H, mode, L.dtype_code(v), stream())
    return out, ld


AR_BLOCK_DEGREES = 8


def _ptr_array(tensors):
    import ctypes
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def ar_sequential_blocked(v, folded, mode):
    """MAF.forward / IAF.inverse, blocked: previous-block contributions on tcgen05, in-block steps in ar_blocked.cu.
    Returns None when the configuration is not taken (no TF32 splits, D not a multiple of 4)."""
    if folded.w_split is None or v.dtype != torch.float32 or folded.D % 4 or AR_BLOCK_DEGREES % 4:
        return None
    pk = folded.blocked
    if pk is None or (pk is not False and pk.block_degrees != AR_BLOCK_DEGREES):
        from . import packing
        pk = packing.blocked_made_pack(folded, AR_BLOCK_DEGREES) or False
        folded.blocked = pk
    if pk is False:
        return None
    v = _c(v)
    B, D = v.shape
    H = pk.H
    nws = L.lib().nf_ar_blocked_workspace_floats(B, D, H)
    ws = torch.empty(nws, dtype=torch.float32, device=v.device)
    out = torch.empty_like(v)
    ld = torch.empty(B, dtype=v.dtype, device=v.device)
    ok = L.try_call("nf_ar_blocked_forward", ptr(v), _ptr_array(pk.w), _ptr_array(pk.w_hi), _ptr_array(pk.w_lo),
                    _ptr_array(pk.b), ptr(pk.gstart), pk.gstart_host.ctypes.data,
                    ptr(ws), ptr(out), ptr(ld), B, D, H, mode, AR_BLOCK_DEGREES, stream())
    return (out, ld) if ok else None


def ar_sequential(v, folded, mode):
    """MAF.forward / IAF.inverse: blocked tensor-core evaluation for wide conditioners, otherwise the one-launch
    incremental kernel; returns None when unsupported (H too large for it, fp64)."""
    if v.dtype != torch.float32:
        return None
    if USE_TENSOR_CORE_GEMM and folded.D == 2 and folded.w_split is not None and v.shape[0] >= AR_TWO_DIM_CHAIN_MIN_ROWS:
        return ar_sequential_two_dim(v, folded, mode)
    if USE_TENSOR_CORE_GEMM and folded.H >= 128 and folded.D >= 2 * AR_BLOCK_DEGREES and v.shape[0] >= 1024:
        res = ar_sequential_blocked(v, folded, mode)
        if res is not None:
            return res
    v = _c(v)
    B, D = v.shape
    out = torch.empty_like(v)
    ld = torch.empty(B, dtype=v.dtype, device=v.device)
    w, b = folded.w, folded.b
    ok = L.try_call("nf_ar_sequential_forward", ptr(v), ptr(w[0]), ptr(b[0]), ptr(w[1]), ptr(b[1]), ptr(w[2]),
                    ptr(b[2]), ptr(w[3]), ptr(b[3]), ptr(folded.gstart), ptr(out), ptr(ld), B, D, folded.H, mode,
                    stream())
    return (out, ld) if ok else None
