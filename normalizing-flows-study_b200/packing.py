"""Host-side weight packing for the fused kernels (derived caches of the nn.Module parameters).

The modules keep the reference's parameter/buffer names and shapes (state_dict compatible, SURVEY A.2);
the kernels want other layouts: transposed / chunked / zero-padded conditioner weights with eval-mode
BatchNorm folded in (stack_small.cuh), and mask-folded, degree-sorted MADE weights.  Packs are rebuilt
whenever a parameter's version counter or storage changes.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional

import numpy as np
import torch

from . import _lib as L

MAGIC_SPLINE = 0x4E465331
MAGIC_AFFINE = 0x4E464131
MAGIC_SPLINE_TC = 0x4E465332
MAGIC_AFFINE_TC = 0x4E464132
MAGIC_MADE_TC = 0x4E464D32
MAGIC_SPLINE_CTX_TC = 0x4E464332
MAGIC_AFFINE_CTX_TC = 0x4E464432
CTX_MAX = 8                     # context columns of the conditional tcgen05 layouts ('NFC2', 'NFD2'; csrc/stack_small.cuh)
HDR, LAYER_HDR, DMAX = 16, 80, 8


_generation = 0


def invalidate_caches() -> None:
    """Drop every derived weight layout (fused stack packs, folded MADE weights, TF32 splits, mask plans) at its next
    use.  Needed after updates that autograd's version counters cannot see: a CUDA-graph replay that contains the
    optimizer step (graphs.GraphedTrainStep calls this itself), `p.data.<op>_()` writes (the reference's EMA code,
    consistency_flow.py:28), raw-pointer writes from another library."""
    global _generation
    _generation += 1


def _version_of(t):
    # inference tensors (created under torch.inference_mode) do not track a version counter
    return -1 if t.is_inference() else t._version


def tensors_key(tensors, extra=()):
    """Cache key that changes when any tensor is modified in place, re-assigned or moved, or when
    invalidate_caches() was called.  `extra`: plain hashable components (dtypes, devices, flags)."""
    return (_generation, tuple(extra)) + tuple(
        (t.data_ptr(), _version_of(t), t.device.index, t.dtype) for t in tensors if t is not None)


def _np(t, dtype=np.float64):
    return t.detach().to("cpu").numpy().astype(dtype)


def _hp(H):
    return 64 if H <= 64 else 128


def _w1s(D):
    return 4 if D <= 3 else 12


def _net_words(HP, W1S, NO):
    return HP * W1S + HP * HP + HP + NO * HP + NO


def _pack_net(W1, b1, W2, b2, W3, b3, out_rows, D, H, HP, W1S, NO):
    """One conditioner block: W1k | W2t | b2 | W3c | b3 (float64 numpy in, float32 words out)."""
    w1k = np.zeros((HP, W1S))
    w1k[:H, :D] = W1
    w1k[:H, W1S - 1] = b1
    w2t = np.zeros((HP, HP))
    w2t[:H, :H] = W2.T
    b2p = np.zeros(HP)
    b2p[:H] = b2
    w3 = np.zeros((NO, HP))
    b3p = np.zeros(NO)
    n = len(out_rows)
    w3[:n, :H] = W3[out_rows]
    b3p[:n] = b3[out_rows]
    w3c = w3.reshape(NO // 4, 4, HP).transpose(0, 2, 1)          # [c][j][q]
    return np.concatenate([w1k.ravel(), w2t.ravel(), b2p, w3c.ravel(), b3p]).astype(np.float32)


def _layer_header(mask, tdims, rescale, bn):
    """80-word per-layer header; ints are stored as raw int32 bit patterns."""
    h = np.zeros(LAYER_HDR, dtype=np.float32)
    hi = h.view(np.int32)
    D = len(mask)
    h[0:D] = mask
    hi[8:8 + len(tdims)] = tdims
    hi[16] = len(tdims)
    if rescale is not None:
        hi[17] = 1
        h[24:24 + D], h[32:32 + D], h[40:40 + D] = rescale
    if bn is not None:
        hi[18] = 1
        mean, sd, gamma, beta, bn_ld = bn
        h[19] = bn_ld
        h[48:48 + D], h[56:56 + D], h[64:64 + D], h[72:72 + D] = mean, sd, gamma, beta
    else:
        h[56:64] = 1.0
        h[64:72] = 1.0
    return h


def _bn_between_consts(bn: torch.nn.BatchNorm1d):
    """Between-layer BatchNorm as an affine on running stats (normalizing_flow_model.py:67-128), computed with the
    same float32 torch expressions as the reference so the constants match bit for bit."""
    with torch.no_grad():
        sd = torch.sqrt(bn.running_var.float() + bn.eps)
        ld = (torch.log(torch.abs(bn.weight.float())) - 0.5 * torch.log(bn.running_var.float() + bn.eps)).sum()
    return (_np(bn.running_mean, np.float32), _np(sd, np.float32), _np(bn.weight, np.float32),
            _np(bn.bias, np.float32), float(ld))


def _rescale(layer, D):
    """(a, lo, c) of the data_min / data_max rescale in float64 (spline_coupling_layer.py:101-102), or None."""
    if layer.data_min is None or layer.data_max is None:
        return None
    lo = np.broadcast_to(_np(torch.as_tensor(layer.data_min)), (D,)).astype(np.float64)
    hi = np.broadcast_to(_np(torch.as_tensor(layer.data_max)), (D,)).astype(np.float64)
    return (2 * layer.bound) / (hi - lo), lo, (hi - lo) / (2 * layer.bound)


def _rescale_arrays(layer, D):
    r = _rescale(layer, D)
    return None if r is None else tuple(a.astype(np.float32) for a in r)


def rescale_tensors(layer, D, dtype, device):
    r = _rescale(layer, D)
    return None if r is None else tuple(torch.tensor(a, dtype=dtype, device=device) for a in r)


def _stack_header(magic, D, H, w3, K, L_, W1S, NO, stride, bns, spline=None, scales=False):
    """The 16 header words (csrc/stack_small.cuh).  w3: HP in the FP32-pipe layouts, nets per layer in the tcgen05 ones.
    spline: the layer whose bound, minimums and 1 - min * K fill words 10-15; zeros otherwise, except that
    scales=True stores 1 - 0 * K = 1 in words 14 and 15 (the FP32-pipe affine layout)."""
    h = np.zeros(HDR, dtype=np.float32)
    h.view(np.int32)[0:10] = [magic, D, H, w3, K, L_, W1S, NO, stride, int(bns is not None)]
    bound, mins = (spline.bound, (spline.min_bin_width, spline.min_bin_height, spline.min_derivative)) \
        if spline is not None else (0.0, (0.0, 0.0, 0.0))
    h[10] = bound
    h[11], h[12], h[13] = mins
    if spline is not None or scales:
        h[14] = np.float32(1.0 - mins[0] * K)
        h[15] = np.float32(1.0 - mins[1] * K)
    return h


def _between_bn(bns, i, n_layers):
    """Constants of the BatchNorm between layer i and i + 1; None after the last layer or without BatchNorm."""
    return _bn_between_consts(bns[i]) if (bns is not None and i < n_layers - 1) else None


def _finish(words, n_words, device):
    """(packed buffer on `device`, host copy of its header as int32 words)."""
    flat = np.concatenate(words).astype(np.float32, copy=False)
    assert flat.size == n_words, (flat.size, n_words)
    return torch.from_numpy(flat).to(device), flat[:HDR].copy().view(np.int32)


def _spline_key(l):
    return (l.data_dim, l.param_net[0].out_features, l.num_bins, l.bound, l.min_bin_width, l.min_bin_height,
            l.min_derivative, l.context_dim)


def _coupling_key(l):
    return (l.data_dim, l.s_net[0].out_features, l.context_dim)


def _alike(layers, key):
    """One fused launch takes one shape: every layer must have the first one's key."""
    k0 = key(layers[0])
    return all(key(l) == k0 for l in layers)


def pack_spline_stack(layers, bns: Optional[List[torch.nn.BatchNorm1d]]):
    """layers: SplineCouplingLayer modules (same D/H/K/bound/minimums).  Returns (packed_device, hdr_host) or None
    when the stack cannot use the fused kernel."""
    l0 = layers[0]
    D, K = l0.data_dim, l0.num_bins
    H = l0.param_net[0].out_features
    if not _alike(layers, _spline_key) or l0.context_dim:
        return None
    if D > DMAX or H > 128 or K < 2 or K > 16 or l0.param_net[0].weight.dtype != torch.float32:
        return None
    if L.lib().nf_spline_stack_packed_floats(D, H, K, len(layers)) < 0:
        return None
    P = 3 * K - 1
    HP, W1S = _hp(H), _w1s(D)
    masks = [_np(l.mask) for l in layers]
    max_dt = max(int((m == 0).sum()) for m in masks)
    NO = 4 * ((max_dt * P + 3) // 4)
    if NO == 0:
        return None
    stride = LAYER_HDR + _net_words(HP, W1S, NO)
    words = [_stack_header(MAGIC_SPLINE, D, H, HP, K, len(layers), W1S, NO, stride, bns, spline=l0)]
    for i, (l, m) in enumerate(zip(layers, masks)):
        tdims = [d for d in range(D) if m[d] == 0]
        words.append(_layer_header(m.astype(np.float32), tdims, _rescale_arrays(l, D), _between_bn(bns, i, len(layers))))
        net = l.param_net
        rows = [d * P + p for d in tdims for p in range(P)]
        words.append(_pack_net(_np(net[0].weight), _np(net[0].bias), _np(net[2].weight), _np(net[2].bias),
                               _np(net[4].weight), _np(net[4].bias), rows, D, H, HP, W1S, NO))
    return _finish(words, HDR + len(layers) * stride, l0.param_net[0].weight.device)


def _fold_bn(W, b, bn: torch.nn.BatchNorm1d):
    """Linear followed by eval-mode BatchNorm1d == Linear with scaled rows (coupling_layer.py:19-24)."""
    s = _np(bn.weight) / np.sqrt(_np(bn.running_var) + bn.eps)
    return W * s[:, None], (b - _np(bn.running_mean)) * s + _np(bn.bias)


def pack_coupling_stack(layers, bns: Optional[List[torch.nn.BatchNorm1d]]):
    """layers: CouplingLayer modules in eval mode."""
    l0 = layers[0]
    D = l0.data_dim
    H = l0.s_net[0].out_features
    if not _alike(layers, _coupling_key) or l0.context_dim:
        return None
    if D > DMAX or H > 128 or l0.s_net[0].weight.dtype != torch.float32:
        return None
    HP, W1S = _hp(H), _w1s(D)
    NO = 4 if D <= 3 else 8
    stride = LAYER_HDR + 2 * _net_words(HP, W1S, NO)
    words = [_stack_header(MAGIC_AFFINE, D, H, HP, 0, len(layers), W1S, NO, stride, bns, scales=True)]
    for i, l in enumerate(layers):
        m = _np(l.mask)
        words.append(_layer_header(m.astype(np.float32), [d for d in range(D) if m[d] == 0], None,
                                   _between_bn(bns, i, len(layers))))
        for net in (l.s_net, l.b_net):
            W1, b1 = _fold_bn(_np(net[0].weight), _np(net[0].bias), net[1])
            W2, b2 = _fold_bn(_np(net[3].weight), _np(net[3].bias), net[4])
            words.append(_pack_net(W1, b1, W2, b2, _np(net[6].weight), _np(net[6].bias), list(range(D)), D, H, HP,
                                   W1S, NO))
    return _finish(words, HDR + len(layers) * stride, l0.s_net[0].weight.device)


@dataclass
class FoldedMade:
    """Mask-folded MADE weights with hidden units sorted by degree (made.py:25-79)."""
    D: int
    H: int
    w: list
    b: list
    kext: list          # per-layer int32 k-extent arrays for layers 1..3 (None entries allowed)
    gstart: torch.Tensor
    w_split: Optional[list] = None      # [(hi, lo)] x 4: 3xTF32 operands of the tensor-core GEMM (float32 only)
    gstart_host: Optional[np.ndarray] = None
    bf16: Optional[object] = None       # made_bf16_pack(self), built on first use of the bf16 fused chain (False: unsupported)
    blocked: Optional[object] = None    # blocked_made_pack(self, .), built on first use of the blocked sequential direction


def fold_made(made) -> Optional[FoldedMade]:
    """Eval-mode BatchNorm (use_batch_norm=True, made.py:93-108) is a per-unit affine on running statistics: it is
    folded into the rows of the preceding masked linear, which leaves the mask's zero structure untouched.  (Callers
    take the layered route in train mode, where the statistics come from the batch.)"""
    if made.output_dim_multiplier != 2:
        return None
    lin = [m for m in made.net if hasattr(m, "mask")]
    bns = [m for m in made.net if isinstance(m, torch.nn.BatchNorm1d)]
    if made.use_batch_norm and (len(bns) != 3 or any(bn.running_mean is None for bn in bns)):
        return None
    D, H = made.input_dim, made.hidden_dim
    deg = np.asarray(made.m[0]).astype(np.int64)
    perm = np.argsort(deg, kind="stable")
    sdeg = deg[perm]
    dev = lin[0].weight.device
    p = torch.as_tensor(perm, device=dev)
    with torch.no_grad():
        eff = [l.weight * l.mask.to(l.weight.dtype) for l in lin]
        bias = [l.bias for l in lin]
        if made.use_batch_norm:
            for i, bn in enumerate(bns):
                sc = bn.weight / torch.sqrt(bn.running_var + bn.eps)
                eff[i] = eff[i] * sc[:, None]
                bias[i] = (bias[i] - bn.running_mean) * sc + bn.bias
        w = [eff[0][p].contiguous(), eff[1][p][:, p].contiguous(), eff[2][p][:, p].contiguous(),
             eff[3][:, p].contiguous()]
        b = [bias[0][p].contiguous(), bias[1][p].contiguous(), bias[2][p].contiguous(),
             bias[3].detach().contiguous()]
    gstart = np.searchsorted(sdeg, np.arange(D + 1), side="left").astype(np.int32)   # #units with degree < g
    # k-extents per 64 output columns
    def hh_ext():
        out = []
        for t in range(0, H, 64):
            last = sdeg[min(t + 63, H - 1)]
            out.append(int(np.searchsorted(sdeg, last, side="right")))
        return torch.tensor(out, dtype=torch.int32, device=dev)

    def out_ext():
        out = []
        for t in range(0, 2 * D, 64):
            cols = np.arange(t, min(t + 64, 2 * D)) % D
            out.append(int(gstart[cols.max()]))
        return torch.tensor(out, dtype=torch.int32, device=dev)

    kext = [hh_ext(), hh_ext(), out_ext()]
    folded = FoldedMade(D, H, w, b, kext, torch.as_tensor(gstart, device=dev))
    folded.gstart_host = np.ascontiguousarray(gstart, dtype=np.int32)
    if w[0].dtype == torch.float32 and w[0].is_cuda:
        from . import ops
        folded.w_split = [ops.split_tf32(t) for t in w]
    return folded


@dataclass
class BlockedMadePack:
    """Operands of nf_ar_blocked_forward (csrc/ar_blocked.cu).  The degree-sorted hidden units are laid out in blocks of
    `block_degrees` consecutive degrees, every block starting at a multiple of 4 units: the gaps are dead units (zero
    weights and biases, so they hold relu(0) = 0 and feed nothing).  H is the padded width; gstart[g] the padded index of
    the first unit of degree >= g (dead units count with the degree in front of them).  w / b: fp32 operands of the
    in-block kernel (output layer as [mu rows | alpha rows], like made.py:136-140); w_hi / w_lo: 3xTF32 operands of the
    slice products, the output layer's rows INTERLEAVED (row 2g = mu_g, row 2g+1 = alpha_g) to match the [B, D, 2]
    layout of the pushed output pre-activations."""
    block_degrees: int
    H: int
    w: list
    b: list
    w_hi: list
    w_lo: list
    gstart: torch.Tensor
    gstart_host: np.ndarray


def blocked_layout(gstart: np.ndarray, block_degrees: int, align: int = 4):
    """(pos, pgstart, Hp): padded index of every sorted unit, padded degree boundaries, padded width.  Blocks always
    start at a multiple of `align`; when it costs at most 10 % more units every DEGREE does (the in-block kernels then
    evaluate a degree's units in exact 4-unit chunks / whole 8-unit tensor-core tiles instead of chunks straddling its
    neighbours).  In that per-degree layout every BLOCK is also padded to a multiple of 2 * align units, the extra `align`
    dead units going to a degree whose padded count is an odd multiple of `align` (it occupies the same number of 8-unit
    tiles afterwards): the slice GEMMs of the blocked route then never see a contraction length K = 4 (mod 32) -- a TMA
    box with 4 live columns out of 32 costs ~25 us per product at 262 144 rows (K = 64: 54 us, K = 68: 79 us,
    profiles/r02az_slice_gemm.jsonl) -- and every output slice starts 32-byte aligned (256-bit row stores)."""
    D = len(gstart) - 1
    H = int(gstart[D])
    counts = np.diff(gstart).astype(np.int64)
    per_degree = int(((counts + align - 1) // align * align).sum()) <= 1.10 * H
    padded = counts.copy()
    if per_degree:
        padded = (counts + align - 1) // align * align
        for g0 in range(0, D, block_degrees):
            g1 = min(g0 + block_degrees, D)
            if int(padded[g0:g1].sum()) % (2 * align) == align:
                odd = [g for g in range(g0, g1) if padded[g] % (2 * align) == align]
                padded[odd[-1]] += align
    pos = np.zeros(H, dtype=np.int64)
    pgstart = np.zeros(D + 1, dtype=np.int32)
    at = 0
    for g in range(D):
        if g % block_degrees == 0 and not per_degree:
            at = (at + align - 1) // align * align
        pgstart[g] = at
        pos[gstart[g]:gstart[g + 1]] = at + np.arange(counts[g])
        at += int(padded[g])
    at = (at + align - 1) // align * align
    pgstart[D] = at
    # a degree's dead units are the gap up to the next degree's start
    return pos, pgstart, max(at, align)


def blocked_made_pack(folded: "FoldedMade", block_degrees: int) -> Optional[BlockedMadePack]:
    w, b = folded.w, folded.b
    if w[0].dtype != torch.float32 or not w[0].is_cuda or folded.gstart_host is None:
        return None
    from . import ops
    D, H = folded.D, folded.H
    pos, pgstart, Hp = blocked_layout(folded.gstart_host, block_degrees)
    dev = w[0].device
    p = torch.as_tensor(pos, device=dev)
    with torch.no_grad():
        w0 = torch.zeros(Hp, D, device=dev); w0[p] = w[0]
        w1 = torch.zeros(Hp, Hp, device=dev); w1[p[:, None], p[None, :]] = w[1]
        w2 = torch.zeros(Hp, Hp, device=dev); w2[p[:, None], p[None, :]] = w[2]
        w3 = torch.zeros(2 * D, Hp, device=dev); w3[:, p] = w[3]
        bb = []
        for i in range(3):
            t = torch.zeros(Hp, device=dev); t[p] = b[i]; bb.append(t)
        bb.append(b[3].contiguous())
        w3i = w3.reshape(2, D, Hp).transpose(0, 1).reshape(2 * D, Hp).contiguous()
        splits = [ops.split_tf32(t) for t in (w0, w1, w2, w3i)]
    return BlockedMadePack(block_degrees, Hp, [w0, w1, w2, w3], bb, [s_[0] for s_ in splits], [s_[1] for s_ in splits],
                           torch.as_tensor(pgstart, device=dev), np.ascontiguousarray(pgstart, dtype=np.int32))


@dataclass
class MadeBf16Pack:
    """Operands of nf_made_chain_bf16_forward (csrc/made_chain_bf16.cu): bf16 weights with the input layer's K padded to
    64 and the output layer laid out as [mu rows 0..D-1 | zero | alpha rows 64..64+D-1 | zero] (128 rows), fp32 biases
    (output bias padded the same way), and per (layer, 128-column block) the number of 16-wide k-steps that hold a
    non-zero weight (block lower-triangular masks: everything beyond is exactly zero and is neither loaded nor multiplied)."""
    w: list
    b: list
    kext16_host: np.ndarray


def made_bf16_pack(folded: FoldedMade):
    D, H = folded.D, folded.H
    if D > 64 or D % 4 or H % 128 or H > 512 or folded.w[0].dtype != torch.float32 or not folded.w[0].is_cuda:
        return False
    dev = folded.w[0].device
    bf = torch.bfloat16
    with torch.no_grad():
        w0 = torch.zeros(H, 64, dtype=bf, device=dev)
        w0[:, :D] = folded.w[0].to(bf)
        w1, w2 = folded.w[1].to(bf).contiguous(), folded.w[2].to(bf).contiguous()
        w3 = torch.zeros(128, H, dtype=bf, device=dev)
        w3[:D] = folded.w[3][:D].to(bf)
        w3[64:64 + D] = folded.w[3][D:].to(bf)
        b3 = torch.zeros(128, dtype=torch.float32, device=dev)
        b3[:D] = folded.b[3][:D]
        b3[64:64 + D] = folded.b[3][D:]
        ws = [w0, w1, w2, w3]
        # last non-zero column (+1) of every 128-row block, in 16-wide k-steps
        lasts = []
        for wm in ws:
            nz = (wm != 0)
            K = wm.shape[1]
            last = torch.where(nz, torch.arange(1, K + 1, device=dev)[None, :], 0).amax(dim=1)        # per row
            pad = (-last.numel()) % 128
            if pad:
                last = torch.cat([last, last.new_zeros(pad)])
            lasts.append(last.view(-1, 128).amax(dim=1))
        host = [t.cpu().numpy() for t in lasts]
    kext = np.zeros((4, 4), dtype=np.int32)
    for l, v in enumerate(host):
        n = min(4, len(v))
        kext[l, :n] = (v[:n] + 15) // 16
    return MadeBf16Pack(ws, [folded.b[0].contiguous(), folded.b[1].contiguous(), folded.b[2].contiguous(), b3],
                        np.ascontiguousarray(kext.reshape(-1)))


# ------------------------------------------------------------------------------------------------
# tensor-core operand images (csrc/tc_common.cuh)
# ------------------------------------------------------------------------------------------------
def _round_tf32(w: np.ndarray) -> np.ndarray:
    bits = np.ascontiguousarray(w, dtype=np.float32).view(np.uint32)
    return ((bits + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def split_tf32(w: np.ndarray):
    """w ~= hi + lo: hi = w rounded to the nearest TF32, lo = (w - hi) rounded to the nearest TF32 (mirrors
    tc::split_tf32_weight; |w - hi - lo| <= 2^-24 |w|)."""
    w = np.ascontiguousarray(w, dtype=np.float32)
    hi = _round_tf32(w)
    return hi, _round_tf32((w - hi).astype(np.float32))


def umma_sw128_image(w: np.ndarray) -> np.ndarray:
    """[rows, K] fp32 (rows % 8 == 0, K % 32 == 0) -> flat float32 array in the UMMA K-major SWIZZLE_128B layout:
    K atoms of 32 floats; inside an atom block row n sits at (n/8)*1024 + (n%8)*128 bytes with its eight 16-byte
    chunks XOR-swizzled by (n%8)."""
    rows, K = w.shape
    assert rows % 8 == 0 and K % 32 == 0
    n = np.arange(rows)[:, None]
    k = np.arange(K)[None, :]
    off = (k >> 5) * (rows * 128) + (n >> 3) * 1024 + (n & 7) * 128 + ((((k & 31) >> 2) ^ (n & 7)) << 4) + (k & 3) * 4
    out = np.zeros(rows * K, dtype=np.float32)
    out[(off // 4).ravel()] = np.ascontiguousarray(w, dtype=np.float32).ravel()
    return out


def umma_sw128_images(w: np.ndarray) -> np.ndarray:
    """hi image followed by lo image (3xTF32 operands)."""
    hi, lo = split_tf32(w)
    return np.concatenate([umma_sw128_image(hi), umma_sw128_image(lo)])


def _pad256(n):
    return (n + 255) & ~255


def _tc_w1k(W1, b1, D, H, W1S, HP=64):
    """W1k[HP][W1S] of the tensor-core layouts: {W1[k][0..D-1], zero pad.., b1[k] at slot W1S-1}; for data_dim <= 3
    (W1S == 4) the units are stored in PAIRS, [w0a w0b | w1a w1b | w2a w2b | ba bb] per pair (a = unit 2p, b = 2p+1), so
    that the kernel's packed-fp32 FMAs (FFMA2) find both units' operands in adjacent registers."""
    w1k = np.zeros((HP, W1S))
    w1k[:H, :D] = W1
    w1k[:H, W1S - 1] = b1
    if W1S == 4:
        w1k = w1k.reshape(HP // 2, 2, 4).transpose(0, 2, 1).reshape(HP, 4)
    return w1k


def _tc_wc(Wc, H, HP=64):
    """Wc[HP/2][CTX_MAX][2] of the conditional layout: context column c of units 2p and 2p+1 at [p][c][0..1], zero beyond
    the C columns of Wc [H, C] and the H units."""
    wc = np.zeros((HP, CTX_MAX))
    wc[:H, :Wc.shape[1]] = Wc
    return wc.reshape(HP // 2, 2, CTX_MAX).transpose(0, 2, 1)


def _tc_net_block(W1, b1, W2, b2, W3rows, b3rows, D, H, W1S, NO3, lead_words, HP=64, Wc=None):
    """One conditioner block of the tensor-core stack layout (csrc/stack_tc.cu: blk_offsets):
    W1k[HP][W1S] (W1S == 4: pair-interleaved, see below) | b2[HP] | b3[NO3] | pad to a 256-word boundary (counting `lead_words` in front) |
    W2 hi image | W2 lo image | W3 hi image | W3 lo image.  W3rows/b3rows: [NO3, H] / [NO3] already in head-column order.
    HP: hidden units padded to 64, or 128 for the affine coupling stack with hidden_dim in (64, 128].
    Wc [H, C]: the context columns of the first Linear (conditional layout), stored by _tc_wc after b3."""
    w1k = _tc_w1k(W1, b1, D, H, W1S, HP)
    b2p = np.zeros(HP)
    b2p[:H] = b2
    parts = [w1k.ravel(), b2p, b3rows] + ([] if Wc is None else [_tc_wc(Wc, H, HP).ravel()])
    small = np.concatenate(parts).astype(np.float32)
    pad = _pad256(lead_words + small.size) - lead_words - small.size
    w2 = np.zeros((HP, HP), dtype=np.float32)
    w2[:H, :H] = W2
    w3 = np.zeros((NO3, HP), dtype=np.float32)
    w3[:, :H] = W3rows
    return np.concatenate([small, np.zeros(pad, dtype=np.float32), umma_sw128_images(w2), umma_sw128_images(w3)])


def pack_made_stack_tc(layers, bns: Optional[List[torch.nn.BatchNorm1d]]):
    """Tensor-core layout of an eval-mode stack of MaskedAutoregressiveFlow / InverseAutoregressiveFlow layers (hidden_dim
    <= 64, data_dim <= 8): per layer `lead (80-word header) | W1k | b2 | b3 | b4[16] | pad | W2 hi/lo | W3 hi/lo | W4 hi/lo`
    from the mask-folded weights (packing.fold_made: eval-mode conditioner BatchNorm folded in; the degree sort of the
    hidden units is a consistent permutation of rows / columns and changes nothing).  Head rows: [mu_0.. | alpha_0..]."""
    l0 = layers[0]
    D = l0.dim
    folded = [l.conditioner.folded() for l in layers]
    if any(f is None for f in folded):
        return None
    H = folded[0].H
    if D > DMAX or H > 64 or any(f.D != D or f.H != H for f in folded) or folded[0].w[0].dtype != torch.float32:
        return None
    nbw = L.lib().nf_made_stack_tc_block_words(D)
    if nbw < 0:
        return None
    W1S, NO = _w1s(D), 16
    words = [_stack_header(MAGIC_MADE_TC, D, H, 1, 0, len(layers), W1S, NO, nbw, bns)]
    for i, f in enumerate(folded):
        lead = _layer_header(np.zeros(D, dtype=np.float32), [], None, _between_bn(bns, i, len(layers)))
        W = [_np(t) for t in f.w]
        b = [_np(t) for t in f.b]
        w1k = _tc_w1k(W[0], b[0], D, H, W1S)
        b2p, b3p, b4p = np.zeros(64), np.zeros(64), np.zeros(NO)
        b2p[:H], b3p[:H], b4p[:2 * D] = b[1], b[2], b[3]
        small = np.concatenate([w1k.ravel(), b2p, b3p, b4p]).astype(np.float32)
        pad = _pad256(LAYER_HDR + small.size) - LAYER_HDR - small.size
        w2 = np.zeros((64, 64), dtype=np.float32); w2[:H, :H] = W[1]
        w3 = np.zeros((64, 64), dtype=np.float32); w3[:H, :H] = W[2]
        w4 = np.zeros((NO, 64), dtype=np.float32); w4[:2 * D, :H] = W[3]
        words += [lead, small, np.zeros(pad, dtype=np.float32), umma_sw128_images(w2), umma_sw128_images(w3), umma_sw128_images(w4)]
    return _finish(words, HDR + len(layers) * nbw, folded[0].w[0].device)


def pack_spline_stack_tc(layers, bns: Optional[List[torch.nn.BatchNorm1d]]):
    """Tensor-core layout of a spline-coupling stack; None when the configuration is outside the kernel's envelope
    (hidden_dim <= 64, num_bins <= 10, <= 2 transformed dims per layer, data_dim <= 8)."""
    if layers[0].context_dim:
        return None
    return _pack_spline_tc(layers, bns, 0)


def pack_spline_stack_ctx_tc(layers, bns: Optional[List[torch.nn.BatchNorm1d]]):
    """Conditional twin of pack_spline_stack_tc ('NFC2', csrc/stack_small.cuh): the same envelope for layers that share
    one context_dim in 1..CTX_MAX; header word 3 holds it and every block gains the Wc section."""
    C = layers[0].context_dim
    if C < 1 or C > CTX_MAX:
        return None
    return _pack_spline_tc(layers, bns, C)


def _pack_spline_tc(layers, bns, C):
    l0 = layers[0]
    D, K = l0.data_dim, l0.num_bins
    H = l0.param_net[0].out_features
    if not _alike(layers, _spline_key):
        return None
    if D > DMAX or H > 64 or K < 2 or K > 10 or l0.param_net[0].weight.dtype != torch.float32:
        return None
    masks = [_np(l.mask) for l in layers]
    max_dt = max(int((m == 0).sum()) for m in masks)
    if max_dt < 1 or max_dt > 2:
        return None
    bw = L.lib().nf_spline_stack_tc_block_words(D, K, max_dt)
    if bw < 0:
        return None
    P = 3 * K - 1
    GS = 8 if K <= 8 else 10                       # slots per parameter group inside a dim's 32 columns
    W1S, NO3 = _w1s(D), 32 * max_dt
    if C:                                          # the Wc section moves the weight images by whole 256-word steps
        small = LAYER_HDR + 64 * W1S + 64 + NO3
        bw += _pad256(small + 64 * CTX_MAX) - _pad256(small)
    magic, w3 = (MAGIC_SPLINE_CTX_TC, C) if C else (MAGIC_SPLINE_TC, 1)
    words = [_stack_header(magic, D, H, w3, K, len(layers), W1S, NO3, bw, bns, spline=l0)]
    for i, (l, m) in enumerate(zip(layers, masks)):
        tdims = [d for d in range(D) if m[d] == 0]
        words.append(_layer_header(m.astype(np.float32), tdims, _rescale_arrays(l, D), _between_bn(bns, i, len(layers))))
        net = l.param_net
        W3, b3 = _np(net[4].weight), _np(net[4].bias)
        W3rows = np.zeros((NO3, H))
        b3rows = np.zeros(NO3)
        for t, d in enumerate(tdims):
            for g, cnt in enumerate((K, K, K - 1)):
                for j in range(cnt):
                    W3rows[t * 32 + g * GS + j] = W3[d * P + g * K + j]
                    b3rows[t * 32 + g * GS + j] = b3[d * P + g * K + j]
        W1 = _np(net[0].weight)
        words.append(_tc_net_block(W1[:, :D], _np(net[0].bias), _np(net[2].weight), _np(net[2].bias),
                                   W3rows, b3rows, D, H, W1S, NO3, LAYER_HDR, Wc=W1[:, D:] if C else None))
    return _finish(words, HDR + len(layers) * bw, l0.param_net[0].weight.device)


def pack_coupling_stack_tc(layers, bns: Optional[List[torch.nn.BatchNorm1d]]):
    """Tensor-core layout of an eval-mode affine coupling stack (hidden_dim <= 128, padded to 64 or 128; data_dim <= 8):
    per layer two net blocks (s_net then b_net), each `lead (80 words: the layer header for s_net, zeros for b_net) |
    W1k | b2 | b3 | pad | W2 hi/lo images | W3 hi/lo images`, conditioner BatchNorm folded into the Linears."""
    if layers[0].context_dim:
        return None
    return _pack_coupling_tc(layers, bns, 0)


def pack_coupling_stack_ctx_tc(layers, bns: Optional[List[torch.nn.BatchNorm1d]]):
    """Conditional twin of pack_coupling_stack_tc ('NFD2', csrc/stack_small.cuh): the same envelope for layers that share
    one context_dim in 1..CTX_MAX; header word 3 holds it and every net block gains the Wc section after b3.  The
    conditioner BatchNorm is folded into the whole [H, D + C] first weight -- it scales rows, context columns included --
    before the weight is split into its x columns (W1k) and context columns (Wc)."""
    C = layers[0].context_dim
    if C < 1 or C > CTX_MAX:
        return None
    return _pack_coupling_tc(layers, bns, C)


def _pack_coupling_tc(layers, bns, C):
    l0 = layers[0]
    D = l0.data_dim
    H = l0.s_net[0].out_features
    if not _alike(layers, _coupling_key):
        return None
    if D > DMAX or H > 128 or l0.s_net[0].weight.dtype != torch.float32:
        return None
    HP = _hp(H)
    nbw = (L.lib().nf_coupling_stack_ctx_tc_block_words_hidden if C else L.lib().nf_coupling_stack_tc_block_words_hidden)(D, H)
    if nbw < 0:
        return None
    W1S, NO3 = _w1s(D), 16
    magic, w3 = (MAGIC_AFFINE_CTX_TC, C) if C else (MAGIC_AFFINE_TC, 2)
    words = [_stack_header(magic, D, H, w3, 0, len(layers), W1S, NO3, nbw, bns)]
    for i, l in enumerate(layers):
        m = _np(l.mask)
        lead = [_layer_header(m.astype(np.float32), [d for d in range(D) if m[d] == 0], None,
                              _between_bn(bns, i, len(layers))),
                np.zeros(LAYER_HDR, dtype=np.float32)]
        for net, ld in zip((l.s_net, l.b_net), lead):
            W1, b1 = _fold_bn(_np(net[0].weight), _np(net[0].bias), net[1])
            W2, b2 = _fold_bn(_np(net[3].weight), _np(net[3].bias), net[4])
            W3rows = np.zeros((NO3, H))
            b3rows = np.zeros(NO3)
            W3rows[:D] = _np(net[6].weight)
            b3rows[:D] = _np(net[6].bias)
            blk = _tc_net_block(W1[:, :D], b1, W2, b2, W3rows, b3rows, D, H, W1S, NO3, LAYER_HDR, HP,
                                Wc=W1[:, D:] if C else None)
            words += [ld, blk]
    return _finish(words, HDR + 2 * len(layers) * nbw, l0.s_net[0].weight.device)
