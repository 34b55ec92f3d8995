"""Flow layers of the hot path: same class names, constructor arguments, attributes and state_dict
layout as the reference's `src.flows` (SURVEY 8b / A.2), with every [B, *]-sized computation running in
libnfb200.so (sm_100a).  Reference files, relative to the reference repository root:

    Flow / SequentialFlow               src/flows/flow/flow.py:4-73, src/flows/flow/sequential_flow.py:5-34
    CouplingLayer                       src/flows/coupling/coupling_layer.py:5-111
    SplineCouplingLayer                 src/flows/spline/spline_coupling_layer.py:6-323
    rational_quadratic_spline           src/flows/spline/rational_quadratic_spline.py:4-104
    MaskedLinear / MADE                 src/flows/autoregressive/masked_linear.py:4-18, made.py:6-140
    MaskedAutoregressiveFlow            src/flows/autoregressive/masked_autoregressive_flow.py:5-78
    InverseAutoregressiveFlow           src/flows/autoregressive/inverse_autoregressive_flow.py:5-103

Two execution routes per layer, chosen per call:
  * fused   (no autograd needed, float32): one launch for the whole layer -- or the whole stack when the
            caller is a container, see ChainPlan -- conditioner included;
  * layered (training, float64, wide layers): conditioner GEMMs + BatchNorm + transform kernels, each an
            autograd Function with a hand-written backward kernel (ops.py).
There is no CPU route: tensors and modules must live on a CUDA device.
"""
from __future__ import annotations


import numpy as np
import torch
import torch.nn as nn

from . import _lib as L
from . import ops, packing


def wants_grad(module: nn.Module, *tensors) -> bool:
    if not torch.is_grad_enabled():
        return False
    if any(t is not None and t.requires_grad for t in tensors):
        return True
    return any(p.requires_grad for p in module.parameters())


def compute_input(v):
    """Inputs arriving in half precision (a caller running under torch.autocast, e.g. the reference's
    MixedPrecisionFlow wrapper, optimization/mixed_precision.py:89-105) are widened: the kernels compute in the
    parameters' float32 / float64, which is what autocast leaves these ops in anyway."""
    if v.dtype in (torch.float16, torch.bfloat16):
        return v.float()
    return v


def on_input_device(fn):
    """Run a module method under the CUDA device of its tensor argument.  The C ABI launches on the *current* device's
    stream; a model that lives on cuda:1 while cuda:0 is current (plain `model.to('cuda:1')`, which works with the
    reference) must therefore switch devices around the launches instead of passing device-1 pointers to device 0."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, v, *args, **kwargs):
        if isinstance(v, torch.Tensor) and v.is_cuda and v.device.index != torch.cuda.current_device():
            with torch.cuda.device(v.device):
                return fn(self, v, *args, **kwargs)
        return fn(self, v, *args, **kwargs)
    return wrapped


_STD_NORMAL_CACHE = {}


def is_std_normal(base_dist, D=None) -> bool:
    """True when `base_dist` is N(0, I): torch.distributions Normal(0, 1) (scalar or [D] parameters), Independent of
    it, or MultivariateNormal with zero mean and identity covariance -- the case every caller of the reference uses
    (README.md:113-114, plots/_common.py:201-202).  Reading the parameters costs one device sync, so the verdict is
    cached per distribution object (torch distributions are immutable)."""
    if base_dist is None:
        return True
    key = id(base_dist)
    hit = _STD_NORMAL_CACHE.get(key)
    if hit is not None and hit[0]() is base_dist:
        return hit[1]
    import weakref
    from torch import distributions as td
    ok = False
    try:
        d = base_dist
        if isinstance(d, td.Independent):
            d = d.base_dist
        if type(d) is td.Normal:
            ok = bool((d.loc == 0).all()) and bool((d.scale == 1).all()) and d.loc.dim() <= 1
            if ok and D is not None and d.loc.dim() == 1 and d.loc.numel() not in (1, D):
                ok = False
        elif type(d) is td.MultivariateNormal and d is base_dist:
            n = d.loc.shape[-1]
            eye = torch.eye(n, dtype=d.loc.dtype, device=d.loc.device)
            ok = d.loc.dim() == 1 and bool((d.loc == 0).all()) and bool((d.scale_tril == eye).all())
            if ok and D is not None and n != D:
                ok = False
    except Exception:
        ok = False
    if len(_STD_NORMAL_CACHE) > 64:
        _STD_NORMAL_CACHE.clear()
    try:
        _STD_NORMAL_CACHE[key] = (weakref.ref(base_dist), ok)
    except TypeError:
        pass
    return ok


class _Context:
    """A validated context: row r of the batch is conditioned on t[r // div] (div = 1: one context row per row; the
    batch size: one row for all; n: n samples per context row).  One object serves every layer of a call."""
    __slots__ = ("t", "div", "_per_row")

    def __init__(self, t, div):
        self.t, self.div, self._per_row = t, div, None

    def layered(self, B):
        """(context rows, div) the layered first Linear reads: one row per row, or a single row for all.  n rows per
        context row (the layered route of sampling) are expanded once per call, not once per layer."""
        if self.div == 1 or self.t.shape[0] == 1:
            return self.t, self.div
        if self._per_row is None:
            self._per_row = self.t.repeat_interleave(self.div, 0)[:B]
        return self._per_row, 1


def _context_dim(module) -> int:
    """C of the conditional layers a flow or container holds (0: none); fixed when the module is built."""
    return getattr(module, "context_dim", 0) or 0


def _shared_context_dim(flows) -> int:
    """The context width of a container: every conditional layer reads the one context, so they must agree."""
    dims = {_context_dim(f) for f in flows} - {0}
    if len(dims) > 1:
        raise ValueError(f"the conditional layers of one model share one context; got context_dim values {sorted(dims)}")
    return dims.pop() if dims else 0


def _as_context(module, context, v, div=None, what="rows"):
    """Validate `context` for a call of `module` on v [B, D] and return it as a _Context (None without one).  context:
    [B, C] (one row per row), [1, C] (broadcast to every row) or, with div = n (sampling), [m, C] for m*n rows.  Raises
    ValueError for a conditional model called without context, a context given to a model without conditional layer,
    and a context of the wrong width, row count, dtype or device; a context is never dropped."""
    C = _context_dim(module)
    if context is None:
        if C:
            raise ValueError(f"{type(module).__name__} has conditional layers (context_dim={C}): pass context=")
        return None
    if not C:
        raise ValueError(f"{type(module).__name__} has no conditional layer (context_dim=0) but a context was passed")
    if isinstance(context, _Context):
        return context
    if not isinstance(context, torch.Tensor) or context.dim() != 2 or context.shape[1] != C:
        shape = tuple(context.shape) if isinstance(context, torch.Tensor) else type(context).__name__
        raise ValueError(f"context must be a [{what}, {C}] tensor (context_dim={C}); got {shape}")
    context = compute_input(context)
    dtype = compute_input(v).dtype if isinstance(v, torch.Tensor) else v[0]
    device = v.device if isinstance(v, torch.Tensor) else v[1]
    if context.dtype != dtype:
        raise ValueError(f"context has dtype {context.dtype}, the flow computes in {dtype}")
    if context.device != torch.device(device):
        raise ValueError(f"context is on {context.device}, the flow's input on {device}")
    if div is None:
        B = v.shape[0]
        if context.shape[0] == B:
            div = 1
        elif context.shape[0] == 1:
            div = max(B, 1)
        else:
            raise ValueError(f"context has {context.shape[0]} rows; expected {B} (one per row) or 1 (broadcast)")
    elif context.shape[0] < 1:
        raise ValueError("context has no rows")
    return _Context(context.contiguous(), int(div))


def _default_base(D, device, dtype=torch.float32):
    from torch import distributions as td
    return td.Normal(torch.zeros(D, device=device, dtype=dtype), torch.ones(D, device=device, dtype=dtype))


def flow_log_prob(flow, x, base_dist, fused_head=None, context=None):
    """Flow.log_prob (flow.py:56-73).  For a standard-normal base the head log N(z; 0, I) + log_det is one kernel
    (nf_std_normal_log_prob_*, with a backward), or -- `fused_head`, no autograd graph needed -- part of the last
    layer's epilogue of the fused stack launch; any other base goes through the torch distribution on the returned z.
    context: the conditional layers' context, [B, C] or [1, C] (see _as_context)."""
    ctx = _as_context(flow, context, x)
    D = x.shape[-1] if x.dim() == 2 else None
    std = x.is_cuda and x.dim() == 2 and is_std_normal(base_dist, D)
    if std and fused_head is not None:
        with torch.cuda.device(x.device):
            lp = fused_head(x) if ctx is None else fused_head(x, ctx)
        if lp is not None:
            return lp
    z, log_det_inv = flow.inverse(x) if ctx is None else flow.inverse(x, ctx)
    if std and z.dtype in (torch.float32, torch.float64):
        return ops.std_normal_log_prob(z, log_det_inv)
    log_p_z = base_dist.log_prob(z)
    if log_p_z.dim() > 1:
        log_p_z = log_p_z.sum(dim=1)
    return log_p_z + log_det_inv


def _event_dim(flow):
    """data_dim of a flow or container (SequentialFlow and the models take it from their first layer)."""
    d = getattr(flow, "data_dim", None)
    if d is None:
        flows = getattr(flow, "flows", None)
        if flows is None and hasattr(flow, "flow"):
            flows = flow.flow.flows
        if flows:
            d = _event_dim(flows[0])
    return d


_U64 = (1 << 64) - 1


class DeviceGenerator:
    """Seed and offset of the on-device N(0, I) draw of sample_and_log_prob, kept in device memory so that the call can
    be captured in a CUDA graph.

    The state is an int64 [4] CUDA tensor {seed, offset, ticket, reserved} (include/nfb200.h, "device-resident generator
    state").  The kernel that draws reads the key (seed, offset) there and moves the offset on by 4 in the same launch,
    so every graph replay draws new samples, and manual_seed makes the replays reproducible.  A DeviceGenerator at
    (s, o) draws the same bits as a torch.Generator with seed s at offset o.  seed=None takes the initial_seed() of
    torch's default CUDA generator of `device`, so torch.manual_seed(s); DeviceGenerator() starts at (s, 0).

    The state is stream-ordered: use one generator from one stream at a time.  manual_seed, get_offset and set_offset
    copy between host and device and raise RuntimeError under stream capture; initial_seed reads a host copy."""

    def __init__(self, device=None, seed=None):
        device = torch.device(device if device is not None else "cuda")
        if device.type != "cuda":
            raise RuntimeError(f"DeviceGenerator keeps its state in CUDA memory; got device {device}")
        torch.cuda.init()
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self._device = device
        if seed is None:
            seed = torch.cuda.default_generators[device.index].initial_seed()
        self._state = torch.zeros(4, dtype=torch.int64, device=device)
        self.manual_seed(seed)

    @property
    def device(self):
        return self._device

    @staticmethod
    def _no_capture(what):
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError(f"DeviceGenerator.{what} copies between host and device and cannot run under CUDA-graph "
                               "capture; call it before capturing or between replays")

    @staticmethod
    def _i64(v):
        v = int(v) & _U64
        return v - (1 << 64) if v >= (1 << 63) else v

    def _write(self, words):
        with torch.cuda.device(self._device):
            self._state.copy_(torch.tensor([self._i64(w) for w in words], dtype=torch.int64))

    def manual_seed(self, seed):
        """State (seed, 0, 0, 0); returns self, like torch.Generator.manual_seed."""
        self._no_capture("manual_seed")
        self._seed = int(seed) & _U64
        self._write((self._seed, 0, 0, 0))
        return self

    def initial_seed(self):
        return self._seed

    def get_offset(self):
        """The offset of the next draw (waits for the draws queued on the current stream)."""
        self._no_capture("get_offset")
        with torch.cuda.device(self._device):
            return int(self._state[1].item()) & _U64

    def set_offset(self, offset):
        offset = int(offset)
        if offset < 0 or offset % 4:
            raise ValueError(f"the offset must be a non-negative multiple of 4, got {offset}")
        self._no_capture("set_offset")
        self._write((self._seed, offset, 0, 0))

    def __repr__(self):
        return f"DeviceGenerator(device={self._device}, seed={self._seed})"


def _draw_state(generator, device):
    """Key of one N(0, I) draw.  A DeviceGenerator: its state tensor, which the drawing kernel reads and advances
    (capturable).  Otherwise (seed, offset): the torch CUDA generator's seed and Philox offset, after which the offset
    moves on by 4 (torch keeps offsets a multiple of 4) -- torch.manual_seed makes a call reproducible, and consecutive
    calls draw new samples."""
    if isinstance(generator, DeviceGenerator):
        return generator._state
    if torch.cuda.is_current_stream_capturing():
        raise RuntimeError("sample_and_log_prob cannot be captured in a CUDA graph: the seed and offset of the draw are "
                           "read on the host, so every replay would repeat the same samples")
    gen = generator
    if gen is None:
        torch.cuda.init()
        gen = torch.cuda.default_generators[device.index if device.index is not None else torch.cuda.current_device()]
    seed, offset = int(gen.initial_seed()), int(gen.get_offset())
    gen.set_offset(offset + 4)
    return seed, offset


def flow_sample_and_log_prob(flow, num_samples, base_dist=None, device=None, generator=None, context=None):
    """(x, log_q): z ~ base, (x, log_det) = flow.forward(z), log_q = log p_base(z) - log_det (summed over the event axis
    as in Flow.log_prob), without materialising z where the route allows it.

    A standard-normal base (None, or any base is_std_normal accepts) is drawn on the device from the counter-based
    stream of csrc/nf_rng.cuh, seeded from `generator` (default: torch's default CUDA generator of `device`; a
    DeviceGenerator keeps seed and offset in device memory, which makes the call capturable in a CUDA graph); float64
    models widen its float32 normals.  A fused stack draws inside its one launch and evaluates log N(z) - log_det in the
    last layer's epilogue (`_sample_fused`); every other route draws z with nf_std_normal_draw, runs forward(z) -- with
    its autograd graph when parameters require grad, the reparameterised gradient -- and the log-q head kernel.  Any
    other base is sampled by torch (rsample where it has one) and cannot take a generator.  Every route draws once, so a
    DeviceGenerator moves on by exactly 4 per call (a fused stack that refuses the call launches nothing).
    context [m, C] (conditional models): num_samples rows per context row, context-major -- row r of the flat [m*n, D]
    draw is conditioned on context row r // n, and the draw itself does not depend on the context; x is returned as
    [m, n, D] and log_q as [m, n]."""
    p = next(flow.parameters(), None)
    device = torch.device(device if device is not None else (p.device if p is not None else "cpu"))
    dtype = p.dtype if p is not None else torch.float32
    D = _event_dim(flow)
    n = int(num_samples)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    ctx = _as_context(flow, context, (dtype, device), div=max(n, 1), what="m")
    rows = n if ctx is None else ctx.t.shape[0] * n
    shaped = (lambda x, lq: (x, lq)) if ctx is None else \
        (lambda x, lq: (x.view(ctx.t.shape[0], n, D), lq.view(ctx.t.shape[0], n)))
    fwd = flow.forward if ctx is None else (lambda z: flow.forward(z, ctx))
    if base_dist is not None and not is_std_normal(base_dist, D):
        if generator is not None:
            raise ValueError("generator= seeds the on-device N(0, I) draw only; torch distributions cannot take a generator")
        z = (base_dist.rsample if base_dist.has_rsample else base_dist.sample)((rows,)).to(device)
        x, log_det = fwd(z)
        log_p_z = base_dist.log_prob(z)
        if log_p_z.dim() > 1:
            log_p_z = log_p_z.sum(dim=1)
        return shaped(x, log_p_z - log_det)
    if isinstance(generator, DeviceGenerator) and generator.device != device:
        raise ValueError(f"the DeviceGenerator lives on {generator.device} but the draw is on {device}")
    if device.type != "cuda":
        raise RuntimeError(L.NO_CPU_PATH)
    with torch.cuda.device(device):
        draw = _draw_state(generator, device)
        fused = getattr(flow, "_sample_fused", None)
        if fused is not None and not wants_grad(flow, None if ctx is None else ctx.t):
            buf = torch.empty((rows, D), dtype=dtype, device=device)
            out = fused(buf, draw) if ctx is None else fused(buf, draw, ctx)
            if out is not None:
                return shaped(*out)
        z = ops.std_normal_draw(*ops._draw_key(draw), rows, D, dtype, device)
        x, log_det = fwd(z)
        return shaped(x, ops.std_normal_log_q(z, log_det))


def _module_tensors(module: nn.Module):
    return list(module.parameters()) + list(module.buffers())


class _PackCache:
    """Derived weight layouts keyed on (parameter versions, storage, device)."""

    def __init__(self):
        self._key = None
        self._val = None
        self._tensors = None
        self._owner_ids = None

    def get(self, tensors, build, extra=()):
        key = packing.tensors_key(tensors, extra)
        if key != self._key:
            self._val = build()
            self._key = key
        return self._val

    def tensors_of(self, modules):
        """Parameter/buffer list of `modules`, walked once (module.parameters() costs ~10 us per module per call; the
        per-call check is then one (data_ptr, version) tuple per tensor).  Re-walked if the module set changes."""
        ids = tuple(id(m) for m in modules)
        if ids != self._owner_ids:
            self._tensors = [t for m in modules for t in _module_tensors(m)]
            self._owner_ids = ids
        return self._tensors


def _fold_bn_eval(W, b, bn):
    """Linear followed by eval-mode BatchNorm1d == Linear with scaled rows (coupling_layer.py:19-24); device tensors."""
    s = bn.weight / torch.sqrt(bn.running_var + bn.eps)
    return W * s[:, None], (b - bn.running_mean) * s + bn.bias


def _tc_layer(W, b, relu):
    W = W.detach().float().contiguous()
    hi, lo = ops.split_tf32(W)
    return hi, lo, b.detach().float().contiguous(), relu, W


def _tc_mlp(v, layers):
    """relu?(... relu?(v W0^T + b0) ...) with cached folded weights: the tcgen05 GEMM (TF32 splits) for every layer it
    takes, the streaming FP32 kernels of nf_gemm for the skinny ones (reduction dimension or output width of a few
    columns: the first / last Linear of a low-dimensional conditioner) -- a 128-wide tensor-core tile would waste > 90 %
    of its work there, and K % 4 != 0 has no TMA row pitch."""
    h = v
    for hi, lo, b, relu, W in layers:
        N, K = W.shape
        out = ops.linear_tc(h, hi, lo, b, relu) if (K % 4 == 0 and K >= 16 and N >= 16) else None
        h = out if out is not None else ops.linear_raw(h, W, b, relu)
    return h


WIDE_TC_MIN_ROWS = 256
# hidden_dim in (64, 128] is outside the tcgen05 SPLINE stack kernels (the affine coupling stack has a 128-wide variant);
# the FP32-pipe stack kernels hold the layer's weights in shared memory at one 4-warp CTA per SM there (RealNVP(2, 10,
# 128), the reference's first published config: 57 ms per 2^20 rows, profiles/r02v_published_before.jsonl) -- from this
# many rows on the GEMM route is several times faster
WIDE_OVER_STACK_MIN_ROWS = 16384


# ------------------------------------------------------------------------------------------------
# base classes
# ------------------------------------------------------------------------------------------------
class Flow(nn.Module):
    """Base class: `forward(z) -> (x, log_det)`, `inverse(x) -> (z, log_det)` (flow.py:4-38)."""

    def __init__(self):
        super().__init__()
        self.data_dim = None
        self.context_dim = 0          # > 0: a conditional layer (or a container holding some), see _as_context

    def forward(self, z):
        raise NotImplementedError

    def inverse(self, x):
        raise NotImplementedError

    def sample(self, num_samples, base_dist=None, device="cpu", context=None):
        """flow.py:40-54 (base_dist=None: standard normal over data_dim / dim).  context [m, C] (conditional flows):
        num_samples rows per context row, returned as [m, n, D]."""
        return sample_from(self, self.data_dim, num_samples, base_dist, device, context)

    def log_prob(self, x, base_dist=None, context=None):
        """flow.py:56-73: log p(z) (summed over the event axis if the base is factorised) + log|det J_inv|.
        A standard-normal base is detected (is_std_normal) and evaluated by the fused head kernels.  context: [B, C]
        or [1, C] for a conditional flow."""
        return flow_log_prob(self, x, base_dist, getattr(self, "_log_prob_fused", None), context)

    def sample_and_log_prob(self, num_samples, base_dist=None, device=None, generator=None, context=None):
        """Samples and their log-density in one pass: z ~ base, (x, log_det) = forward(z), log_q = log p_base(z) - log_det.
        device=None: the parameters' device; dtype: the parameters'.  A standard-normal base (None or N(0, I)) is drawn on
        the GPU from `generator` (torch.Generator on that device; None = torch's default CUDA generator, so
        torch.manual_seed makes the call reproducible); float64 models widen the float32 draw.  Raises RuntimeError under
        CUDA-graph capture, ValueError for a generator with any other base.  context [m, C] (conditional flows): x
        [m, n, D] and log_q [m, n].  See flow_sample_and_log_prob."""
        return flow_sample_and_log_prob(self, num_samples, base_dist, device, generator, context)


def sample_from(flow, D, num_samples, base_dist, device, context):
    """Flow.sample: z ~ base (a torch distribution), x = forward(z); with context [m, C], m * num_samples rows,
    context-major, returned as [m, n, D]."""
    if base_dist is None:
        base_dist = _default_base(D, device)
    if context is None:
        z = base_dist.sample((num_samples,)).to(device)
        x, _ = flow.forward(z)
        return x
    p = next(flow.parameters(), None)
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:           # as flow_sample_and_log_prob: 'cuda' is the current one
        device = torch.device("cuda", torch.cuda.current_device())
    ctx = _as_context(flow, context, (p.dtype if p is not None else torch.float32, device),
                      div=max(int(num_samples), 1), what="m")
    m = ctx.t.shape[0]
    z = base_dist.sample((m * num_samples,)).to(device)
    x, _ = flow.forward(z, ctx)
    return x.view(m, num_samples, -1)


def _apply_layer(flow, v, inverse, ctx):
    """One layer of a container: conditional layers get the container's context, the others are called as before."""
    if ctx is not None and _context_dim(flow):
        return flow._run(v, inverse, ctx)
    return flow.inverse(v) if inverse else flow.forward(v)


class SequentialFlow(Flow):
    """Flows applied in order; inverse walks them backwards (sequential_flow.py:5-34)."""

    def __init__(self, flows):
        super().__init__()
        if not isinstance(flows, (list, nn.ModuleList)):
            raise ValueError("flows must be a list or nn.ModuleList")
        self.flows = nn.ModuleList(flows)
        self.context_dim = _shared_context_dim(self.flows)
        self._chain = ChainPlan()

    def _log_prob_fused(self, x, ctx=None):
        out = self._chain.run(self.flows, None, self.training, x, True, head=True, ctx=ctx)
        return None if out is None else out[1]

    def _sample_fused(self, x, draw, ctx=None):
        return self._chain.run(self.flows, None, self.training, x, False, sample=draw, ctx=ctx)

    @on_input_device
    def _run(self, v, inverse, ctx=None):
        fused = self._chain.run(self.flows, None, self.training, v, inverse, ctx=ctx)
        if fused is not None:
            return fused
        total = torch.zeros(v.size(0), device=v.device)         # float32 accumulator, as the reference
        for flow in (reversed(self.flows) if inverse else self.flows):
            v, ld = _apply_layer(flow, v, inverse, ctx)
            total += ld
        return v, total

    def forward(self, z, context=None):
        return self._run(z, False, _as_context(self, context, z))

    def inverse(self, x, context=None):
        return self._run(x, True, _as_context(self, context, x))


class _Coupling(Flow):
    """Shared driver of CouplingLayer and SplineCouplingLayer: their one-launch route, which `_run` takes first when no
    autograd graph is needed and `fusable` holds, and which draws the input in the kernel for sample_and_log_prob."""
    _stack = None       # key of run_stack's family table

    def _fused(self, v, inverse, sample=None, ctx=None):
        return run_stack(self._stack, self._pack, self._pack.tensors_of([self]), [self], None, v, inverse, sample=sample,
                         ctx=ctx)

    def _sample_fused(self, x, draw, ctx=None):
        """The layer's own fused route of forward (one launch), drawing its input in the kernel."""
        return self._fused(x, False, draw, ctx) if self.fusable(x) else None

    def forward(self, z, context=None):
        return self._run(z, False, _as_context(self, context, z))

    def inverse(self, x, context=None):
        return self._run(x, True, _as_context(self, context, x))


# ------------------------------------------------------------------------------------------------
# affine coupling
# ------------------------------------------------------------------------------------------------
def _coupling_net(data_dim, hidden_dim, context_dim=0):
    return nn.Sequential(
        nn.Linear(data_dim + context_dim, hidden_dim), nn.BatchNorm1d(hidden_dim), nn.ReLU(),
        nn.Linear(hidden_dim, hidden_dim), nn.BatchNorm1d(hidden_dim), nn.ReLU(),
        nn.Linear(hidden_dim, data_dim))


class CouplingLayer(_Coupling):
    """RealNVP affine coupling layer (coupling_layer.py:5-111).

    s = clamp(s_net(x*mask), +-10), b = clamp(b_net(x*mask), +-10);
    forward  x = z*mask + (1-mask)*(z*exp(s)+b),     log_det =  sum((1-mask)*s)
    inverse  z = x*mask + (1-mask)*((x-b)*exp(-s)),  log_det = -sum((1-mask)*s);  NaN/Inf -> 0.

    context_dim = C > 0 makes it conditional, p(x | c): both conditioners read [x * mask, c] (context columns last, as in
    nflows), so s_net[0] and b_net[0] are Linear(data_dim + C, hidden_dim); the context is not masked.  forward /
    inverse then take context= [B, C] or [1, C] (broadcast).
    """

    def __init__(self, data_dim, hidden_dim, mask, context_dim=0):
        super().__init__()
        if int(context_dim) != context_dim or context_dim < 0:
            raise ValueError(f"context_dim must be a non-negative integer, got {context_dim!r}")
        self.context_dim = int(context_dim)
        self.data_dim = data_dim
        self.register_buffer("mask", mask)
        self.s_net = _coupling_net(data_dim, hidden_dim, self.context_dim)
        self.b_net = _coupling_net(data_dim, hidden_dim, self.context_dim)
        self._initialize_weights()
        self._pack = _PackCache()
        self._wide = _PackCache()

    def _initialize_weights(self):
        """xavier-normal hidden layers with zero bias, zero final layer => identity at init (:98-111)."""
        for net in (self.s_net, self.b_net):
            for layer in list(net)[:-1]:
                if isinstance(layer, nn.Linear):
                    nn.init.xavier_normal_(layer.weight, gain=1.0)
                    nn.init.zeros_(layer.bias)
        for net in (self.s_net, self.b_net):
            nn.init.zeros_(net[-1].weight)
            nn.init.zeros_(net[-1].bias)

    @property
    def _stack(self):             # key of run_stack's family table
        return "coupling_ctx" if self.context_dim else "coupling"

    # -- layered route -------------------------------------------------------------------------
    def _conditioner(self, net, v, ctx=None):
        # x*mask is folded into the first weight's columns (same zero/NaN propagation as the product x*mask); the
        # context columns [x*mask, c] go through linear_ctx without its ReLU, so that a train-mode BatchNorm normalises
        # the full pre-activation, context included, as after a concatenated input
        if ctx is not None:
            c, div = ctx.layered(v.shape[0])
            h = ops.linear_ctx(v, c, net[0].weight, net[0].bias, self.mask, div, relu=False)
        else:
            h = ops.linear(v, net[0].weight, net[0].bias, mask=self.mask)
        h = ops.batchnorm_relu(h, net[1])
        h = ops.linear(h, net[3].weight, net[3].bias)
        h = ops.batchnorm_relu(h, net[4])
        return ops.linear(h, net[6].weight, net[6].bias)

    def fusable(self, v):
        H = self.s_net[0].out_features
        if H > 64 and v.shape[0] >= WIDE_OVER_STACK_MIN_ROWS and not USE_TENSOR_CORES and ops.USE_TENSOR_CORE_GEMM:
            return False                              # no tcgen05 stack kernel: see WIDE_OVER_STACK_MIN_ROWS
        return (not self.training and v.dtype == torch.float32 and self.s_net[0].weight.dtype == torch.float32
                and self.data_dim <= packing.DMAX and H <= 128)

    @on_input_device
    def _run(self, v, inverse, ctx=None):
        v = compute_input(v)
        ct = None if ctx is None else ctx.t
        if not wants_grad(self, v, ct) and self.fusable(v):
            out = self._fused(v, inverse, ctx=ctx)
            if out is not None:
                return out
        if (ctx is None and not wants_grad(self, v) and not self.training and USE_TENSOR_CORES and ops.USE_TENSOR_CORE_GEMM
                and v.dtype == torch.float32 and self.s_net[0].weight.dtype == torch.float32 and v.shape[0] >= WIDE_TC_MIN_ROWS):
            # wide eval route: mask and eval-mode BatchNorm folded into the Linears once per weight version, TF32 splits
            # cached, three tensor-core GEMMs per net (the layered route re-folds and re-splits on every call)
            nets = self._wide.get(self._wide.tensors_of([self]), self._fold_wide)
            return ops.affine_coupling(v, _tc_mlp(v, nets[0]), _tc_mlp(v, nets[1]), self.mask, inverse)
        s_raw = self._conditioner(self.s_net, v, ctx)
        b_raw = self._conditioner(self.b_net, v, ctx)
        return ops.affine_coupling(v, s_raw, b_raw, self.mask, inverse)

    def _fold_wide(self):
        with torch.no_grad():
            out = []
            for net in (self.s_net, self.b_net):
                W0, b0 = _fold_bn_eval(net[0].weight * self.mask[None, :], net[0].bias, net[1])
                W1, b1 = _fold_bn_eval(net[3].weight, net[3].bias, net[4])
                out.append([_tc_layer(W0, b0, True), _tc_layer(W1, b1, True), _tc_layer(net[6].weight, net[6].bias, False)])
            return out


# ------------------------------------------------------------------------------------------------
# rational-quadratic spline coupling
# ------------------------------------------------------------------------------------------------
class SplineCouplingLayer(_Coupling):
    """Neural-spline coupling layer on [-bound, bound] with identity tails (spline_coupling_layer.py:6-323).

    context_dim = C > 0 makes it conditional, p(x | c): the conditioner's input is [x_rescaled * mask, c] (context
    columns last, as in nflows), so param_net[0] is Linear(data_dim + C, hidden_dim); the context is neither rescaled
    nor masked.  forward / inverse then take context= [B, C] or [1, C] (broadcast)."""

    def __init__(self, data_dim, hidden_dim, mask, num_bins=10, bound=5.0, min_bin_width=1e-3, min_bin_height=1e-3,
                 min_derivative=1e-3, data_min=None, data_max=None, context_dim=0):
        super().__init__()
        if int(context_dim) != context_dim or context_dim < 0:
            raise ValueError(f"context_dim must be a non-negative integer, got {context_dim!r}")
        self.context_dim = int(context_dim)
        self.data_dim = data_dim
        self.num_bins = num_bins
        self.bound = bound
        self.min_bin_width = min_bin_width
        self.min_bin_height = min_bin_height
        self.min_derivative = min_derivative
        self.data_min = data_min
        self.data_max = data_max
        self.register_buffer("mask", mask)
        self.param_net = nn.Sequential(
            nn.Linear(data_dim + self.context_dim, hidden_dim), nn.ReLU(),
            nn.Linear(hidden_dim, hidden_dim), nn.ReLU(),
            nn.Linear(hidden_dim, data_dim * (3 * num_bins - 1)))
        self._initialize_weights()
        self._pack = _PackCache()
        self._aux = _PackCache()
        self._wide = _PackCache()

    def _initialize_weights(self):
        """:311-323."""
        for layer in list(self.param_net)[:-1]:
            if isinstance(layer, nn.Linear):
                nn.init.xavier_normal_(layer.weight, gain=1.0)
                nn.init.zeros_(layer.bias)
        nn.init.zeros_(self.param_net[-1].weight)
        nn.init.zeros_(self.param_net[-1].bias)

    @property
    def _stack(self):             # key of run_stack's family table
        return "spline_ctx" if self.context_dim else "spline"

    @property
    def _mins(self):
        return (self.min_bin_width, self.min_bin_height, self.min_derivative)

    def _aux_tensors(self, v):
        """(tidx int32 [Dt] on device, rescale (a, lo, c) or None, transformed dims as a host list)."""
        def build():
            tlist = torch.nonzero(self.mask.detach().to("cpu") == 0).flatten().tolist()
            tidx = torch.tensor(tlist, dtype=torch.int32, device=v.device)
            return tidx, packing.rescale_tensors(self, self.data_dim, v.dtype, v.device), tlist
        return self._aux.get([self.mask], build, extra=(v.dtype, v.device))

    def fusable(self, v):
        H = self.param_net[0].out_features
        if H > 64 and v.shape[0] >= WIDE_OVER_STACK_MIN_ROWS and USE_TENSOR_CORES and ops.USE_TENSOR_CORE_GEMM:
            return False                              # see WIDE_OVER_STACK_MIN_ROWS
        return (v.dtype == torch.float32 and self.param_net[0].weight.dtype == torch.float32
                and self.data_dim <= packing.DMAX and H <= 128 and 2 <= self.num_bins <= 16)

    @on_input_device
    def _run(self, v, inverse, ctx=None):
        v = compute_input(v)
        ct = None if ctx is None else ctx.t
        if not wants_grad(self, v, ct) and self.fusable(v):
            out = self._fused(v, inverse, ctx=ctx)
            if out is not None:
                return out
        tidx, rescale, tlist = self._aux_tensors(v)
        net = self.param_net
        vin = v
        if rescale is not None:                       # conditioner sees the rescaled input (:101-102)
            vin = ops.feature_affine(v, rescale[1], None, rescale[0], -float(self.bound))
        if ctx is not None:                           # [x_rescaled * mask, c] -> first Linear, without concatenating
            c, div = ctx.layered(v.shape[0])
            h = ops.linear_ctx(vin, c, net[0].weight, net[0].bias, self.mask, div)
        elif (not wants_grad(self, v) and USE_TENSOR_CORES and ops.USE_TENSOR_CORE_GEMM and v.dtype == torch.float32 and net[0].weight.dtype == torch.float32
                and v.shape[0] >= WIDE_TC_MIN_ROWS and tlist):
            layers = self._wide.get(self._wide.tensors_of([self]), lambda: self._fold_wide(tlist))
            return ops.spline_transform(v, _tc_mlp(vin, layers), self.mask, tidx, self.num_bins, inverse, self.bound,
                                        self._mins, rescale, compact=True)
        else:
            h = ops.linear(vin, net[0].weight, net[0].bias, mask=self.mask, relu=True)
        h = ops.linear(h, net[2].weight, net[2].bias, relu=True)
        # head restricted to the transformed dims: the reference evaluates all D*(3K-1) outputs and discards the rows
        # of the conditioning dims (SURVEY D9); no used value changes
        w4, b4 = self._head_rows(net[4], tlist)
        params = ops.linear(h, w4, b4)
        return ops.spline_transform(v, params, self.mask, tidx, self.num_bins, inverse, self.bound, self._mins,
                                    rescale, compact=True)

    def _fold_wide(self, tlist):
        """Mask-folded first Linear, compact head, TF32 splits: cached per weight version for the no-grad route."""
        with torch.no_grad():
            net = self.param_net
            w4, b4 = self._head_rows(net[4], tlist)
            return [_tc_layer(net[0].weight * self.mask[None, :], net[0].bias, True),
                    _tc_layer(net[2].weight, net[2].bias, True), _tc_layer(w4, b4, False)]

    def _head_rows(self, lin, t):
        """Rows d*(3K-1)+j of the last Linear for the transformed dims d in `t`: a contiguous slice (a view) for the
        half-split masks of RealNVPSpline, an index_select otherwise."""
        P = 3 * self.num_bins - 1
        if not t:
            return lin.weight[:0], lin.bias[:0]
        if t == list(range(t[0], t[0] + len(t))):
            return lin.weight[t[0] * P:(t[-1] + 1) * P], lin.bias[t[0] * P:(t[-1] + 1) * P]
        rows = torch.cat([torch.arange(d * P, (d + 1) * P, device=lin.weight.device) for d in t])
        return lin.weight.index_select(0, rows), lin.bias.index_select(0, rows)


def rational_quadratic_spline(inputs, widths, heights, derivatives, inverse=False, min_bin_width=1e-3,
                              min_bin_height=1e-3, min_derivative=1e-3, epsilon=1e-6):
    """Public spline on [0,1] (rational_quadratic_spline.py:4-104): per-element outputs and log|dy/dx|.
    `epsilon` is accepted and ignored, as in the reference (it is overwritten with 1e-6, :19)."""
    inputs, widths, heights, derivatives = (compute_input(t) for t in (inputs, widths, heights, derivatives))
    K = widths.shape[-1]
    x = inputs.reshape(-1)
    y, ld = ops.rqs_unit(x, widths.reshape(-1, K), heights.reshape(-1, K), derivatives.reshape(-1, K - 1), inverse,
                         (min_bin_width, min_bin_height, min_derivative))
    return y.view(inputs.shape), ld.view(inputs.shape)


# ------------------------------------------------------------------------------------------------
# MADE / MAF / IAF
# ------------------------------------------------------------------------------------------------
class MaskedLinear(nn.Linear):
    """nn.Linear whose weight is multiplied by a fixed binary mask (masked_linear.py:4-18)."""

    def __init__(self, in_features, out_features, mask, bias=True):
        super().__init__(in_features, out_features, bias)
        self.register_buffer("mask", mask)

    @on_input_device
    def forward(self, input):
        return ops.linear(input, self.weight, self.bias, mask=self.mask)


def made_degrees(input_dim, hidden_dim):
    """Hidden-unit degrees (made.py:25-41): interleaved [0,0,1,1,...] for D==2, floor(linspace) for D>2."""
    if input_dim > 1:
        if input_dim == 2:
            return np.array([0, 0, 1, 1] * (hidden_dim // 4 + 1))[:hidden_dim]
        return np.floor(np.linspace(0, input_dim - 1, hidden_dim)).astype(int)
    return np.zeros(hidden_dim, dtype=int)


class MADE(nn.Module):
    """Masked autoencoder conditioner: in->H, H->H, H->H, H->mult*D masked linears with ReLUs (made.py:6-140)."""

    def __init__(self, input_dim, hidden_dim, output_dim_multiplier=2, use_batch_norm=False):
        super().__init__()
        self.input_dim = input_dim
        self.hidden_dim = hidden_dim
        self.output_dim_multiplier = output_dim_multiplier
        self.use_batch_norm = use_batch_norm
        self.m = {-1: np.arange(input_dim), 0: made_degrees(input_dim, hidden_dim), 1: np.arange(input_dim)}
        self.masks = self.create_masks()
        self.net = self.create_network()
        self._fold = _PackCache()

    def create_masks(self):
        """in->h: deg(j) <= deg(a); h->h: deg(b) <= deg(a); h->out: deg(a) < i, strict (made.py:47-79)."""
        d_in, d_h, d_out = self.m[-1], self.m[0], self.m[1]
        m_in = (d_in[None, :] <= d_h[:, None]).astype(np.float32)                  # [H, D]
        m_hh = (d_h[None, :] <= d_h[:, None]).astype(np.float32)                   # [H, H]
        m_out = np.tile((d_h[None, :] < d_out[:, None]).astype(np.float32), (self.output_dim_multiplier, 1))
        # on torch's default device, like the nn.Linear parameters beside them (a model built under
        # `with torch.device("cuda")` is then on one device as a whole)
        dev = torch.get_default_device()
        return [torch.from_numpy(m).to(dev) for m in (m_in, m_hh, m_out)]

    def create_network(self):
        """made.py:81-134 (xavier-normal gain 0.5 hidden layers, N(0, 0.01^2) final layer, zero biases)."""
        H = self.hidden_dim
        linears = [MaskedLinear(self.input_dim, H, mask=self.masks[0]),
                   MaskedLinear(H, H, mask=self.masks[1]),
                   MaskedLinear(H, H, mask=self.masks[1]),
                   MaskedLinear(H, self.input_dim * self.output_dim_multiplier, mask=self.masks[2])]
        layers = []
        for lin in linears[:-1]:
            layers.append(lin)
            if self.use_batch_norm:
                layers.append(nn.BatchNorm1d(H))
            layers.append(nn.ReLU())
        layers.append(linears[-1])
        for lin in linears[:-1]:
            nn.init.xavier_normal_(lin.weight, gain=0.5)
            nn.init.zeros_(lin.bias)
        nn.init.normal_(linears[-1].weight, mean=0.0, std=0.01)
        nn.init.zeros_(linears[-1].bias)
        return nn.Sequential(*layers)

    def forward(self, x, out_rows=None):
        """Layered route: masked linears with the ReLU (or BatchNorm+ReLU) fused into the producing kernel.
        out_rows=(r0, r1) evaluates only output features [r0, r1) of the last masked linear (ARQS needs the 3K-1
        outputs of one dimension per step; the reference computes all of them and slices, arqs.py:56-64)."""
        mods = list(self.net)
        i, h = 0, x
        while i < len(mods):
            m = mods[i]
            if isinstance(m, MaskedLinear):
                nxt = mods[i + 1] if i + 1 < len(mods) else None
                if out_rows is not None and i == len(mods) - 1:
                    r0, r1 = out_rows
                    h = ops.linear(h, m.weight[r0:r1], None if m.bias is None else m.bias[r0:r1], mask=m.mask[r0:r1])
                    i += 1
                elif isinstance(nxt, nn.ReLU):
                    h = ops.linear(h, m.weight, m.bias, mask=m.mask, relu=True)
                    i += 2
                elif isinstance(nxt, nn.BatchNorm1d) and i + 2 < len(mods) and isinstance(mods[i + 2], nn.ReLU):
                    h = ops.batchnorm_relu(ops.linear(h, m.weight, m.bias, mask=m.mask), nxt)
                    i += 3
                else:
                    h = ops.linear(h, m.weight, m.bias, mask=m.mask)
                    i += 1
            else:
                h = m(h)
                i += 1
        return h

    def folded(self):
        """Mask-folded, degree-sorted weights for the fused kernels (None when BatchNorm / mult != 2)."""
        return self._fold.get(self._fold.tensors_of([self]), lambda: packing.fold_made(self))


class _AffineAutoregressive(Flow):
    """Shared driver of MAF and IAF: one direction is a single MADE pass, the other is D-step sequential."""
    _parallel_is_inverse = True
    _mode_parallel = L.AR_MAF_INVERSE
    _mode_sequential = L.AR_MAF_FORWARD

    def __init__(self, dim, hidden_dim=64, use_batch_norm=False):
        super().__init__()
        self.data_dim = dim
        self.dim = dim
        self.conditioner = MADE(dim, hidden_dim, 2, use_batch_norm=use_batch_norm)

    @on_input_device
    def _parallel(self, v):
        v = compute_input(v)
        if not wants_grad(self, v) and not (self.conditioner.use_batch_norm and self.training):
            f = self.conditioner.folded()
            if f is not None and f.w[0].dtype == v.dtype:
                return ops.made_affine(v, f, self._mode_parallel)
        return ops.affine_ar(v, self.conditioner(v), self._mode_parallel)

    @on_input_device
    def _sequential(self, v):
        v = compute_input(v)
        if not wants_grad(self, v) and not (self.conditioner.use_batch_norm and self.training):
            f = self.conditioner.folded()
            if f is not None and f.w[0].dtype == v.dtype:
                out = ops.ar_sequential(v, f, self._mode_sequential)
                if out is not None:
                    return out
        # D dependent steps, each re-evaluating the conditioner on the partially filled output
        # (masked_autoregressive_flow.py:55-67 / inverse_autoregressive_flow.py:76-91)
        cur = torch.zeros_like(v)
        ld = None
        for i in range(self.dim):
            cur, ld = ops.ar_step(cur, v, self.conditioner(cur), ld, i, self._mode_sequential)
        return ops.ar_finish(cur, v, ld, self._mode_sequential)


class MaskedAutoregressiveFlow(_AffineAutoregressive):
    """MAF: `inverse` (density) is one parallel pass, `forward` (sampling) is sequential
    (masked_autoregressive_flow.py:5-78)."""

    def inverse(self, x):
        return self._parallel(x)

    def forward(self, z):
        return self._sequential(z)

    def _log_prob_fused(self, x):
        """bf16 fused-chain mode: the N(0,I) head is part of the chain kernel's last epilogue (one launch, z not stored)."""
        x = compute_input(x)
        if (not ops.MADE_CHAIN_BF16 or wants_grad(self, x) or x.shape[0] < 128
                or (self.conditioner.use_batch_norm and self.training)):
            return None
        f = self.conditioner.folded()
        if f is None or f.w[0].dtype != x.dtype:
            return None
        out = ops.made_chain_bf16(x, f, self._mode_parallel, head=True)
        return None if out is None else out[1]


class InverseAutoregressiveFlow(_AffineAutoregressive):
    """IAF: `forward` (sampling) is one parallel pass, `inverse` (density) is sequential
    (inverse_autoregressive_flow.py:5-103)."""
    _mode_parallel = L.AR_IAF_FORWARD
    _mode_sequential = L.AR_IAF_INVERSE

    def __init__(self, dim, hidden_dim=64, use_batch_norm=False):
        super().__init__(dim, hidden_dim, use_batch_norm)
        final = self.conditioner.net[-1]                 # re-drawn N(0, 0.01^2) final layer (:21-28)
        nn.init.normal_(final.weight, mean=0.0, std=0.01)
        nn.init.zeros_(final.bias)

    def forward(self, z):
        return self._parallel(z)

    def inverse(self, x):
        return self._sequential(x)

    def _sample_fused(self, x, draw):
        """bf16 fused-chain mode (the route forward takes there): the draw, then one chain launch whose epilogue evaluates
        log N(z) - log_det on the input row."""
        if (not ops.MADE_CHAIN_BF16 or not ops.USE_TENSOR_CORE_GEMM or x.shape[0] < 128
                or (self.conditioner.use_batch_norm and self.training)):
            return None
        f = self.conditioner.folded()
        if f is None or f.w[0].dtype != x.dtype:
            return None
        out = ops.made_chain_bf16(x, f, self._mode_parallel, draw=draw)
        if isinstance(out, torch.Tensor):      # the chain refused after the draw: go on with that z, never draw twice
            y, log_det = self.forward(out)
            return y, ops.std_normal_log_q(out, log_det)
        return out


class ARQS(Flow):
    """Autoregressive rational-quadratic-spline flow (src/flows/spline/arqs.py:7-114): a MADE conditioner with 3K-1
    outputs per dimension and the public [0,1] spline.  As in the reference, BOTH directions are D-step sequential
    loops that re-evaluate the conditioner on the partially filled output; here every step runs the three hidden
    masked linears, only the 3K-1 head rows of the current dimension, and one fused spline-step kernel."""

    def __init__(self, dim, hidden_dim=128, num_bins=8, layers=2, data_min=None, data_max=None, use_batch_norm=False):
        super().__init__()
        self.dim = dim
        self.data_dim = dim
        self.num_bins = num_bins
        self.data_min = data_min
        self.data_max = data_max
        self.conditioner = MADE(input_dim=dim, hidden_dim=hidden_dim, output_dim_multiplier=3 * num_bins - 1,
                                use_batch_norm=use_batch_norm)

    def _rescale(self, v, to_unit):
        """(x - data_min) / (data_max - data_min) and its inverse (arqs.py:28-42); identity when either bound is None."""
        if self.data_min is None or self.data_max is None:
            return v
        span = self.data_max - self.data_min            # python scalars subtract in double, as in the reference
        lo = torch.as_tensor(self.data_min, dtype=v.dtype, device=v.device).expand(v.shape[1]).contiguous()
        span = torch.as_tensor(span, dtype=v.dtype, device=v.device).expand(v.shape[1]).contiguous()
        if to_unit:
            return ops.feature_affine(v, lo, span, None, None)
        return ops.feature_affine(v, None, None, span, lo)

    @on_input_device
    def _run(self, v, inverse):
        v = compute_input(v)
        vr = self._rescale(v, True)
        P = 3 * self.num_bins - 1
        cur = torch.zeros_like(vr)
        ld = None
        for i in range(self.dim):
            params = self.conditioner(cur, out_rows=(i * P, (i + 1) * P))
            cur, ld = ops.arqs_step(cur, vr, params, ld, i, self.num_bins, inverse)
        if ld is None:
            ld = torch.zeros(v.shape[0], dtype=torch.float32, device=v.device)
        return self._rescale(cur, False), ld

    def forward(self, z):
        return self._run(z, False)

    def inverse(self, x):
        return self._run(x, True)


USE_TENSOR_CORES = True      # tcgen05 stack kernels (3xTF32, fp32-accurate); False forces the FP32-pipe kernels


# family -> (tcgen05 packer, FP32-pipe packer, tcgen05 entry point, FP32-pipe entry point)
_STACKS = {"spline": (packing.pack_spline_stack_tc, packing.pack_spline_stack, "nf_spline_stack_tc", "nf_spline_stack"),
           "coupling": (packing.pack_coupling_stack_tc, packing.pack_coupling_stack, "nf_coupling_stack_tc",
                        "nf_coupling_stack"),
           # conditional layers: tcgen05 only, outside its envelope the layered route
           "spline_ctx": (packing.pack_spline_stack_ctx_tc, None, "nf_spline_stack_ctx_tc", None),
           "coupling_ctx": (packing.pack_coupling_stack_ctx_tc, None, "nf_coupling_stack_ctx_tc", None)}


def run_stack(family, cache: _PackCache, tensors, flows, bns, v, inverse, head=False, sample=None, ctx=None):
    """Spline-coupling or eval-mode affine coupling stack in one launch: the tcgen05 kernel when USE_TENSOR_CORES is set
    and the configuration fits it (spline: hidden_dim <= 64; affine: hidden_dim <= 128), the FP32-pipe kernel otherwise
    -- also when the tcgen05 launch refuses the configuration.  sample=(seed, offset): the in-kernel N(0, I) draw into v,
    returning (x, log_q) (see ops.stack).  ctx: the _Context of the conditional families "spline_ctx" and
    "coupling_ctx"."""
    pack_tc, pack, entry_tc, entry = _STACKS[family]

    def build():
        tcp = pack_tc(flows, bns) if USE_TENSOR_CORES else None
        return ("tc", tcp) if tcp is not None else ("simt", pack(flows, bns) if pack is not None else None)
    kind, pk = cache.get(tensors, build, extra=(USE_TENSOR_CORES,))
    if pk is None:
        return None
    if kind == "tc":
        out = ops.stack(entry_tc, pk[0], pk[1], v, inverse, head, sample,
                        context=None if ctx is None else (ctx.t, ctx.div))
        if out is not None or pack is None:
            return out
        pk = pack(flows, bns)
        if pk is None:
            return None
    return ops.stack(entry, pk[0], pk[1], v, inverse, head, sample)


# ------------------------------------------------------------------------------------------------
# whole-stack fusion used by the containers (SequentialFlow, models.NormalizingFlowModel)
# ------------------------------------------------------------------------------------------------
class ChainPlan:
    """Runs a homogeneous stack of coupling layers (+ optional between-layer BatchNorm affines on running
    statistics, normalizing_flow_model.py:25-128) as ONE kernel launch when no autograd graph is needed:
    a row is a few bytes, so keeping it in registers across all layers removes every intermediate HBM trip."""

    def __init__(self):
        self._pack = _PackCache()

    def run(self, flows, bns, training, v, inverse, head=False, sample=None, ctx=None):
        """(y, log_det) from one fused launch, or None when the chain must be walked layer by layer.
        head=True (inverse only): (None, log_prob) with the standard-normal Flow.log_prob head evaluated in the last
        layer's epilogue -- z is never written.
        sample=(seed, offset) (forward only): the sampling twin of the head -- v is the [n, D] output buffer, the rows are
        the N(0, I) draw of csrc/nf_rng.cuh made in the kernel, and the result is (x, log N(z) - log_det).
        ctx (a _Context): every layer must be a SplineCouplingLayer or CouplingLayer with that context width, float32
        context included."""
        flows = list(flows)
        v = compute_input(v)
        if not flows or not v.is_cuda or v.dim() != 2:
            return None
        if bns is not None and training:          # train mode moves the running statistics layer by layer
            return None
        kind = type(flows[0])
        made = kind in (MaskedAutoregressiveFlow, InverseAutoregressiveFlow)
        if not made and (kind not in (CouplingLayer, SplineCouplingLayer) or any(type(f) is not kind for f in flows)
                         or not all(f.fusable(v) for f in flows)):
            return None
        if ctx is not None and (made or ctx.t.dtype != torch.float32
                                or any(f.context_dim != ctx.t.shape[1] for f in flows)):
            return None
        mods = flows + (list(bns) if bns is not None else [])
        tensors = self._pack.tensors_of(mods)
        if torch.is_grad_enabled() and (v.requires_grad or any(t.requires_grad for t in tensors)
                                        or (ctx is not None and ctx.t.requires_grad)):
            return None
        if made:
            return self._run_made_stack(flows, bns, tensors, v, inverse, head, sample)
        return run_stack(flows[0]._stack, self._pack, tensors, flows, bns, v, inverse, head, sample, ctx)

    def _run_made_stack(self, flows, bns, tensors, v, inverse, head, sample):
        """Homogeneous MAF / IAF stack, hidden_dim <= 64, data_dim <= 8 (the sequential direction: data_dim == 2):
        one tcgen05 launch (made_stack_tc_kernel).  None -> the layers run one by one."""
        kind = type(flows[0])
        if not USE_TENSOR_CORES or any(type(f) is not kind for f in flows) or v.dtype != torch.float32:
            return None
        f0 = flows[0]
        D, H = f0.dim, f0.conditioner.hidden_dim
        if D > packing.DMAX or H > 64 or v.shape[1] != D:
            return None
        if any(f.dim != D or f.conditioner.hidden_dim != H or (f.conditioner.use_batch_norm and f.training)
               or f.conditioner.output_dim_multiplier != 2 for f in flows):
            return None
        parallel = (inverse == (kind is MaskedAutoregressiveFlow))      # MAF: density is the parallel pass; IAF: sampling
        if not parallel and D != 2:
            return None
        if head and not inverse:
            return None
        pk = self._pack.get(tensors, lambda: packing.pack_made_stack_tc(flows, bns), extra=("made_tc",))
        if pk is None:
            return None
        mode = f0._mode_parallel if parallel else f0._mode_sequential
        return ops.stack("nf_made_stack_tc", pk[0], pk[1], v, inverse, head, sample, (mode,))
