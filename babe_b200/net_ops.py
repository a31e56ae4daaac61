"""Fused element-wise glue of the CQTDiff+ residual layers (csrc/net_ops.cu) behind
``torch.autograd.Function`` boundaries.

One dilated-convolution layer of ``ResnetBlock.forward`` (networks/cqtdiff+.py:470-482)

    x -> (x + conv(gelu(norm(x) * (affine(sigma) + 1))) * gate(sigma)) / sqrt(2)

is ~8 PyTorch kernels forward and ~16 backward around the convolution, most of them
non-vectorised broadcast multiplies (45 % of the sampler step in the round-1 launch
list).  Here it is 3 launches forward and 3 backward around the cuDNN convolution;
only the layer input is saved for the backward pass.  Gradients are produced for the
activations only: the functions are used when the parameters are frozen (sampling);
``denoiser.py`` falls back to the composite PyTorch expression otherwise.
"""
import ctypes
import weakref

import torch
import torch.nn.functional as F

from . import profiling
from ._lib import check, lib

RSQRT2 = 0.7071067811865476


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


# Arrival counters of the kernels whose last CTA finishes a group's statistics: one per (n, group), zero
# between calls (every kernel resets the ones it used).  N * G <= N * C <= 65535 (``usable``).  Calls
# sharing counters must not overlap, so there is one buffer per (device, stream): kernels on one stream
# run in order, and two streams never count on the same buffer.
_COUNTERS = {}


def _counters(device):
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    c = _COUNTERS.get(key)
    if c is None:
        c = _COUNTERS[key] = torch.zeros(65536, dtype=torch.int32, device=device)
    return c


def gn_stats(x, groups):
    """Finished statistics {mean, std} of every (sample, group) of x, and the number of partial slices
    they were summed from."""
    N, C, Fd, T = x.shape
    P = Fd * T
    S = lib().babe_gn_slices(N, C, groups, P)
    part = torch.empty(N * groups * S * 2, dtype=torch.float64, device=x.device)
    stats = torch.empty(N * groups, 2, dtype=torch.float32, device=x.device)
    with profiling.op("gn_stats", 1, 4 * x.numel()):
        check(lib().babe_gn_stats(_p(x), _p(part), _p(stats), _p(_counters(x.device)), N, C, groups, P, S,
                                  _stream()), "gn_stats")
    return stats, S


def gn_film_gelu(x, stats, S, gamma, aff, groups, eps):
    """``(stats, S)``: what gn_stats (or gate_residual with ``groups``) returned.  The record is finished and
    no kernel reads S; it stays in the tuple so that the four glue wrappers keep their positional
    signatures (tests/test_net_ops_plumbing_cpu.py substitutes them by position)."""
    N, C, Fd, T = x.shape
    h = torch.empty_like(x)
    with profiling.op("gn_film_gelu", 1, 8 * x.numel()):
        check(lib().babe_gn_film_gelu(_p(x), _p(h), _p(stats), _p(gamma), _p(aff), N, C, groups,
                                      Fd * T, eps, _stream()), "gn_film_gelu")
    return h


def gate_residual(x0, v, gate, scale=RSQRT2, *, groups=None):
    """(x0 + v * gate[n,c]) * scale; ``x0`` and ``gate`` may be None.  With ``groups``: also the group
    statistics of the result, returned as ``out, (stats, S)`` like gn_stats(out, groups)."""
    N, C, Fd, T = v.shape
    P = Fd * T
    out = torch.empty_like(v)
    with profiling.op("gate_residual", 1, (8 if x0 is None else 12) * v.numel()):
        if groups is None:
            check(lib().babe_gate_residual(_p(x0), _p(v), _p(gate), _p(out), N, C, P, scale, _stream()),
                  "gate_residual")
            return out
        S = C // groups * lib().babe_net_chunks(P)
        part = torch.empty(N * groups * S * 2, dtype=torch.float64, device=v.device)
        stats = torch.empty(N * groups, 2, dtype=torch.float32, device=v.device)
        check(lib().babe_gate_residual_stats(_p(x0), _p(v), _p(gate), _p(out), _p(part), _p(stats),
                                             _p(_counters(v.device)), N, C, groups, P, scale, _stream()),
              "gate_residual")
    return out, (stats, S)


def gn_film_gelu_bwd(gh, x, gy, stats, S, gamma, aff, groups, eps, res_scale=RSQRT2, *, gate_prev=None):
    """g_x of the layer (``gy`` may be None).  With ``gate_prev``: returns ``gx, gv`` where
    gv = gate_residual(None, gx, gate_prev, res_scale) comes from the same kernel."""
    N, C, Fd, T = x.shape
    P = Fd * T
    scratch = torch.empty(N * C * lib().babe_net_chunks(P), dtype=torch.float64, device=x.device)
    coef = torch.empty(N * groups, dtype=torch.float32, device=x.device)
    gx = torch.empty_like(x)
    gv = torch.empty_like(x) if gate_prev is not None else None
    with profiling.op("gn_bwd_reduce", 1, 8 * x.numel()):
        check(lib().babe_gn_film_gelu_bwd_reduce(_p(gh), _p(x), _p(stats), _p(scratch), _p(coef),
                                                 _p(_counters(x.device)), _p(gamma), _p(aff), N, C, groups, P,
                                                 eps, _stream()), "gn_bwd_reduce")
    nbytes = (16 if gy is not None else 12) + (4 if gv is not None else 0)
    with profiling.op("gn_film_gelu_bwd", 1, nbytes * x.numel()):
        check(lib().babe_gn_film_gelu_bwd(_p(gh), _p(x), _p(gy), _p(gx), _p(stats), _p(coef), _p(gamma), _p(aff),
                                          _p(gate_prev), _p(gv), N, C, groups, P, eps, res_scale, _stream()),
              "gn_film_gelu_bwd")
    return gx if gv is None else (gx, gv)


def _same_padding(weight, dilation):
    kh, kw = weight.shape[-2:]
    if kh % 2 == 0 or kw % 2 == 0:
        raise ValueError("fused residual layer needs odd kernel sizes")
    return (dilation[0] * (kh - 1) // 2, dilation[1] * (kw - 1) // 2)


def _rows(t, N, C):
    t = t.detach().reshape(-1, C)
    if t.shape[0] != N:
        t = t.expand(N, C)
    return t.contiguous().float()


# ---------------------------------------------------------------------------
# The stride-1 "same" convolution y = conv(h, W) can be evaluated by cuDNN either as a forward
# convolution or as the input-gradient of the convolution with W' = W^T flipped -- the same
# sums in a different kernel.  Which is faster depends on the shape (at 8 x 256 x 448 x 32 the
# dgrad kernel takes 0.39 ms and the fprop kernel 0.99 ms on B200, at 8 x 64 x 64 x 2048 they
# are equal), so both are timed once per (shape, dilation) and the faster one is kept.
# ---------------------------------------------------------------------------
_FLIPPED = {}          # id(weight object) -> (weakref to it, its version, flipped-transposed copy)
_CONV_CHOICE = {}
AUTOTUNE_CONV = True


def _flipped(weight):
    """W^T flipped for ``weight`` (the caller's persistent tensor object, e.g. the nn.Parameter), cached
    per OBJECT: the entry is valid while that very object is alive and its version counter unchanged,
    and is dropped when the object dies -- a recycled address or id can never return a stale copy."""
    k = id(weight)
    ent = _FLIPPED.get(k)
    if ent is not None and ent[0]() is weight and ent[1] == weight._version:
        return ent[2]
    flipped = weight.detach().transpose(0, 1).flip(2, 3).contiguous()

    def _drop(_, k=k):
        _FLIPPED.pop(k, None)
    _FLIPPED[k] = (weakref.ref(weight, _drop), weight._version, flipped)
    return flipped


def _time(fn):
    fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    fn()
    fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e)


def conv_same(inp, weight, pad, dilation, transposed=False, wobj=None):
    """transposed=False: conv2d(inp, weight); True: its input-gradient for grad_output = inp.
    ``wobj``: the persistent tensor object ``weight`` was detached from (cache key of the flipped copy)."""
    wobj = weight if wobj is None else wobj
    if transposed:
        size = (inp.shape[0], weight.shape[1], inp.shape[2], inp.shape[3])
        direct = lambda: torch.nn.grad.conv2d_input(size, weight, inp, 1, pad, dilation)
        other = lambda: F.conv2d(inp, _flipped(wobj), None, 1, pad, dilation)
    else:
        size = (inp.shape[0], weight.shape[0], inp.shape[2], inp.shape[3])
        direct = lambda: F.conv2d(inp, weight, None, 1, pad, dilation)
        other = lambda: torch.nn.grad.conv2d_input(size, _flipped(wobj), inp, 1, pad, dilation)
    if not AUTOTUNE_CONV:
        return direct()
    key = (tuple(inp.shape), tuple(weight.shape), tuple(dilation), transposed, inp.device.index)
    choice = _CONV_CHOICE.get(key)
    if choice is None:
        choice = 0 if _time(direct) <= _time(other) else 1
        _CONV_CHOICE[key] = choice
    return direct() if choice == 0 else other()


class _ResChain(torch.autograd.Function):
    """The dilated layers of one ResnetBlock in sequence.  Each layer's output carries the statistics the
    next layer normalises with (gate_residual with ``groups``), and in the backward pass each layer's g_x
    kernel also writes g_v of the layer before it (gn_film_gelu_bwd with ``gate_prev``), so only the first
    layer reads its input for statistics and only the last one has a separate g_v pass.  Saved: every
    layer's input and statistics record."""

    @staticmethod
    def forward(ctx, x, layers, groups, eps):
        x = x.contiguous()
        N, C = x.shape[:2]
        cfg = []
        stats = gn_stats(x, groups)
        xs, recs = [], []
        for i, (gamma, aff, gate, weight, dilation) in enumerate(layers):
            gamma = gamma.detach().reshape(-1).contiguous().float()
            aff, gate = _rows(aff, N, C), _rows(gate, N, C)
            wobj, weight = weight, weight.detach()
            pad = _same_padding(weight, dilation)
            h = gn_film_gelu(x, *stats, gamma, aff, groups, eps)
            v = conv_same(h, weight, pad, dilation, wobj=wobj)
            del h
            xs.append(x)
            recs.append(stats)
            if i + 1 < len(layers):
                x, stats = gate_residual(x, v, gate, groups=groups)
            else:
                x = gate_residual(x, v, gate)
            # the caller's weight object: key of the flipped-copy cache
            cfg.append((gamma, aff, gate, weight, wobj, pad, dilation))
        ctx.save_for_backward(*xs, *(st for st, _ in recs))
        ctx.slices = [S for _, S in recs]
        ctx.cfg = (cfg, groups, eps)
        return x

    @staticmethod
    def backward(ctx, gy):
        cfg, groups, eps = ctx.cfg
        n = len(cfg)
        saved = ctx.saved_tensors
        gy = gy.contiguous()
        gv = gate_residual(None, gy, cfg[-1][2])
        for i in range(n - 1, -1, -1):
            gamma, aff, gate, weight, wobj, pad, dilation = cfg[i]
            gh = conv_same(gv, weight, pad, dilation, transposed=True, wobj=wobj).contiguous()
            del gv
            rec = (saved[n + i], ctx.slices[i])
            if i > 0:
                gy, gv = gn_film_gelu_bwd(gh, saved[i], gy, *rec, gamma, aff, groups, eps, gate_prev=cfg[i - 1][2])
            else:
                gy = gn_film_gelu_bwd(gh, saved[i], gy, *rec, gamma, aff, groups, eps)
            del gh
        return gy, None, None, None


class _ConvSame(torch.autograd.Function):
    """Bias-free stride-1 "same" convolution with a frozen weight: both directions go through
    ``conv_same`` (the faster of cuDNN's two formulations per shape)."""

    @staticmethod
    def forward(ctx, x, weight, dilation):
        wobj, weight = weight, weight.detach()
        pad = _same_padding(weight, dilation)
        ctx.save_for_backward(weight)
        ctx.cfg = (dilation, pad)
        ctx.wobj = wobj
        return conv_same(x.contiguous(), weight, pad, dilation, wobj=wobj)

    @staticmethod
    def backward(ctx, g):
        weight, = ctx.saved_tensors
        dilation, pad = ctx.cfg
        return conv_same(g.contiguous(), weight, pad, dilation, transposed=True, wobj=ctx.wobj), None, None


def _pair(d):
    return (d, d) if isinstance(d, int) else tuple(d)


def conv_frozen(x, weight, dilation):
    return _ConvSame.apply(x, weight, _pair(dilation))


class _AddScale(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b):
        return gate_residual(a.contiguous(), b.contiguous(), None)

    @staticmethod
    def backward(ctx, g):
        g = gate_residual(None, g.contiguous(), None)
        return g, g


def _frozen(*ts):
    return not (torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in ts))


def usable(x, *params):
    """The fused path applies to CUDA float32 activations with frozen parameters."""
    return (x.is_cuda and x.dtype == torch.float32 and x.dim() == 4 and _frozen(*params)
            and x.shape[0] * x.shape[1] <= 65535)          # one grid row per (n, c) plane


def res_layer(x, gamma, aff, gate, weight, dilation, groups, eps):
    """(x + conv(gelu(groupnorm(x) * gamma * (aff + 1))) * gate) / sqrt(2), conv with "same" padding."""
    return _ResChain.apply(x, ((gamma, aff, gate, weight, _pair(dilation)),), groups, eps)


def res_chain(x, layers, groups, eps):
    """res_layer applied in turn for every (gamma, aff, gate, weight, dilation) of ``layers``."""
    return _ResChain.apply(x, tuple((g, a, t, w, _pair(d)) for g, a, t, w, d in layers), groups, eps)


def add_scale(a, b):
    """(a + b) / sqrt(2)"""
    return _AddScale.apply(a, b)


# ---------------------------------------------------------------------------
# x2 anti-aliased time resampling (UpDownResample, networks/cqtdiff+.py:522-580)
# ---------------------------------------------------------------------------
def _resample(x, taps, mode):
    """mode 0 down / 1 up / 2 gradient of down / 3 gradient of up, along the last axis."""
    x = x.contiguous()
    Tin = x.shape[-1]
    T = {0: Tin, 1: Tin, 2: 2 * Tin, 3: Tin // 2}[mode]          # x-side row length
    Tout = {0: T // 2, 1: 2 * T, 2: T, 3: T}[mode]
    rows = x.numel() // Tin
    out = torch.empty(*x.shape[:-1], Tout, dtype=x.dtype, device=x.device)
    w = (ctypes.c_float * len(taps))(*taps)
    with profiling.op("resample2", 1, 4 * (x.numel() + out.numel())):
        check(lib().babe_resample2(_p(x), _p(out), rows, T, mode, w, len(taps), _stream()), "resample2")
    return out


class _Resample(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, taps, up):
        ctx.taps, ctx.up = taps, up
        return _resample(x, taps, 1 if up else 0)

    @staticmethod
    def backward(ctx, g):
        return _resample(g, ctx.taps, 3 if ctx.up else 2), None, None


def resample2(x, taps, up):
    """UpDownResample.forward for mode "T": x[..., T] -> [..., 2T] (up) or [..., T/2] (down)."""
    return _Resample.apply(x, tuple(float(t) for t in taps), bool(up))
