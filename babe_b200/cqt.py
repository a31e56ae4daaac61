"""``CQT_nsgt``: drop-in for the class the reference imports from the third-party
package ``cqt_nsgt_pytorch`` (networks/cqtdiff+.py:9,620 of eloimoliner/BABE),
running on the sm_100a kernels of ``csrc/cqt_ops.cu``.

Host side = plan construction only (band geometry, windows, duals, FFT
factorisation, twiddle tables; float64 numpy, once per instance).  ``fwd``,
``bwd`` and ``apply_hpf_DC`` are explicit ``torch.autograd.Function``
boundaries whose backward passes are the adjoint kernels (the synthesis kernel
with the analysis windows and vice versa), so the denoiser can be
differentiated through both transforms as testing/blind_bwe_sampler.py:120
requires.

The transform follows the specification in ``oracle/nsgt.py`` (PARITY
UNPINNED versus upstream: the upstream package is not available offline; see
DESIGN.md).  CUDA only -- no CPU fallback.
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib, profiling
from ._lib import BabeError, CqtPlan, FftFactors, check, lib

_RADIX_ORDER = (16, 8, 4, 2, 3, 5, 7, 11, 13, 17, 19, 23)
_TW_LO = 1024


def _factor(n):
    """Stage radices for the shared-memory Stockham FFT (csrc/smemfft.cuh)."""
    out, m = [], n
    for r in _RADIX_ORDER:
        while m % r == 0:
            out.append(r)
            m //= r
    if m != 1:
        raise BabeError(f"length {n} has a prime factor > 23 (unsupported)")
    if len(out) > _lib.MAX_FACTORS:
        raise BabeError(f"length {n} needs too many FFT stages")
    f = FftFactors()
    f.n, f.nf = n, len(out)
    for i, r in enumerate(out):
        f.radix[i] = r
    return f


def _split(nc):
    """n1 * n2 = nc, as square as possible (two shared-memory passes)."""
    best = None
    for d in range(1, int(math.isqrt(nc)) + 1):
        if nc % d == 0:
            best = d
    n1, n2 = nc // best, best
    if n1 > 1500:
        raise BabeError(f"segment length {2 * nc}: no balanced factorisation fits shared memory")
    return n1, n2


def _roots(n):
    m = np.arange(n, dtype=np.float64)
    w = np.exp(-2j * np.pi * m / n)
    return np.stack((w.real, w.imag), -1).astype(np.float32)


def _two_level(n):
    lo = np.exp(-2j * np.pi * np.arange(_TW_LO, dtype=np.float64) / n)
    hi = np.exp(-2j * np.pi * (_TW_LO * np.arange((n >> 10) + 1, dtype=np.float64)) / n)
    w = np.concatenate((lo, hi))
    return np.stack((w.real, w.imag), -1).astype(np.float32)


def _window(kind, L):
    i = np.arange(L, dtype=np.float64)
    if isinstance(kind, (tuple, list)) and kind[0] == "kaiser":
        r = 2.0 * i / L - 1.0
        return np.i0(float(kind[1]) * np.sqrt(np.clip(1.0 - r * r, 0.0, None))) / np.i0(float(kind[1]))
    if kind == "hann":
        return 0.5 - 0.5 * np.cos(2.0 * np.pi * i / L)
    if kind == "hamming":
        return 0.54 - 0.46 * np.cos(2.0 * np.pi * i / L)
    raise NotImplementedError(f"window {kind!r} (supported: ('kaiser', beta), 'hann', 'hamming')")


def _nextpow2(v):
    return 1 << max(0, int(math.ceil(math.log2(max(1, v)))))


class _Geometry:
    """Band layout of the octave-rasterised NSGT (specification: oracle/nsgt.py
    items 1-5, 7, 9)."""

    def __init__(self, numocts, binsoct, fs, Ls, window):
        K, Nc = numocts * binsoct, Ls // 2
        fmax = fs / 2 - 1e-6
        fmin = fmax / 2 ** numocts
        odiv = numocts / (K - 1)
        q = 2 ** (odiv / 2) / (2 ** odiv - 1) / 2
        fb = fmin * 2.0 ** (np.arange(K, dtype=np.float64) * odiv) * Ls / fs
        p = np.rint(fb).astype(np.int64)
        lg = np.maximum(4, np.rint(fb / q).astype(np.int64))
        p[K - 1] = int(np.rint((fb[K - 2] + Nc) / 2))
        lg[K - 1] = max(4, int(np.rint(Nc - fb[K - 2])))
        M = [_nextpow2(int(lg[o * binsoct:(o + 1) * binsoct].max())) for o in range(numocts)]
        for o in range(numocts - 2, -1, -1):
            M[o] = max(M[o], M[o + 1] // 2)
        for o in range(1, numocts):
            M[o] = max(M[o], 2 * M[o - 1])
        self.p, self.lg, self.M, self.K, self.Nc = p, lg, M, K, Nc
        self.off = np.concatenate(([0], np.cumsum(lg)[:-1])).astype(np.int64)
        self.sum_lg = int(lg.sum())
        Mband = np.repeat(np.asarray(M, dtype=np.float64), binsoct)
        # frame-operator diagonal over [0, Nc] (DC and Nyquist bands included)
        D = np.zeros(Nc + 1)
        bands = [(0, _window(window, max(4, 2 * int(p[0]))), float(max(4, 2 * int(p[0])))),
                 (Nc, _window(window, max(4, 2 * (Nc - int(p[K - 1])))), float(max(4, 2 * (Nc - int(p[K - 1])))))]
        g_all = []
        for j in range(K):
            gj = _window(window, int(lg[j]))
            g_all.append(gj)
            bands.append((int(p[j]), gj, Mband[j]))
        for centre, gj, Mj in bands:
            k = centre - len(gj) // 2 + np.arange(len(gj))
            ok = (k >= 0) & (k <= Nc)
            np.add.at(D, k[ok], Mj * gj[ok] ** 2)
        g = np.zeros(self.sum_lg)
        gd = np.zeros(self.sum_lg)
        hp = np.zeros(Nc + 1)
        mrep = np.zeros(self.sum_lg)
        for j in range(K):
            gj = g_all[j]
            k = int(p[j]) - int(lg[j]) // 2 + np.arange(int(lg[j]))
            ok = (k >= 0) & (k <= Nc)
            sl = slice(int(self.off[j]), int(self.off[j]) + int(lg[j]))
            gg = np.where(ok, gj, 0.0)
            dd = np.zeros_like(gj)
            dd[ok] = gj[ok] / D[k[ok]]
            g[sl], gd[sl], mrep[sl] = gg, dd, Mband[j]
            np.add.at(hp, k[ok], Mband[j] * gj[ok] * dd[ok])
        self.g, self.gd, self.mrep, self.Hhpf = g, gd, mrep, hp
        start = p - lg // 2
        end = start + lg
        if np.any(np.diff(start) < 0) or np.any(np.diff(end) < 0):
            raise BabeError("band windows are not monotone; unsupported configuration")
        k = np.arange(Nc + 1)
        self.jlo = np.searchsorted(end, k, side="right").astype(np.int32)       # first j with end_j > k
        self.jhi = (np.searchsorted(start, k, side="right") - 1).astype(np.int32)  # last j with start_j <= k
        # per-bin sources of the synthesis overlap-add: offsets into one row of band spectra, <= 3 bands per bin
        # (int4 entries, the fourth is unused)
        cover = int((self.jhi - self.jlo + 1).max())
        self.bin_src = None
        if cover <= 3:
            src = np.full((Nc + 1, 4), self.sum_lg, dtype=np.int32)    # sum_lg: the row's zero entry (no band)
            for s in range(cover):
                j = self.jlo.astype(np.int64) + s
                ok = j <= self.jhi
                jj = np.where(ok, j, 0)
                i = k - start[jj]
                ok &= (i >= 0) & (i < lg[jj])
                src[ok, s] = (self.off[jj] + i)[ok]
            self.bin_src = src


class _Plan:
    """Device tables + the ``babe_cqt_plan`` struct handed to the C ABI."""

    def __init__(self, geo, numocts, binsoct, Ls, device):
        self.device = torch.device(device)
        self.keep = []
        dev = lambda a: self._dev(a)
        Nc = Ls // 2
        n1, n2 = _split(Nc)
        plan = CqtPlan()
        plan.Ls, plan.Nc = Ls, Nc
        plan.f1, plan.f2 = _factor(n1), _factor(n2)
        plan.roots1, plan.roots2 = dev(_roots(n1)), dev(_roots(n2))
        plan.tw_nc, plan.tw_ls = dev(_two_level(Nc)), dev(_two_level(Ls))
        plan.numocts, plan.binsoct = numocts, binsoct
        for o in range(numocts):
            plan.M[o] = geo.M[o]
            plan.fm[o] = _factor(geo.M[o])
            plan.rootsm[o] = dev(_roots(geo.M[o]))
        plan.band_p = dev(geo.p.astype(np.int32))
        plan.band_lg = dev(geo.lg.astype(np.int32))
        plan.band_off = dev(geo.off.astype(np.int32))
        plan.sum_lg = geo.sum_lg
        plan.bin_jlo, plan.bin_jhi = dev(geo.jlo), dev(geo.jhi)
        plan.bin_src = dev(geo.bin_src) if geo.bin_src is not None else None
        self.c = plan
        self.n1, self.n2 = n1, n2
        self.coef_per_row = int(binsoct * sum(geo.M))
        f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(self.device)
        self.win_g = f32(geo.g)                             # analysis (fwd)
        self.win_gdM = f32(geo.gd * geo.mrep)               # synthesis (bwd)
        self.win_gM = f32(geo.g / geo.mrep)                 # backward of fwd
        self.win_gdMM = f32(geo.gd * geo.mrep * geo.mrep)   # backward of bwd
        self.Hhpf = f32(geo.Hhpf)
        self.Hlpf = f32(1.0 - geo.Hhpf)
        half = np.full(Nc + 1, 0.5)
        half[0] = half[-1] = 1.0
        self.scale_fwd_adj = f32(half * Ls)                 # Re(Ls * IFFT) as an irfft
        two = np.full(Nc + 1, 2.0)
        two[0] = two[-1] = 1.0
        self.scale_bwd_adj = f32(two / Ls)                  # adjoint of irfft
        self._ws = {}

    def _dev(self, arr):
        t = torch.from_numpy(np.ascontiguousarray(arr)).to(self.device)
        self.keep.append(t)
        return ctypes.c_void_p(t.data_ptr())

    def workspace(self, rows):
        n = lib().babe_cqt_workspace(ctypes.byref(self.c), int(rows))
        # one scratch buffer per batch size, reused across calls on the same stream
        buf = self._ws.get(rows)
        if buf is None or buf.numel() * 4 < n:
            buf = torch.empty((n + 3) // 4, dtype=torch.float32, device=self.device)
            self._ws[rows] = buf            # never drop a buffer: a captured CUDA graph may hold its address
        return buf, n


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _analysis(plan, x, win, scale, planar=False):
    rows = x.shape[0]
    if planar:
        outs = [torch.empty((rows, 2, plan.c.binsoct, plan.c.M[o]), dtype=torch.float32, device=x.device)
                for o in range(plan.c.numocts)]
    else:
        outs = [torch.empty((rows, plan.c.binsoct, plan.c.M[o]), dtype=torch.complex64, device=x.device)
                for o in range(plan.c.numocts)]
    ptrs = (ctypes.c_void_p * plan.c.numocts)(*[o.data_ptr() for o in outs])
    ws, n = plan.workspace(rows)
    # algorithmic bytes (SURVEY 8d): read x, write the complex coefficients
    with profiling.op("cqt_analysis", 4, rows * (4 * plan.c.Ls + 8 * plan.coef_per_row)):
        check(lib().babe_cqt_analysis(ctypes.byref(plan.c), _p(x), ptrs, int(planar), rows, _p(win), _p(scale),
                                      _p(ws), n, _stream()), "cqt_analysis")
    return outs


def _synthesis(plan, cs, win, scale, planar=False):
    rows = cs[0].shape[0]
    cs = [c.contiguous() for c in cs]
    x = torch.empty((rows, plan.c.Ls), dtype=torch.float32, device=cs[0].device)
    ptrs = (ctypes.c_void_p * plan.c.numocts)(*[c.data_ptr() for c in cs])
    ws, n = plan.workspace(rows)
    with profiling.op("cqt_synthesis", 4, rows * (4 * plan.c.Ls + 8 * plan.coef_per_row)):
        check(lib().babe_cqt_synthesis(ctypes.byref(plan.c), ptrs, int(planar), _p(x), rows, _p(win), _p(scale),
                                       _p(ws), n, _stream()), "cqt_synthesis")
    return x


def _spectral(plan, x, H):
    rows = x.shape[0]
    y = torch.empty_like(x)
    ws, n = plan.workspace(rows)
    with profiling.op("spectral_filter", 5, rows * 8 * plan.c.Ls):
        check(lib().babe_spectral_filter(ctypes.byref(plan.c), _p(x), _p(y), rows, _p(H), _p(ws), n,
                                         _stream()), "spectral_filter")
    return y


class _CqtFwd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, plan):
        ctx.plan, ctx.rows = plan, x.shape[0]
        return tuple(_analysis(plan, x, plan.win_g, None))

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *gcs):
        plan = ctx.plan
        gcs = [g if g is not None else
               torch.zeros((ctx.rows, plan.c.binsoct, plan.c.M[o]), dtype=torch.complex64, device=plan.device)
               for o, g in enumerate(gcs)]
        return _synthesis(plan, gcs, plan.win_gM, plan.scale_fwd_adj), None


class _CqtBwd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, plan, *cs):
        ctx.plan = plan
        return _synthesis(plan, list(cs), plan.win_gdM, None)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        plan = ctx.plan
        return (None, *_analysis(plan, g.contiguous(), plan.win_gdMM, plan.scale_bwd_adj))


class _CqtFwdPlanar(torch.autograd.Function):
    """fwd with real (B,2,binsoct,T_o) outputs; the gradient of a real plane pair is the same
    complex cotangent (dL/dRe + i dL/dIm), so the backward is the planar synthesis with g/M."""

    @staticmethod
    def forward(ctx, x, plan):
        ctx.plan, ctx.rows = plan, x.shape[0]
        return tuple(_analysis(plan, x, plan.win_g, None, planar=True))

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *gcs):
        plan = ctx.plan
        gcs = [g if g is not None else
               torch.zeros((ctx.rows, 2, plan.c.binsoct, plan.c.M[o]), dtype=torch.float32, device=plan.device)
               for o, g in enumerate(gcs)]
        return _synthesis(plan, gcs, plan.win_gM, plan.scale_fwd_adj, planar=True), None


class _CqtBwdPlanar(torch.autograd.Function):
    @staticmethod
    def forward(ctx, plan, *cs):
        ctx.plan = plan
        return _synthesis(plan, list(cs), plan.win_gdM, None, planar=True)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        plan = ctx.plan
        return (None, *_analysis(plan, g.contiguous(), plan.win_gdMM, plan.scale_bwd_adj, planar=True))


class _SpectralFilter(torch.autograd.Function):
    """irfft(rfft(x) H) with real H: symmetric, hence its own adjoint."""

    @staticmethod
    def forward(ctx, x, plan, H):
        ctx.plan, ctx.H = plan, H
        return _spectral(plan, x, H)

    @staticmethod
    def backward(ctx, g):
        return _SpectralFilter.apply(g.contiguous(), ctx.plan, ctx.H), None, None


class CQT_nsgt:
    """Invertible octave-rasterised constant-Q transform.

    Constructor as called at networks/cqtdiff+.py:620:
    ``CQT_nsgt(numocts, binsoct, mode="oct", window=("kaiser", beta), fs=...,
    audio_len=..., dtype=torch.float32, device=...)``.
    """

    def __init__(self, numocts, binsoct, mode="oct", window="hann", flex_Q=None, fs=44100,
                 audio_len=44100, device="cuda", dtype=torch.float32):
        if mode != "oct":
            raise NotImplementedError(f"mode {mode!r}: only 'oct' (the mode the reference uses, "
                                      "networks/cqtdiff+.py:620) is implemented")
        if dtype != torch.float32:
            raise NotImplementedError("float32 only")
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        if device.type != "cuda":
            raise BabeError(f"CQT_nsgt on {device}: babe_b200 runs on CUDA only (no CPU fallback)")
        if audio_len % 2 != 0:
            raise BabeError("odd audio_len is unsupported")
        if numocts > _lib.MAX_OCTAVES:
            raise BabeError(f"numocts > {_lib.MAX_OCTAVES}")
        self.numocts, self.binsoct, self.mode, self.fs, self.Ls = numocts, binsoct, mode, fs, audio_len
        self.device, self.dtype = device, dtype
        self.geometry = _Geometry(numocts, binsoct, fs, audio_len, window)
        self.size_per_oct = list(self.geometry.M)
        self.plan = _Plan(self.geometry, numocts, binsoct, audio_len, device)

    def _rows(self, x):
        if not (torch.is_tensor(x) and x.is_cuda and x.dtype == torch.float32):
            raise BabeError("CQT_nsgt expects CUDA float32 tensors")
        if x.device != self.device or x.device.index not in (None, torch.cuda.current_device()):
            raise BabeError(f"input on {x.device}, plan on {self.device}, current device "
                            f"cuda:{torch.cuda.current_device()}: they must agree")
        if x.shape[-1] != self.Ls:
            raise ValueError(f"input length {x.shape[-1]} != audio_len {self.Ls}")
        rows = x.reshape(-1, self.Ls).contiguous()
        # the kernels read the rows as float2 / float4: a contiguous view at an odd float offset (a slice of a longer
        # buffer) is copied into fresh, aligned storage
        return rows if rows.data_ptr() % 16 == 0 else rows.clone()

    def fwd(self, x):
        """x (B,C,T) -> list of numocts complex64 tensors (B,C,binsoct,T_o),
        lowest octave first, T_{o+1} = 2 T_o (networks/cqtdiff+.py:743,750)."""
        lead = x.shape[:-1]
        outs = _CqtFwd.apply(self._rows(x), self.plan)
        return [o.reshape(*lead, self.binsoct, o.shape[-1]) for o in outs]

    def bwd(self, cs):
        """list of (B,C,binsoct,T_o) complex64 -> (B,C,audio_len) (networks/cqtdiff+.py:841)."""
        if len(cs) != self.numocts:
            raise ValueError(f"expected {self.numocts} octaves")
        lead = cs[0].shape[:-2]
        flat = []
        for o, c in enumerate(cs):
            if not (c.is_cuda and c.dtype == torch.complex64):
                raise BabeError("CQT_nsgt.bwd expects CUDA complex64 tensors")
            if c.shape[-2:] != (self.binsoct, self.size_per_oct[o]):
                raise ValueError(f"octave {o}: shape {tuple(c.shape)}")
            flat.append(c.reshape(-1, self.binsoct, self.size_per_oct[o]).contiguous())
        return _CqtBwd.apply(self.plan, *flat).reshape(*lead, self.Ls)

    def fwd_planar(self, x):
        """x (B,T) -> list of float32 (B,2,binsoct,T_o): exactly the tensors the denoiser builds from
        ``fwd`` with view_as_real/permute/contiguous (networks/cqtdiff+.py:750-753), written directly."""
        return list(_CqtFwdPlanar.apply(self._rows(x), self.plan))

    def bwd_planar(self, cs):
        """list of float32 (B,2,binsoct,T_o) -> (B,audio_len); replaces the permute/contiguous/
        view_as_complex of networks/cqtdiff+.py:826-830 followed by ``bwd``."""
        flat = []
        for o, c in enumerate(cs):
            if c.shape[1:] != (2, self.binsoct, self.size_per_oct[o]) or c.dtype != torch.float32 or not c.is_cuda:
                raise ValueError(f"octave {o}: expected CUDA float32 (B,2,{self.binsoct},{self.size_per_oct[o]})")
            flat.append(c.contiguous())
        return _CqtBwdPlanar.apply(self.plan, *flat)

    # upstream names
    nsgtf = fwd
    nsigtf = bwd

    def apply_hpf_DC(self, x):
        """Remove what the DC and Nyquist bands carry ("oct" mode discards
        them): irfft(rfft(x) Hhpf) (testing/blind_bwe_sampler.py:156)."""
        return _SpectralFilter.apply(self._rows(x), self.plan, self.plan.Hhpf).reshape(x.shape)

    def apply_lpf_DC(self, x):
        return _SpectralFilter.apply(self._rows(x), self.plan, self.plan.Hlpf).reshape(x.shape)

    # raw transforms (used by the tests / benchmarks)
    def rfft(self, x):
        rows = self._rows(x)
        X = torch.empty((rows.shape[0], self.Ls // 2 + 1), dtype=torch.complex64, device=rows.device)
        ws, n = self.plan.workspace(rows.shape[0])
        check(lib().babe_rfft(ctypes.byref(self.plan.c), _p(rows), _p(X), rows.shape[0], None, _p(ws), n,
                              _stream()), "rfft")
        return X

    def irfft(self, X):
        X = X.contiguous()
        x = torch.empty((X.shape[0], self.Ls), dtype=torch.float32, device=X.device)
        ws, n = self.plan.workspace(X.shape[0])
        check(lib().babe_irfft(ctypes.byref(self.plan.c), _p(X), _p(x), X.shape[0], None, _p(ws), n,
                               _stream()), "irfft")
        return x
