"""Tensor-level wrappers around the C ABI (no autograd here).

Every function takes and returns CUDA float32 tensors, launches on torch's
current stream and raises on any failure.  PyTorch only owns the memory and
the stream; all arithmetic happens in the sm_100a kernels of
``babe_b200/csrc``.
"""
import ctypes

import numpy as np
import torch

from . import _lib, profiling
from ._lib import BabeError, FitConfig, check, lib

_TABLES = {}


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _cuda_f32(t, name):
    if not torch.is_tensor(t):
        raise TypeError(f"{name} must be a tensor")
    if not t.is_cuda:
        raise BabeError(f"{name} is on {t.device}: babe_b200 runs on CUDA tensors only "
                        "(there is no CPU fallback)")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    if t.device.index != torch.cuda.current_device():
        raise BabeError(f"{name} is on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
                        "kernels launch on the current device -- call torch.cuda.set_device first")
    return t.detach().contiguous()


def _filter_out(out, x):
    """The output tensor of the filter ops: new, or ``out`` once it is known to hold exactly x's B * T floats (the
    kernels write them from its base pointer, so a smaller, strided or other-typed ``out`` would be overrun)."""
    if out is None:
        return torch.empty_like(x)
    if not (torch.is_tensor(out) and out.is_cuda and out.dtype == torch.float32 and out.device == x.device
            and out.shape == x.shape and out.is_contiguous()):
        what = f"{out.dtype} {tuple(out.shape)} on {out.device}" if torch.is_tensor(out) else type(out).__name__
        raise ValueError(f"out must be a contiguous float32 tensor of shape {tuple(x.shape)} on {x.device}, got {what}")
    return out


def num_frames(T, nfft):
    """utils/blind_bwe_utils.py:22-23: padded by NFFT, hop NFFT/2, center=False."""
    return 1 + T // (nfft // 2)


def stft_tables(nfft, device):
    """(window, twiddle) device tensors for one NFFT, cached per device.
    The window is ``torch.hamming_window`` itself, i.e. bit-identical to the
    one the reference builds at utils/blind_bwe_utils.py:19."""
    key = (int(nfft), torch.device(device).index if torch.device(device).index is not None
           else torch.cuda.current_device())
    if key not in _TABLES:
        if not lib().babe_stft_supported(int(nfft)):
            raise BabeError(f"unsupported NFFT {nfft} (supported: 512, 1024, 2048, 4096)")
        win = np.empty(nfft, dtype=np.float32)
        tw = np.empty(2 * nfft, dtype=np.float32)
        check(lib().babe_stft_tables_host(int(nfft), win.ctypes.data, tw.ctypes.data), "stft_tables")
        window = torch.hamming_window(window_length=nfft).to(device)
        _TABLES[key] = (window, torch.from_numpy(tw).to(device))
    return _TABLES[key]


# ---------------------------------------------------------------------------
def design_filter(fc, A, freqs, gain_db=None, strict=True):
    """H[F] from breakpoints fc[K], A[K] (device tensors).  strict=True checks
    the device status word (one sync) and raises IndexError exactly when the
    reference does (utils/blind_bwe_utils.py:111)."""
    fc = _cuda_f32(fc, "fc").reshape(-1)
    A = _cuda_f32(A, "A").reshape(-1)
    freqs = _cuda_f32(freqs, "f")
    if fc.numel() != A.numel():
        raise ValueError("fc and A must have the same number of breakpoints")
    g = None if gain_db is None else _cuda_f32(gain_db, "G").reshape(-1)
    H = torch.empty_like(freqs)
    status = torch.zeros(1, dtype=torch.int32, device=freqs.device) if strict else None
    with profiling.op("design_filter", 1, 8 * freqs.numel()):
        check(lib().babe_design_filter(_p(fc), _p(A), fc.numel(), _p(g), _p(freqs), freqs.numel(),
                                       _p(H), _p(status), _stream()), "design_filter")
    if strict and int(status.item()) != 0:
        raise IndexError("index 0 is out of bounds for dimension 0 with size 0")
    return H


def design_filter_vjp(fc, A, freqs, gH, gain_db=None):
    fc = _cuda_f32(fc, "fc").reshape(-1)
    A = _cuda_f32(A, "A").reshape(-1)
    freqs = _cuda_f32(freqs, "f")
    gH = _cuda_f32(gH, "gH")
    g = None if gain_db is None else _cuda_f32(gain_db, "G").reshape(-1)
    gfc = torch.empty_like(fc)
    gA = torch.empty_like(A)
    gg = torch.empty(1, dtype=torch.float32, device=fc.device) if g is not None else None
    with profiling.op("design_filter_vjp", 1, 8 * freqs.numel()):
        check(lib().babe_design_filter_vjp(_p(fc), _p(A), fc.numel(), _p(g), _p(freqs), freqs.numel(),
                                           _p(gH), _p(gfc), _p(gA), _p(gg), _stream()),
              "design_filter_vjp")
    return gfc, gA, gg


def apply_filter(x, nfft, H=None, freqs=None, fc=None, A=None, adjoint=False, sub=None,
                 row_scale=None, row_sumsq=None, out=None):
    """Fused STFT -> H -> iSTFT on x[B,T].  Pass either H[F] or (freqs, fc, A)."""
    x = _cuda_f32(x, "x")
    if x.dim() != 2:
        raise ValueError("x must be (B, T)")
    B, T = x.shape
    win, tw = stft_tables(nfft, x.device)
    K = 0
    if H is not None:
        H = _cuda_f32(H, "H")
        if H.numel() != nfft // 2 + 1:
            raise ValueError(f"H must have {nfft // 2 + 1} bins, got {H.numel()}")
    else:
        freqs = _cuda_f32(freqs, "f")
        fc = _cuda_f32(fc, "fc").reshape(-1)
        A = _cuda_f32(A, "A").reshape(-1)
        K = fc.numel()
        if freqs.numel() != nfft // 2 + 1 or A.numel() != K:
            raise ValueError("bad filter parameter shapes")
    if sub is not None:
        sub = _cuda_f32(sub, "sub")
        if sub.shape != x.shape:
            raise ValueError("sub must match x")
    if row_scale is not None:
        row_scale = _cuda_f32(row_scale, "row_scale")
        if row_scale.numel() != B:
            raise ValueError("row_scale must have B entries")
    if row_sumsq is not None and (row_sumsq.dtype != torch.float64 or row_sumsq.numel() != B):
        raise ValueError("row_sumsq must be float64[B]")
    y = _filter_out(out, x)
    ws, nbytes = None, 0
    if row_sumsq is not None:
        nbytes = lib().babe_apply_filter_workspace(B, T, int(nfft))
        ws = torch.empty(nbytes // 8, dtype=torch.float64, device=x.device)
    # algorithmic bytes (SURVEY 8d): read x, write y (+ read sub)
    with profiling.op("apply_filter_adj" if adjoint else "apply_filter", 2 if row_sumsq is not None else 1,
                      (12 if sub is not None else 8) * B * T):
        check(lib().babe_apply_filter(_p(x), _p(y), B, T, int(nfft), _p(win), _p(tw), _p(H), _p(freqs),
                                      _p(fc), _p(A), K, int(bool(adjoint)), _p(sub), _p(row_scale),
                                      _p(row_sumsq), _p(ws), nbytes, None, _stream()), "apply_filter")
    return y


def _row_params(x, fc, A):
    """Shape checks of the per-row filter parameters: fc, A (B, K) with the B of x (B, T)."""
    if not (torch.is_tensor(x) and torch.is_tensor(fc) and torch.is_tensor(A)):
        raise TypeError("x, fc and A must be tensors")
    if x.dim() != 2:
        raise ValueError("x must be (B, T)")
    if fc.dim() != 2 or A.shape != fc.shape or fc.shape[0] != x.shape[0]:
        raise ValueError(f"fc and A must both be (B, K) with B = {x.shape[0]} rows of x, got "
                         f"{tuple(fc.shape)} and {tuple(A.shape)}")


def apply_filter_rows(x, nfft, freqs, fc, A, adjoint=False, sub=None, row_scale=None, row_sumsq=None, out=None,
                      status=None):
    """``apply_filter`` with one filter per row: row b of x[B,T] goes through the H designed from fc[b], A[b]
    (fc, A: (B, K)).  ``status`` (optional int32[B]) flags the rows whose design the reference would reject."""
    _row_params(x, fc, A)
    x = _cuda_f32(x, "x")
    fc = _cuda_f32(fc, "fc")
    A = _cuda_f32(A, "A")
    freqs = _cuda_f32(freqs, "f")
    B, T = x.shape
    K = fc.shape[1]
    if freqs.numel() != nfft // 2 + 1:
        raise ValueError(f"freqs must have {nfft // 2 + 1} bins, got {freqs.numel()}")
    win, tw = stft_tables(nfft, x.device)
    if sub is not None:
        sub = _cuda_f32(sub, "sub")
        if sub.shape != x.shape:
            raise ValueError("sub must match x")
    if row_scale is not None:
        row_scale = _cuda_f32(row_scale, "row_scale")
        if row_scale.numel() != B:
            raise ValueError("row_scale must have B entries")
    if row_sumsq is not None and (row_sumsq.dtype != torch.float64 or row_sumsq.numel() != B):
        raise ValueError("row_sumsq must be float64[B]")
    if status is not None and (status.dtype != torch.int32 or status.numel() != B):
        raise ValueError("status must be int32[B]")
    y = _filter_out(out, x)
    ws, nbytes = None, 0
    if row_sumsq is not None:
        nbytes = lib().babe_apply_filter_workspace(B, T, int(nfft))
        ws = torch.empty(nbytes // 8, dtype=torch.float64, device=x.device)
    with profiling.op("apply_filter_rows_adj" if adjoint else "apply_filter_rows",
                      2 if row_sumsq is not None else 1, (12 if sub is not None else 8) * B * T):
        check(lib().babe_apply_filter_rows(_p(x), _p(y), B, T, int(nfft), _p(win), _p(tw), _p(freqs), _p(fc), _p(A),
                                           K, int(bool(adjoint)), _p(sub), _p(row_scale), _p(row_sumsq), _p(ws),
                                           nbytes, _p(status), _stream()), "apply_filter_rows")
    return y


def stft(x, nfft, frames=0, in_env_div=False, bin_scale=None):
    x = _cuda_f32(x, "x")
    B, T = x.shape
    win, tw = stft_tables(nfft, x.device)
    M = frames if frames else num_frames(T, nfft)
    if bin_scale is not None:
        bin_scale = _cuda_f32(bin_scale, "bin_scale")
    X = torch.empty(B, nfft // 2 + 1, M, 2, dtype=torch.float32, device=x.device)
    with profiling.op("stft", 1, 4 * B * T + X.numel() * 4):
        check(lib().babe_stft(_p(x), _p(X), B, T, int(nfft), int(frames), _p(win), _p(tw),
                              int(bool(in_env_div)), _p(bin_scale), _stream()), "stft")
    return X


def istft(X, nfft, out_len=None, bin_scale=None, out_env_div=True):
    X = _cuda_f32(X, "X")
    if X.data_ptr() % 8:
        X = X.clone()           # k_istft reads the bins as float2: a view at an odd float offset goes to fresh storage
    B, F, M, two = X.shape
    if F != nfft // 2 + 1 or two != 2:
        raise ValueError("X must be (B, NFFT/2+1, frames, 2)")
    full = nfft + (nfft // 2) * (M - 1)
    out_len = full if out_len is None else out_len
    win, tw = stft_tables(nfft, X.device)
    if bin_scale is not None:
        bin_scale = _cuda_f32(bin_scale, "H")
    y = torch.empty(B, out_len, dtype=torch.float32, device=X.device)
    with profiling.op("istft", 1, X.numel() * 4 + y.numel() * 4):
        check(lib().babe_istft(_p(X), _p(y), B, M, int(nfft), int(out_len), _p(win), _p(tw),
                               _p(bin_scale), int(bool(out_env_div)), _stream()), "istft")
    return y


def stft_stats(x, y, nfft, mode=0):
    """float64[3,F]: (sum|X|^2, sum|X||Y|, sum|Y|^2) or, mode 1, the cross term
    sum Re(conj(X) STFT(y/env)) in row 0."""
    x = _cuda_f32(x, "x")
    y = _cuda_f32(y, "y")
    if x.shape != y.shape or x.dim() != 2:
        raise ValueError("x and y must both be (B, T)")
    B, T = x.shape
    win, tw = stft_tables(nfft, x.device)
    F = nfft // 2 + 1
    nbytes = lib().babe_stft_stats_workspace(B, T, int(nfft))
    ws = torch.empty(nbytes // 4, dtype=torch.float32, device=x.device)
    abc = torch.empty(3, F, dtype=torch.float64, device=x.device)
    with profiling.op("stft_stats", 2, 8 * B * T):
        check(lib().babe_stft_stats(_p(x), _p(y), B, T, int(nfft), _p(win), _p(tw), int(mode), _p(abc),
                                    _p(ws), nbytes, _stream()), "stft_stats")
    return abc


def stft_stats_rows(x, y, nfft):
    """float64[B,3,F]: ``stft_stats`` (mode 0) of every row on its own."""
    if not (torch.is_tensor(x) and torch.is_tensor(y)):
        raise TypeError("x and y must be tensors")
    if x.shape != y.shape or x.dim() != 2:
        raise ValueError("x and y must both be (B, T)")
    x = _cuda_f32(x, "x")
    y = _cuda_f32(y, "y")
    B, T = x.shape
    win, tw = stft_tables(nfft, x.device)
    F = nfft // 2 + 1
    nbytes = lib().babe_stft_stats_rows_workspace(B, T, int(nfft))
    ws = torch.empty(nbytes // 4, dtype=torch.float32, device=x.device)
    abc = torch.empty(B, 3, F, dtype=torch.float64, device=x.device)
    with profiling.op("stft_stats_rows", 2, 8 * B * T):
        check(lib().babe_stft_stats_rows(_p(x), _p(y), B, T, int(nfft), _p(win), _p(tw), _p(abc), _p(ws), nbytes,
                                         _stream()), "stft_stats_rows")
    return abc


def spec_mag_stats(X, Xref, H=None, w=None):
    """float64[4,F]: a, b, c and s_k = sum (w_k (H_k|X| - |Xref|))^2."""
    X = _cuda_f32(X, "X")
    Xref = _cuda_f32(Xref, "Xref")
    if X.shape != Xref.shape or X.dim() != 4 or X.shape[-1] != 2:
        raise ValueError("X and Xref must both be (B, F, frames, 2)")
    B, F, M, _ = X.shape
    H = None if H is None else _cuda_f32(H, "H")
    w = None if w is None else _cuda_f32(w, "w")
    out = torch.empty(4, F, dtype=torch.float64, device=X.device)
    with profiling.op("spec_mag_stats", 1, 2 * X.numel() * 4):
        check(lib().babe_spec_mag_stats(_p(X), _p(Xref), _p(H), _p(w), B, F, M, _p(out), _stream()),
              "spec_mag_stats")
    return out


def spec_mag_grad(X, Xref, H, w, coef, want_X=True, want_Xref=False):
    """Gradients of || w (H|X| - |Xref|) ||_2 wrt the spectrograms; coef: 1-element CUDA tensor (g / norm)."""
    X = _cuda_f32(X, "X")
    Xref = _cuda_f32(Xref, "Xref")
    B, F, M, _ = X.shape
    H = None if H is None else _cuda_f32(H, "H")
    w = None if w is None else _cuda_f32(w, "w")
    coef = _cuda_f32(coef, "coef").reshape(1)
    gX = torch.empty_like(X) if want_X else None
    gR = torch.empty_like(Xref) if want_Xref else None
    with profiling.op("spec_mag_grad", 1, 4 * X.numel() * (2 + int(want_X) + int(want_Xref))):
        check(lib().babe_spec_mag_grad(_p(X), _p(Xref), _p(H), _p(w), _p(coef), B, F, M, _p(gX), _p(gR), _stream()),
              "spec_mag_grad")
    return gX, gR


def spec_dist_stats(X, Xref, w=None, mode=0):
    """float64[F] per-bin sums of squares of the complex (mode 0) / log-magnitude (mode 2) spectrogram distance;
    mode 3: per-bin sum of Re(conj(X) Xref)."""
    X = _cuda_f32(X, "X")
    Xref = _cuda_f32(Xref, "Xref")
    if X.shape != Xref.shape or X.dim() != 4 or X.shape[-1] != 2:
        raise ValueError("X and Xref must both be (B, F, frames, 2)")
    B, F, M, _ = X.shape
    w = None if w is None else _cuda_f32(w, "w")
    out = torch.empty(F, dtype=torch.float64, device=X.device)
    with profiling.op("spec_dist_stats", 1, 2 * X.numel() * 4):
        check(lib().babe_spec_dist_stats(_p(X), _p(Xref), _p(w), int(mode), B, F, M, _p(out), _stream()),
              "spec_dist_stats")
    return out


def spec_dist_grad(X, Xref, w, coef, mode=0, want_X=True, want_Xref=False):
    """Gradients of the mode-0 / mode-2 spectrogram distance wrt the spectrograms; coef: 1-element CUDA tensor."""
    X = _cuda_f32(X, "X")
    Xref = _cuda_f32(Xref, "Xref")
    B, F, M, _ = X.shape
    w = None if w is None else _cuda_f32(w, "w")
    coef = _cuda_f32(coef, "coef").reshape(1)
    gX = torch.empty_like(X) if want_X else None
    gR = torch.empty_like(Xref) if want_Xref else None
    with profiling.op("spec_dist_grad", 1, 4 * X.numel() * (2 + int(want_X) + int(want_Xref))):
        check(lib().babe_spec_dist_grad(_p(X), _p(Xref), _p(w), _p(coef), int(mode), B, F, M, _p(gX), _p(gR),
                                        _stream()), "spec_dist_grad")
    return gX, gR


def fit_params(abc, w, freqs, params, cfg, return_iters=False):
    """Run the device-resident projected gradient descent IN PLACE on
    params[2,K] (float32, CUDA, contiguous)."""
    if abc.dtype != torch.float64 or not abc.is_cuda:
        raise TypeError("abc must be a CUDA float64 tensor")
    if not (params.is_cuda and params.dtype == torch.float32 and params.is_contiguous()
            and params.dim() == 2 and params.shape[0] == 2):
        raise TypeError("params must be a contiguous CUDA float32 tensor of shape (2, K)")
    w = _cuda_f32(w, "w")
    freqs = _cuda_f32(freqs, "f")
    F = freqs.numel()
    abc = abc.contiguous()
    iters = torch.zeros(1, dtype=torch.int32, device=params.device) if return_iters else None
    with profiling.op("fit_params", 1, 3 * F * 8):
        check(lib().babe_fit_params(_p(abc), _p(w), _p(freqs), F, _p(params), params.shape[1],
                                    ctypes.byref(cfg), _p(iters), _stream()), "fit_params")
    return (params, iters) if return_iters else params


def fit_params_rows(abc, w, freqs, params, cfg, return_iters=False):
    """``fit_params`` on every row on its own, IN PLACE on params[B,2,K] from abc[B,3,F] (``stft_stats_rows``);
    with ``return_iters`` also the int32[B] iteration counts."""
    if not (torch.is_tensor(abc) and torch.is_tensor(params)):
        raise TypeError("abc and params must be tensors")
    if params.dim() != 3 or params.shape[1] != 2:
        raise ValueError(f"params must be (B, 2, K), got {tuple(params.shape)}")
    if abc.dim() != 3 or abc.shape[0] != params.shape[0] or abc.shape[1] != 3:
        raise ValueError(f"abc must be (B, 3, F) with B = {params.shape[0]}, got {tuple(abc.shape)}")
    if not (abc.is_cuda and params.is_cuda):
        raise BabeError("abc and params must be CUDA tensors: babe_b200 runs on CUDA tensors only "
                        "(there is no CPU fallback)")
    if abc.dtype != torch.float64:
        raise TypeError("abc must be a CUDA float64 tensor")
    if not (params.dtype == torch.float32 and params.is_contiguous()):
        raise TypeError("params must be a contiguous CUDA float32 tensor of shape (B, 2, K)")
    w = _cuda_f32(w, "w")
    freqs = _cuda_f32(freqs, "f")
    F = freqs.numel()
    if abc.shape[2] != F:
        raise ValueError(f"abc has {abc.shape[2]} bins, freqs {F}")
    B, K = params.shape[0], params.shape[2]
    abc = abc.contiguous()
    iters = torch.zeros(B, dtype=torch.int32, device=params.device) if return_iters else None
    with profiling.op("fit_params_rows", 1, 3 * F * 8 * B):
        check(lib().babe_fit_params_rows(_p(abc), _p(w), _p(freqs), F, _p(params), B, K, ctypes.byref(cfg),
                                         _p(iters), _stream()), "fit_params_rows")
    return (params, iters) if return_iters else params


def row_noise(seeds, shape_or_a, draw, slot=0, scale=None, row_scale=None, mult=1.0, out=None):
    """Keyed standard normal noise, one seed per row (``k_row_noise``, DESIGN.md 4.8):
    ``out[b, n] = a[b, n] + eps[b, n] * mult * scale * row_scale[b]``, eps[b, n] a function of (seeds[b], draw + slot,
    n) alone.  ``seeds``: int64 CUDA tensor (B,) (read as uint64).  ``shape_or_a``: (B, T) for the bare noise (a = 0)
    or the float32 (B, T) tensor a.  ``draw``: draw index, an int or a CUDA int32 tensor of one element (read by the
    kernel at run time, so a captured graph replays with its current value).  ``scale``: optional CUDA float32 tensor
    of one element; ``row_scale``: optional CUDA float32 (B,); ``mult``: host float.  ``out`` may be ``a``."""
    if not torch.is_tensor(seeds):
        raise TypeError("seeds must be an int64 tensor")
    if not seeds.is_cuda:
        raise BabeError(f"seeds is on {seeds.device}: babe_b200 runs on CUDA tensors only (there is no CPU fallback)")
    if seeds.dtype != torch.int64 or seeds.dim() != 1:
        raise ValueError(f"seeds must be a 1-D int64 tensor, got {seeds.dtype} of shape {tuple(seeds.shape)}")
    seeds = seeds.contiguous()
    dev = seeds.device
    a = None
    if torch.is_tensor(shape_or_a):
        a = _cuda_f32(shape_or_a, "a")
        shape = tuple(a.shape)
    else:
        shape = tuple(int(v) for v in shape_or_a)
    if len(shape) != 2 or shape[0] != seeds.numel():
        raise ValueError(f"noise of shape {shape}: must be (B, T) with B = {seeds.numel()} seeds")
    B, T = shape
    if torch.is_tensor(draw):
        if not draw.is_cuda:
            raise BabeError(f"draw is on {draw.device}: pass an int or a CUDA int32 tensor")
        if draw.dtype != torch.int32 or draw.numel() != 1:
            raise ValueError("draw must be an int or a CUDA int32 tensor of one element")
    else:
        draw = torch.full((1,), int(draw), dtype=torch.int32, device=dev)
    if scale is not None:
        scale = _cuda_f32(scale, "scale")
        if scale.numel() != 1:
            raise ValueError("scale must have one element")
    if row_scale is not None:
        row_scale = _cuda_f32(row_scale, "row_scale")
        if row_scale.numel() != B:
            raise ValueError(f"row_scale must have B = {B} entries, got {row_scale.numel()}")
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=dev)
    else:
        _cuda_f32(out, "out")
        if tuple(out.shape) != shape or not out.is_contiguous():
            raise ValueError(f"out must be a contiguous float32 tensor of shape {shape}")
    if slot < 0:
        raise ValueError("slot must be >= 0")
    # algorithmic bytes: write the noise (+ read a)
    with profiling.op("row_noise", 1, (8 if a is not None else 4) * B * T):
        check(lib().babe_row_noise(_p(out), _p(a), _p(seeds), B, T, _p(draw), int(slot), _p(scale), _p(row_scale),
                                   float(mult), _stream()), "row_noise")
    return out


# ---------------------------------------------------------------------------
_FIR_TABLES = {}


def fir_tables(taps, device):
    """(G_fwd, G_adj, L, pad_left) for a tap vector: spectra of the zero padded taps for the
    overlap-save kernel (float64 FFT on the host, once per filter)."""
    b = taps.detach().reshape(-1).to("cpu", torch.float64).numpy()
    key = (b.tobytes(), str(device))
    if key not in _FIR_TABLES:
        N, L = 4096, b.shape[0]
        if L > N // 2 + 1:
            raise BabeError(f"FIR with {L} taps: at most {N // 2 + 1} are supported")

        def table(v):
            g = np.conj(np.fft.fft(np.concatenate((v, np.zeros(N - L))))) / N
            return torch.from_numpy(np.stack((g.real, g.imag), -1).astype(np.float32)).to(device)
        _FIR_TABLES[key] = (table(b), table(b[::-1].copy()), L, (L - 1) // 2)
    return _FIR_TABLES[key]


def fir_filter(x, taps, adjoint=False):
    """torch.nn.functional.conv1d(x[:,None], taps[None,None], padding="same") on x[B,T]
    (utils/bandwidth_extension.py:76-95), or its transpose wrt x."""
    x = _cuda_f32(x, "x")
    if x.dim() != 2:
        raise ValueError("x must be (B, T)")
    B, T = x.shape
    Gf, Ga, L, pl = fir_tables(taps, x.device)
    _, tw = stft_tables(4096, x.device)
    y = torch.empty_like(x)
    with profiling.op("fir_filter", 1, 8 * B * T):
        check(lib().babe_fir_filter(_p(x), _p(y), B, T, _p(tw), _p(Ga if adjoint else Gf), L,
                                    (L - 1 - pl) if adjoint else pl, _stream()), "fir_filter")
    return y
