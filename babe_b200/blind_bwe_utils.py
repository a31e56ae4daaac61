"""Drop-in replacement for ``utils.blind_bwe_utils`` of eloimoliner/BABE.

Same function names, positional order and defaults as
utils/blind_bwe_utils.py so that ``testing/blind_bwe_sampler.py`` and the
testers run unchanged after ``sys.modules['utils.blind_bwe_utils'] = this``
(see ``babe_b200.install``).  Every numeric function runs in the sm_100a
kernels behind the C ABI (include/babe_b200.h) and participates in autograd
through explicit ``torch.autograd.Function`` boundaries with analytic
backward kernels.  CUDA tensors only -- there is no CPU fallback.
"""
import torch

from . import ops

STRICT_INDEX_ERROR = True   # reproduce design_filter's IndexError (costs one sync)


# ---------------------------------------------------------------------------
# autograd boundaries
# ---------------------------------------------------------------------------
class _FilterOp(torch.autograd.Function):
    """y = A_H x (or A_H^T x).  Linear in x, so its backward wrt x is the same
    Function with the adjoint flag flipped -- differentiable to any order.
    Reference: utils/blind_bwe_utils.py:6-13 and its autograd backward."""

    @staticmethod
    def forward(ctx, x, H, nfft, adjoint):
        ctx.nfft, ctx.adjoint = nfft, adjoint
        ctx.save_for_backward(x, H)
        return ops.apply_filter(x, nfft, H=H, adjoint=adjoint)

    @staticmethod
    def backward(ctx, g):
        x, H = ctx.saved_tensors
        gx = gH = None
        if ctx.needs_input_grad[0]:
            gx = _FilterOp.apply(g.contiguous(), H, ctx.nfft, not ctx.adjoint)
        if ctx.needs_input_grad[1]:
            # dL/dH_k = c_k/N sum Re(conj(STFT(a)) STFT(b/env)); for the forward
            # operator (a,b) = (x,g), for the adjoint the roles swap.
            a, b = (x, g) if not ctx.adjoint else (g, x)
            d = ops.stft_stats(a.detach(), b.detach().contiguous(), ctx.nfft, mode=1)[0]
            c = torch.full_like(d, 2.0)
            c[0] = 1.0
            c[-1] = 1.0
            gH = (d * c / ctx.nfft).to(torch.float32)
        return gx, gH, None, None


class _DesignFilter(torch.autograd.Function):
    """utils/blind_bwe_utils.py:82-119 (:41-80 with a gain); analytic VJP per
    SURVEY Appendix A.2 instead of autograd through masked index ops."""

    @staticmethod
    def forward(ctx, fc, A, f, G):
        ctx.save_for_backward(fc, A, f, G if G is not None else torch.empty(0, device=f.device))
        ctx.has_gain = G is not None
        return ops.design_filter(fc, A, f, gain_db=G, strict=STRICT_INDEX_ERROR)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gH):
        fc, A, f, G = ctx.saved_tensors
        gfc, gA, gG = ops.design_filter_vjp(fc, A, f, gH.contiguous(),
                                            gain_db=G if ctx.has_gain else None)
        return (gfc.reshape(fc.shape), gA.reshape(A.shape), None,
                gG.reshape(G.shape) if ctx.has_gain else None)


class _Stft(torch.autograd.Function):
    """utils/blind_bwe_utils.py:15-26; backward = windowed overlap-add of the
    rfft adjoint (babe_istft with bin_scale N*c', no envelope division)."""

    @staticmethod
    def forward(ctx, x, nfft):
        ctx.nfft, ctx.T = nfft, x.shape[-1]
        return ops.stft(x, nfft)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gX):
        nfft = ctx.nfft
        scale = torch.full((nfft // 2 + 1,), 0.5 * nfft, dtype=torch.float32, device=gX.device)
        scale[0] = nfft
        scale[-1] = nfft
        return ops.istft(gX.contiguous(), nfft, out_len=ctx.T, bin_scale=scale, out_env_div=False), None


class _FilterIstft(torch.autograd.Function):
    """utils/blind_bwe_utils.py:28-39."""

    @staticmethod
    def forward(ctx, X, H, nfft):
        ctx.nfft = nfft
        ctx.save_for_backward(X, H)
        return ops.istft(X, nfft, bin_scale=H, out_env_div=True)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        X, H = ctx.saved_tensors
        nfft = ctx.nfft
        M = X.shape[2]
        c = torch.full((nfft // 2 + 1,), 2.0 / nfft, dtype=torch.float32, device=g.device)
        c[0] = 1.0 / nfft
        c[-1] = 1.0 / nfft
        # adjoint of irfft applied to the windowed frames of g / envelope
        if not ctx.needs_input_grad[1]:
            # only the spectrogram's gradient is wanted (H fixed, the usual guidance case): H rides in the STFT
            # kernel's per-bin scale, no separate pass over the spectrogram
            return ops.stft(g.contiguous(), nfft, frames=M, in_env_div=True, bin_scale=c * H), None, None
        Gs = ops.stft(g.contiguous(), nfft, frames=M, in_env_div=True, bin_scale=c)
        gX = gH = None
        if ctx.needs_input_grad[0]:
            gX = Gs * H[None, :, None, None]
        if ctx.needs_input_grad[1]:
            gH = ops.spec_dist_stats(X, Gs, None, mode=3).to(torch.float32)      # per-bin sum of Re(conj(X) G)
        return gX, gH, None


class _SpecMagNorm(torch.autograd.Function):
    """|| w (H |X| - |Xref|) ||_2 of utils/blind_bwe_utils.py:250-296 (and
    :130-141 with w = H-only).  One pass over both spectrograms; backward wrt H
    from the per-bin sums a_k, b_k saved by the forward."""

    @staticmethod
    def forward(ctx, X, Xref, H, w):
        st = ops.spec_mag_stats(X, Xref, H=H, w=w)
        norm64 = torch.sqrt(st[3].sum())
        spec = (X, Xref) if (X.requires_grad or Xref.requires_grad) else (torch.empty(0, device=H.device),) * 2
        ctx.save_for_backward(st, H, w if w is not None else torch.empty(0, device=H.device), norm64, *spec)
        ctx.has_w = w is not None
        return norm64.to(torch.float32)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        st, H, w, norm64, X, Xref = ctx.saved_tensors
        gX = gR = gH = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            # what autograd gives the reference through sqrt(re^2 + im^2) (utils/blind_bwe_utils.py:254-257)
            coef = (g.double() / norm64).to(torch.float32)
            gX, gR = ops.spec_mag_grad(X, Xref, H, w if ctx.has_w else None, coef,
                                       want_X=ctx.needs_input_grad[0], want_Xref=ctx.needs_input_grad[1])
        if ctx.needs_input_grad[2]:
            w2 = (w.double() ** 2) if ctx.has_w else 1.0
            gH = (g.double() * w2 * (H.double() * st[0] - st[1]) / norm64).to(torch.float32)
        return gX, gR, gH, None


# ---------------------------------------------------------------------------
# the reference's public functions
# ---------------------------------------------------------------------------
def apply_filter(x, H, NFFT):
    """utils/blind_bwe_utils.py:6-13."""
    return _FilterOp.apply(x, H, int(NFFT), False)


class _RowFilterOp(torch.autograd.Function):
    """y_b = A_{fc_b, A_b} x_b (or its adjoint): one filter per row, designed inside the kernel.  Linear in x; the
    filter parameters get no gradient."""

    @staticmethod
    def forward(ctx, x, freqs, fc, A, nfft, adjoint):
        ctx.nfft, ctx.adjoint = nfft, adjoint
        ctx.save_for_backward(freqs, fc, A)
        return ops.apply_filter_rows(x, nfft, freqs, fc, A, adjoint=adjoint)

    @staticmethod
    def backward(ctx, g):
        freqs, fc, A = ctx.saved_tensors
        gx = None
        if ctx.needs_input_grad[0]:
            gx = _RowFilterOp.apply(g.contiguous(), freqs, fc, A, ctx.nfft, not ctx.adjoint)
        return gx, None, None, None, None, None


def apply_filter_rows(x, freqs, fc, A, NFFT):
    """Row b of x (B, T) through the lowpass designed from fc[b], A[b] (fc, A: (B, K))."""
    return _RowFilterOp.apply(x, freqs, fc.contiguous(), A.contiguous(), int(NFFT), False)


def apply_stft(x, NFFT):
    """utils/blind_bwe_utils.py:15-26."""
    return _Stft.apply(x, int(NFFT))


def apply_filter_istft(X, H, NFFT):
    """utils/blind_bwe_utils.py:28-39."""
    return _FilterIstft.apply(X, H, int(NFFT))


def _as_param(v, f):
    """Breakpoints may be lists, Python numbers, 0-d / 1-elt tensors (scalar
    branch, utils/blind_bwe_utils.py:114-118) or (K,) tensors (:52-59)."""
    if torch.is_tensor(v):
        return v.to(device=f.device, dtype=torch.float32).reshape(-1)
    if isinstance(v, (list, tuple)):
        if len(v) > 0 and torch.is_tensor(v[0]):
            return torch.stack([t.reshape(()) for t in v]).to(device=f.device, dtype=torch.float32)
        return torch.tensor([float(t) for t in v], dtype=torch.float32, device=f.device)
    return torch.tensor([float(v)], dtype=torch.float32, device=f.device)


def design_filter(fc, A, f):
    """utils/blind_bwe_utils.py:82-119."""
    return _DesignFilter.apply(_as_param(fc, f), _as_param(A, f), f, None)


def design_filter_G(fc, A, G, f):
    """utils/blind_bwe_utils.py:41-80."""
    return _DesignFilter.apply(_as_param(fc, f), _as_param(A, f), f, _as_param(G, f))



class _SpecDist(torch.autograd.Function):
    """The STFT-guidance distances on spectrograms: mode 0 = || w X - w Xref ||_2 (utils/blind_bwe_utils.py:148-197),
    mode 1 = || w|X| - w|Xref| ||_2 and mode 2 = its log10(. + 1e-8) form (:198-248).  One reduction kernel forward,
    one element-wise kernel backward (what the reference's autograd chain computes), no weighted copies in HBM."""

    @staticmethod
    def forward(ctx, X, Xref, w, mode):
        if mode == 1:
            ss = ops.spec_mag_stats(X, Xref, H=None, w=w)[3]
        else:
            ss = ops.spec_dist_stats(X, Xref, w=w, mode=mode)
        norm64 = torch.sqrt(ss.sum())
        ctx.mode, ctx.has_w = mode, w is not None
        ctx.save_for_backward(X, Xref, w if w is not None else torch.empty(0, device=X.device), norm64)
        return norm64.to(torch.float32)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        X, Xref, w, norm64 = ctx.saved_tensors
        w = w if ctx.has_w else None
        coef = (g.double() / norm64).to(torch.float32)
        want = dict(want_X=ctx.needs_input_grad[0], want_Xref=ctx.needs_input_grad[1])
        if ctx.mode == 1:
            gX, gR = ops.spec_mag_grad(X, Xref, None, w, coef, **want)
        else:
            gX, gR = ops.spec_dist_grad(X, Xref, w, coef, mode=ctx.mode, **want)
        return gX, gR, None, None


def freq_weight_vector(freq_weight, F, device):
    """Per-bin multiplier for each ``freq_weight`` string
    (utils/blind_bwe_utils.py:260-293); unknown strings apply no weighting,
    like the reference's fall-through."""
    fr = torch.linspace(0, 1, F).to(device)
    table = {
        "linear": lambda: fr,
        "log": lambda: torch.log2(1 + fr),
        "sqrt": lambda: torch.sqrt(fr),
        "log2": lambda: torch.log2(fr),
        "log10": lambda: torch.log10(fr),
        "cubic": lambda: fr ** 3,
        "quadratic": lambda: fr ** 2,
        "logcubic": lambda: torch.log2(1 + fr ** 3),
        "logquadratic": lambda: torch.log2(1 + fr ** 2),
        "squared": lambda: fr ** 4,
    }
    if freq_weight in table:
        return table[freq_weight]()
    return None


def apply_filter_and_norm_STFTmag(X, Xref, H):
    """utils/blind_bwe_utils.py:130-141."""
    return _SpecMagNorm.apply(X, Xref, H, None)


def apply_norm_filter(H, H2):
    """utils/blind_bwe_utils.py:143-146 (an F-element vector norm)."""
    return torch.linalg.norm(H.reshape(-1) - H2.reshape(-1), ord=2)


def apply_norm_STFT_fweighted(y, den_rec, freq_weight="linear", NFFT=1024):
    """utils/blind_bwe_utils.py:148-197."""
    X = apply_stft(den_rec, NFFT)
    Xref = apply_stft(y, NFFT)
    w = freq_weight_vector(freq_weight, X.shape[1], X.device)
    return _SpecDist.apply(X, Xref, w, 0)


def apply_norm_STFTmag_fweighted(y, den_rec, freq_weight="linear", NFFT=1024, logmag=False):
    """utils/blind_bwe_utils.py:198-248."""
    X = apply_stft(den_rec, NFFT)
    Xref = apply_stft(y, NFFT)
    w = freq_weight_vector(freq_weight, X.shape[1], X.device)
    return _SpecDist.apply(X, Xref, w, 2 if logmag == True else 1)  # noqa: E712  (the reference compares with == True)


def apply_filter_and_norm_STFTmag_fweighted(X, Xref, H, freq_weight="linear"):
    """utils/blind_bwe_utils.py:250-296."""
    w = freq_weight_vector(freq_weight, X.shape[1], X.device)
    return _SpecMagNorm.apply(X, Xref, H, w)


def plot_filter(ref_filter, est_filter, NFFT=1024, fs=44100):
    """utils/blind_bwe_utils.py:298-306 -- plotting pass-through (needs plotly)."""
    import plotly.express as px
    f = torch.fft.rfftfreq(NFFT, d=1 / fs).to(ref_filter.device)
    Href = design_filter(ref_filter[0], ref_filter[1], f)
    H = design_filter(est_filter[0], est_filter[1], f)
    fig = px.line(x=f.cpu(), y=20 * torch.log10(H.cpu().detach()), log_x=True,
                  title='Frequency response of a low pass filter',
                  labels={'x': 'Frequency (Hz)', 'y': 'Magnitude (dB)'})
    fig.add_scatter(x=f.cpu(), y=20 * torch.log10(Href.cpu().detach()), mode='lines', name='Reference')
    return fig


def animation_filter(path, data_filters, t, NFFT=1024, fs=44100, name="animation_filter", NT=15):
    """utils/blind_bwe_utils.py:308-355 -- plotting pass-through (needs plotly,
    pandas); the filter responses come from the CUDA design kernel."""
    import pandas as pd
    import plotly.express as px
    dev = data_filters.device if data_filters.is_cuda else torch.device("cuda")
    f = torch.fft.rfftfreq(NFFT, d=1 / fs)
    nsteps = data_filters.shape[0]
    idx = [int(torch.floor(i)) for i in torch.linspace(0, nsteps - 1, min(nsteps, NT))]
    rows = [design_filter(data_filters[i, 0].to(dev), data_filters[i, 1].to(dev), f.to(dev)).cpu()
            for i in idx]
    allX = torch.stack(rows, 0)
    sigma = t[idx].cpu()
    ff = f.unsqueeze(0).expand(allX.shape[0], -1).reshape(-1)
    ss = sigma.unsqueeze(-1).expand(-1, allX.shape[1]).reshape(-1)
    df = pd.DataFrame({"f": ff.numpy(), "h": 20 * torch.log10(allX.reshape(-1)).numpy(),
                       "sigma": ss.numpy()})
    fig = px.line(df, x="f", y="h", animation_frame="sigma", log_x=True)
    fig.write_html(path + "/" + name + ".html", auto_play=False)
    return fig
