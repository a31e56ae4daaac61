"""CPU: plumbing of the per-row filter mode (one filter estimate per row of y).  Argument checks of the row
operators, the modes that exclude per-row filters, and the sampler's per-row bookkeeping with the three row
operators replaced by per-row loops over their oracle restatements: B rows in one per-row call must give what B
shared-mode calls with B = 1 give when every row draws its noise from its own generator.  The kernels themselves
are checked on the GPU (tests/test_per_row_filter_gpu.py)."""
import pytest
import torch

from conftest import rel_l2
from toy_model import ToyDenoiser


# --------------------------------------------------------------------------- argument checks
def test_row_ops_reject_cpu_tensors_and_bad_shapes():
    from babe_b200 import ops
    from babe_b200._lib import BabeError
    x = torch.zeros(3, 8192)
    f = torch.fft.rfftfreq(4096, d=1 / 22050)
    fc, A = torch.full((3, 2), 500.0), torch.full((3, 2), -20.0)
    with pytest.raises(BabeError):
        ops.apply_filter_rows(x, 4096, f, fc, A)
    with pytest.raises(BabeError):
        ops.stft_stats_rows(x, x, 4096)
    with pytest.raises(BabeError):
        ops.fit_params_rows(torch.zeros(3, 3, 2049, dtype=torch.float64), torch.ones(2049), f,
                            torch.zeros(3, 2, 2), None)
    # fc / A must be (B, K) with the B of x; a flat or mismatched parameter set is not reinterpreted
    for bad_fc, bad_A in ((fc[0], A[0]), (fc[:2], A[:2]), (fc, A[:, :1]), (fc[None], A[None])):
        with pytest.raises(ValueError):
            ops.apply_filter_rows(x, 4096, f, bad_fc, bad_A)
    with pytest.raises(ValueError):
        ops.stft_stats_rows(x, x[:2], 4096)
    with pytest.raises(ValueError):
        ops.fit_params_rows(torch.zeros(2, 3, 2049, dtype=torch.float64), torch.ones(2049), f,
                            torch.zeros(3, 2, 2), None)
    with pytest.raises(ValueError):
        ops.fit_params_rows(torch.zeros(3, 3, 2049, dtype=torch.float64), torch.ones(2049), f,
                            torch.zeros(3, 2), None)


def _sampler(**kw):
    from babe_b200 import edm, sampler
    args = sampler.make_args(audio_len=8192, T=4, NFFT=1024, max_iter=3, **kw)
    return sampler.BlindSamplerFused(ToyDenoiser(), edm.EDM(args), args, rid=False), args


def test_knob_and_excluded_modes():
    from babe_b200 import segments
    s, args = _sampler()
    assert s.filter_per_row is False
    s, args = _sampler(filter_per_row=True)
    assert s.filter_per_row is True and args.tester.blind_bwe.filter_per_row is True
    y = torch.zeros(2, 8192)
    s.joint = True
    with pytest.raises(ValueError, match="joint"):
        s.predict_blind_bwe(y)
    s.joint = False
    with pytest.raises(NotImplementedError, match="compute_sweep"):
        s.predict_blind_bwe(y, compute_sweep=True)
    args.tester.posterior_sampling.stft_distance.use = True
    with pytest.raises(NotImplementedError, match="STFT-distance"):
        s.predict_blind_bwe(y)
    args.tester.posterior_sampling.stft_distance.use_multires = True
    with pytest.raises(NotImplementedError, match="use_multires"):
        s.predict_blind_bwe(y)
    with pytest.raises(ValueError, match="joint"):
        segments.restore_recording(s, torch.zeros(1, 30000), 8192, joint=True, batched=True)
    # per-row start parameters: (2, K) or (B, 2, K) only
    args.tester.posterior_sampling.stft_distance.use = False
    args.tester.posterior_sampling.stft_distance.use_multires = False
    with pytest.raises(ValueError, match="per-row filter parameters"):
        s.predict_blind_bwe(y, init_params=torch.zeros(3, 2, 5))


# --------------------------------------------------------------------------- sampler bookkeeping on the oracle
@pytest.fixture
def oracle_row_ops(monkeypatch):
    from babe_b200 import blind_bwe_utils as bu, ops
    from oracle import filter_fit as ofit, stft_filter as osf

    def stft_stats(x, y, nfft, mode=0):
        return torch.stack(osf.stft_mag_stats(x.double(), y.double(), nfft))

    def fit_params(abc, w, freqs, params, cfg, return_iters=False):
        sr = int(round(float(freqs[1]) * 2 * (freqs.numel() - 1)))
        oc = ofit.FitConfig(nfft=2 * (freqs.numel() - 1), sample_rate=sr, fcmin=cfg.fcmin, fcmax=cfg.fcmax,
                            Amin=cfg.Amin, Amax=cfg.Amax, max_iter=cfg.max_iter, tol=(cfg.tol_fc, cfg.tol_A),
                            mu=(cfg.mu_fc, cfg.mu_A), clamp_fc=bool(cfg.clamp_fc), clamp_A=bool(cfg.clamp_A),
                            only_negative_A=bool(cfg.only_negative_A))
        p, it = ofit.fit_params_from_stats(abc[0].float(), abc[1].float(), abc[2].float(), params, oc)
        params.copy_(p)
        return (params, torch.tensor([it])) if return_iters else params

    def apply_filter(x, nfft, H=None, freqs=None, fc=None, A=None, adjoint=False, sub=None, row_scale=None,
                     row_sumsq=None, out=None):
        if H is None:
            H = osf.design_filter(fc, A, freqs)
        y = osf.apply_filter_adjoint(x, H, nfft) if adjoint else osf.apply_filter(x, H, nfft)
        if sub is not None:
            y = y - sub
        if row_sumsq is not None:
            row_sumsq += (y.double() ** 2).sum(1)
        if row_scale is not None:
            y = y * row_scale[:, None]
        return y

    def apply_filter_rows(x, nfft, freqs, fc, A, adjoint=False, sub=None, row_scale=None, row_sumsq=None,
                          out=None, status=None):
        rows = []
        for b in range(x.shape[0]):
            ss = None if row_sumsq is None else row_sumsq[b:b + 1]
            rows.append(apply_filter(x[b:b + 1], nfft, freqs=freqs, fc=fc[b], A=A[b], adjoint=adjoint,
                                     sub=None if sub is None else sub[b:b + 1],
                                     row_scale=None if row_scale is None else row_scale[b:b + 1], row_sumsq=ss))
        return torch.cat(rows, 0)

    def stft_stats_rows(x, y, nfft):
        return torch.stack([stft_stats(x[b:b + 1], y[b:b + 1], nfft) for b in range(x.shape[0])])

    def fit_params_rows(abc, w, freqs, params, cfg, return_iters=False):
        its = [fit_params(abc[b], w, freqs, params[b], cfg, True)[1] for b in range(params.shape[0])]
        return (params, torch.cat(its)) if return_iters else params

    for name, fn in (("stft_stats", stft_stats), ("fit_params", fit_params), ("apply_filter", apply_filter),
                     ("apply_filter_rows", apply_filter_rows), ("stft_stats_rows", stft_stats_rows),
                     ("fit_params_rows", fit_params_rows)):
        monkeypatch.setattr(ops, name, fn)
    monkeypatch.setattr(bu, "freq_weight_vector", lambda kind, F, device: osf.freq_weight_vector(kind, F))


def _row_noise(gens, rows):
    return lambda shape, dev: torch.stack([torch.randn(shape[1], generator=gens[r]) for r in rows]).to(dev)


def test_per_row_sampler_equals_single_row_calls(oracle_row_ops, golden):
    """Per-row fit statistics, fit, guidance filter and guidance normaliser: B rows in one call == B calls on one
    row each (same noise per row), on the oracle operators."""
    from babe_b200 import edm, sampler
    g = golden("fit_sampler.npz")
    y1 = torch.from_numpy(g["y"])[:1]
    y = torch.cat([y1, 0.5 * y1.roll(777, -1), 2.0 * y1.flip(-1)], 0)          # three different recordings
    args = sampler.make_args(sample_rate=int(g["sr"]), audio_len=y.shape[1], T=4, NFFT=int(g["nfft"]), max_iter=5)
    s = sampler.BlindSamplerFused(ToyDenoiser(), edm.EDM(args), args, rid=False)
    s.filter_per_row = True
    s.noise_fn = _row_noise([torch.Generator().manual_seed(10 + r) for r in range(3)], range(3))
    x, p, den, t, filt = s.predict_blind_bwe(y.clone(), rid=True, max_steps=2)
    assert x.shape == y.shape and p.shape == (3, 2, 5) and filt.shape == (4, 3, 2, 5)
    s.filter_per_row = False
    for r in range(3):
        s.noise_fn = _row_noise({r: torch.Generator().manual_seed(10 + r)}, [r])
        xr, pr = s.predict_blind_bwe(y[r:r + 1].clone(), max_steps=2)
        assert rel_l2(x[r:r + 1], xr) < 1e-6, r
        assert rel_l2(p[r], pr) < 1e-6, r
    # the rows really got different filters
    assert not torch.allclose(p[0], p[2])
