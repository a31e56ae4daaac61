#!/usr/bin/env python
"""Teacher-forcing goldens from the UNMODIFIED reference (needs BABE_REFERENCE set to a checkout of eloimoliner/BABE):

    python tests/golden/make_golden_tf.py      ->  tests/golden/teacher_forced.npz, optional_branches.npz

* ``fit_iters_*``: the filter parameters after EVERY ONE of the 100 iterations of
  ``BlindSampler.fit_params`` (testing/blind_bwe_sampler.py:533-595).  The loop body is re-entered with
  ``max_iter = 1`` from the previous iterate, which performs exactly the arithmetic of the 100-iteration call
  (asserted below against the 100-iteration result) without touching the reference file.
* ``step_*``: the state of ``BlindSampler.predict_blind_bwe`` (:619-769) around every sampler step -- x entering
  the step, the noise drawn, the filter before / after, the denoised estimate, x leaving the step -- recorded by
  wrapping ``move_timestep`` / ``fit_params`` / ``torch.randn`` from the outside.
* ``optional_branches.npz``: two-step runs of the non-default branches of ``get_rec_grads`` and of the loop
  (:63-73, :80-86, :99-115): data consistency, smooth-L1, cosine, STFT / STFT-magnitude / log-magnitude distances.
  Each array is stored once (the file stays under 1 MB): the observation of every run is ``fit_sampler.npz``'s
  ``y`` (its first 4000 samples for the STFT distances), and runs of one length draw the same noise
  (``opt_draws_4096``, ``opt_draws_4000``) except SNR_observations, which draws more (``opt_snr_draws``).

A test that starts the CUDA kernels from each reference iterate / state and compares ONE iteration / ONE step
closes the parity argument that the chained comparisons (chaotic amplification of fp32 rounding in the
mu = 1000 gradient descent) cannot.
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as mg            # noqa: E402  (sets up sys.path / plotly stubs, imports the reference)
from make_golden import BlindSampler, EDM, ToyDenoiser, ref_ops, make_args, piano_like   # noqa: E402


def _np(d):
    return {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in d.items()}


def fit_iterates(sampler, args, xden, y, p0, n=100):
    args.tester.blind_bwe.optimization.max_iter = 1
    its = [p0.clone()]
    p = p0.clone()
    for _ in range(n):
        p = sampler.fit_params(xden.clone(), y.clone(), p.clone()).detach().clone()
        its.append(p.clone())
    args.tester.blind_bwe.optimization.max_iter = n
    full = sampler.fit_params(xden.clone(), y.clone(), p0.clone()).detach()
    # the reference's early stop (:586-588) may end the n-iteration call early; up to there the chains agree
    ident = [bool(torch.equal(full, q)) for q in its]
    assert any(ident), "max_iter=1 chain does not reproduce the full call"
    return torch.stack(its), full, ident.index(True)


def gen_fit():
    out = {}
    # case A: the inputs of fit_sampler.npz (NFFT 1024, K = 5)
    g = dict(np.load(os.path.join(HERE, "fit_sampler.npz")))
    args = make_args(nfft=int(g["nfft"]), sr=int(g["sr"]), audio_len=g["y"].shape[1], T=4, max_iter=100)
    sampler = BlindSampler(ToyDenoiser(), EDM(args), args, rid=False)
    sampler.freqs = torch.fft.rfftfreq(int(g["nfft"]), d=1 / int(g["sr"]))
    its, full, stop = fit_iterates(sampler, args, torch.from_numpy(g["fit_xden"]), torch.from_numpy(g["y"]),
                                   torch.from_numpy(g["fit_p0"]))
    assert torch.equal(full, torch.from_numpy(g["fit_p_100"]))
    out["fit_iters_n1024"], out["fit_stop_n1024"] = its, stop
    # case B: NFFT 4096 (the shipped configuration), inputs of operator_n4096.npz
    g4 = dict(np.load(os.path.join(HERE, "operator_n4096.npz")))
    args4 = make_args(nfft=4096, sr=int(g4["sr"]), audio_len=g4["x"].shape[1], T=4, max_iter=100)
    s4 = BlindSampler(ToyDenoiser(), EDM(args4), args4, rid=False)
    s4.freqs = torch.fft.rfftfreq(4096, d=1 / int(g4["sr"]))
    p0 = torch.Tensor([args4.tester.blind_bwe.initial_conditions.fc, args4.tester.blind_bwe.initial_conditions.A])
    its4, full4, stop4 = fit_iterates(s4, args4, torch.from_numpy(g4["x"]), torch.from_numpy(g4["yobs"]), p0)
    out["fit_iters_n4096"], out["fit_stop_n4096"] = its4, stop4
    # case C: K = 7 formal variant
    p0f = torch.from_numpy(g["fit7_p0"])
    its7, full7, stop7 = fit_iterates(sampler, args, torch.from_numpy(g["fit_xden"]), torch.from_numpy(g["y"]), p0f)
    out["fit_iters_k7"], out["fit_stop_k7"] = its7, stop7
    return out


class Recorder:
    """Wraps methods of a BlindSampler INSTANCE and torch.randn to log the states of the loop."""

    def __init__(self, sampler):
        self.s = sampler
        self.draws, self.x_in, self.x_hat, self.t_hat, self.p_in, self.p_out = [], [], [], [], [], []
        self._mt, self._fp, self._randn = sampler.move_timestep, sampler.fit_params, torch.randn

    def __enter__(self):
        def randn(*a, **k):
            r = self._randn(*a, **k)
            self.draws.append(r.clone())
            return r

        def move_timestep(x, t, gamma, *a, **k):
            self.x_in.append(x.detach().clone())
            xh, th = self._mt(x, t, gamma, *a, **k)
            self.x_hat.append(xh.detach().clone())
            self.t_hat.append(th.detach().clone())
            return xh, th

        def fit_params(xden, y, p):
            self.p_in.append(p.detach().clone())
            q = self._fp(xden, y, p)
            self.p_out.append(q.detach().clone())
            return q
        torch.randn = randn
        self.s.move_timestep = move_timestep
        self.s.fit_params = fit_params
        return self

    def __exit__(self, *a):
        torch.randn = self._randn
        self.s.move_timestep, self.s.fit_params = self._mt, self._fp


def gen_steps():
    g = dict(np.load(os.path.join(HERE, "fit_sampler.npz")))
    nfft, sr = int(g["nfft"]), int(g["sr"])
    y = torch.from_numpy(g["y"])
    args = make_args(nfft=nfft, sr=sr, audio_len=y.shape[1], T=4, max_iter=20)
    sampler = BlindSampler(ToyDenoiser(), EDM(args), args, rid=False)
    torch.manual_seed(42)
    with Recorder(sampler) as rec:
        x, p, den, t, filt = sampler.predict_blind_bwe(y.clone(), rid=True)
    assert np.allclose(x.numpy(), g["sampler_x"]) and np.allclose(p.numpy(), g["sampler_params"])
    T = args.tester.T
    x_out = rec.x_in[1:] + [x]
    # fit calls: two per step except the last (Euler) step
    first, second = [], []
    k = 0
    for i in range(T):
        first.append(k)
        k += 1
        if float(t[i + 1]) != 0:
            second.append(k)
            k += 1
        else:
            second.append(first[-1])
    assert k == len(rec.p_in)
    return {"step_y": y, "step_t": t, "step_draws": torch.stack(rec.draws),          # draw 0: the initial x
            "step_x_in": torch.stack(rec.x_in), "step_x_hat": torch.stack(rec.x_hat),
            "step_t_hat": torch.stack(rec.t_hat), "step_x_out": torch.stack(x_out),
            "step_p_in": torch.stack([rec.p_in[j] for j in first]),
            "step_p_mid": torch.stack([rec.p_out[j] for j in first]),
            "step_p_out": torch.stack([rec.p_out[j] for j in second]),
            "step_x_den": den, "step_nfft": nfft, "step_sr": sr, "step_max_iter": 20}


def gen_optional():
    g = dict(np.load(os.path.join(HERE, "fit_sampler.npz")))
    nfft, sr = int(g["nfft"]), int(g["sr"])
    out = {}
    for variant in ("data_consistency", "smoothl1", "cosine", "stft", "stft_mag", "stft_logmag", "snr"):
        y = torch.from_numpy(g["y"]).clone()
        T_len = y.shape[1]
        if variant.startswith("stft"):
            y = y[:, :4000].contiguous()       # T % hop == 0 gives an all-zero frame and NaN gradients in the reference
            T_len = 4000
        args = make_args(nfft=nfft, sr=sr, audio_len=T_len, T=2, max_iter=2)
        ps = args.tester.posterior_sampling
        if variant == "data_consistency":
            ps.data_consistency = True
        elif variant in ("smoothl1", "cosine"):
            ps.norm = variant
        elif variant == "snr":
            ps.SNR_observations = 30
        else:
            ps.stft_distance.use = True
            ps.stft_distance.nfft = 1024
            ps.freq_weighting = "sqrt"
            ps.stft_distance.mag = variant != "stft"
            ps.stft_distance.logmag = variant == "stft_logmag"
        sampler = BlindSampler(ToyDenoiser(), EDM(args), args, rid=False)
        torch.manual_seed(1)
        with Recorder(sampler) as rec:
            x, p = sampler.predict_blind_bwe(y.clone(), rid=False)
        assert torch.equal(y, torch.from_numpy(g["y"])[:, :T_len])
        draws = torch.stack(rec.draws)
        key = "opt_snr_draws" if variant == "snr" else f"opt_draws_{T_len}"
        assert key not in out or torch.equal(out[key], draws), variant
        out[key] = draws
        out[f"opt_{variant}_x"] = x
        out[f"opt_{variant}_p"] = p
        print("optional", variant, float(x.abs().mean()), p.flatten()[:3].tolist())
    return out


def gen_specgrad():
    """autograd of apply_filter_and_norm_STFTmag_fweighted wrt BOTH spectrograms (utils/blind_bwe_utils.py:250-296)."""
    g = dict(np.load(os.path.join(HERE, "operator_n1024.npz")))
    nfft = int(g["nfft"])
    X = ref_ops.apply_stft(torch.from_numpy(g["x"]), nfft).requires_grad_(True)
    Y = ref_ops.apply_stft(torch.from_numpy(g["yobs"]), nfft).requires_grad_(True)
    H = torch.from_numpy(g["H"])
    out = {}
    for wk in ("sqrt", "None"):
        nrm = ref_ops.apply_filter_and_norm_STFTmag_fweighted(X, Y, H, wk)
        gX, gY = torch.autograd.grad(3.0 * nrm, (X, Y))
        out[f"specgrad_{wk}_gX"], out[f"specgrad_{wk}_gXref"] = gX, gY
    return out


if __name__ == "__main__":
    torch.set_num_threads(8)
    tf = {}
    tf.update(gen_specgrad())
    tf.update(gen_fit())
    tf.update(gen_steps())
    np.savez_compressed(os.path.join(HERE, "teacher_forced.npz"), **_np(tf))
    np.savez_compressed(os.path.join(HERE, "optional_branches.npz"), **_np(gen_optional()))
    print("ok", {k: np.asarray(v).shape for k, v in _np(tf).items()})
