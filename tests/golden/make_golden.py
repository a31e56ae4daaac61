#!/usr/bin/env python
"""Generate golden vectors by importing the UNMODIFIED reference.

Needs BABE_REFERENCE set to a checkout of eloimoliner/BABE:

    python tests/golden/make_golden.py

Writes ``tests/golden/*.npz``.  The reference (eloimoliner/BABE) ships no
tests or fixtures, so these vectors -- produced by its own code on seeded
inputs -- are what pins the oracle (``oracle/``) and, through it, the CUDA
path.  Imports: ``utils/blind_bwe_utils.py``, ``testing/blind_bwe_sampler.py``
and ``diff_params/edm.py`` with a stub for the missing ``plotly`` module
(utils/blind_bwe_utils.py:3) and a ``SimpleNamespace`` standing in for Hydra.
"""
import os
import sys
import types
from types import SimpleNamespace as NS

import numpy as np
import torch

REF = os.environ.get("BABE_REFERENCE") or sys.exit("set BABE_REFERENCE to a checkout of eloimoliner/BABE")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))          # tests/ for toy_model
sys.path.insert(0, REF)
for name in ("plotly", "plotly.express"):
    sys.modules.setdefault(name, types.ModuleType(name))

import utils.blind_bwe_utils as ref_ops            # noqa: E402
from testing.blind_bwe_sampler import BlindSampler  # noqa: E402
from diff_params.edm import EDM                    # noqa: E402
from toy_model import ToyDenoiser                  # noqa: E402

WEIGHTS = ["linear", "None", "log", "sqrt", "cubic", "quadratic", "logcubic",
           "logquadratic", "squared"]


def make_args(nfft=1024, sr=22050, audio_len=4096, T=4, max_iter=100, K=5,
              xi=0.2, start_sigma=0.2):
    fc = [280, 285, 290, 295, 300][:K]
    A = [-15, -17, -20, -25, -30][:K]
    return NS(
        exp=NS(sample_rate=sr, audio_len=audio_len),
        diff_params=NS(sigma_data=0.063, sigma_min=1e-5, sigma_max=10, P_mean=-1.2, P_std=1.2,
                       ro=13, ro_train=13, Schurn=5, Snoise=1, Stmin=0, Stmax=50,
                       aweighting=NS(use_aweighting=False, ntaps=101)),
        tester=NS(
            T=T, order=2, filter_out_cqt_DC_Nyq=True,
            diff_params=NS(same_as_training=False, sigma_data=0.063, sigma_min=1e-4, sigma_max=1,
                           ro=8, Schurn=20, Snoise=1.0, Stmin=0, Stmax=50),
            posterior_sampling=NS(xi=xi, data_consistency=False, norm=2, SNR_observations="None",
                                  start_sigma=start_sigma, freq_weighting="None",
                                  freq_weighting_filter="sqrt", smoothl1_beta=1,
                                  stft_distance=NS(use=False, mag=False, use_multires=False,
                                                   nfft=2048, logmag=False)),
            blind_bwe=NS(fcmin=20, fcmax="nyquist", Amin=-50, Amax=30, NFFT=nfft,
                         sigma_den_estimate=0.0,
                         initial_conditions=NS(fc=fc, A=A),
                         optimization=NS(max_iter=max_iter, tol=[5e-3, 5e-3], mu=[1000, 10],
                                         clamp_fc=True, clamp_A=True, only_negative_A=True)),
            complete_recording=NS(inpaint_DC=True),
        ),
    )


def piano_like(B, T, sr, seed):
    """SURVEY 8(d) synthetic input, small note count."""
    g = torch.Generator().manual_seed(seed)
    n = torch.arange(T, dtype=torch.float64)
    out = torch.zeros(B, T, dtype=torch.float64)
    for b in range(B):
        for _ in range(6):
            k = int(torch.randint(20, 76, (1,), generator=g))
            f0 = 27.5 * 2 ** (k / 12)
            n0 = int(torch.randint(0, max(1, T // 2), (1,), generator=g))
            tt = (n - n0).clamp(min=0) / sr
            for hh in range(1, 13):
                if hh * f0 >= sr / 2:
                    break
                out[b] += (n >= n0) * hh ** -1.2 * torch.exp(-tt * hh / 1.5) * torch.sin(2 * np.pi * hh * f0 * tt)
    out = out / out.std(dim=1, keepdim=True) * 0.063
    return out.float()


def gen_operator(nfft, T, B, seed, tag):
    torch.manual_seed(seed)
    sr = 22050
    x = piano_like(B, T, sr, seed) + 0.01 * torch.randn(B, T)
    f = torch.fft.rfftfreq(nfft, d=1 / sr)
    fc = torch.tensor([400.0, 900.0, 1000.0, 2500.0, 6000.0])
    A = torch.tensor([-6.0, -12.0, -20.0, -30.0, -45.0])
    out = {"x": x, "f": f, "fc": fc, "A": A, "nfft": nfft, "sr": sr}
    H = ref_ops.design_filter(fc, A, f)
    out["H"] = H
    out["H_scalar"] = ref_ops.design_filter(torch.tensor(1000.0), torch.tensor(-20.0), f)
    out["H_list"] = ref_ops.design_filter([1000.0], [-20.0], f)
    out["H_G"] = ref_ops.design_filter_G(fc, A, torch.tensor(-3.0), f)
    # duplicates in one bin and a breakpoint exactly at the last bin
    fc2 = torch.tensor([f[7] + 0.3, f[7] + 0.9, f[8] + 0.1, f[-1]])
    A2 = torch.tensor([-3.0, -5.0, -9.0, -12.0])
    out["fc_dup"], out["A_dup"] = fc2, A2
    out["H_dup"] = ref_ops.design_filter(fc2, A2, f)
    X = ref_ops.apply_stft(x, nfft)
    out["X"] = X
    out["y"] = ref_ops.apply_filter(x, H, nfft)
    out["istft"] = ref_ops.apply_filter_istft(X.clone(), H, nfft)
    # gradients (autograd of the reference)
    r = torch.randn(B, T)
    out["r"] = r
    xg = x.clone().requires_grad_(True)
    Hg = H.clone().requires_grad_(True)
    yy = ref_ops.apply_filter(xg, Hg, nfft)
    gx, gH = torch.autograd.grad((yy * r).sum(), (xg, Hg))
    out["gx"], out["gH"] = gx, gH
    fcg = fc.clone().requires_grad_(True)
    Ag = A.clone().requires_grad_(True)
    Hh = ref_ops.design_filter(fcg, Ag, f)
    cot = torch.randn(f.shape)
    out["cotH"] = cot
    gfc, gA = torch.autograd.grad((Hh * cot).sum(), (fcg, Ag))
    out["gfc"], out["gA"] = gfc, gA
    # losses
    yobs = ref_ops.apply_filter(x, ref_ops.design_filter(torch.tensor([1000.0, 3000.0]), torch.tensor([-20.0, -30.0]), f), nfft)
    yobs = yobs + 0.002 * torch.randn(B, T)
    out["yobs"] = yobs
    Y = ref_ops.apply_stft(yobs, nfft)
    for wk in WEIGHTS:
        out["norm_fw_" + wk] = ref_ops.apply_filter_and_norm_STFTmag_fweighted(X, Y, H, wk)
        out["norm_stft_" + wk] = ref_ops.apply_norm_STFT_fweighted(yobs, x, wk, nfft)
        out["norm_mag_" + wk] = ref_ops.apply_norm_STFTmag_fweighted(yobs, x, wk, nfft)
    out["norm_logmag_sqrt"] = ref_ops.apply_norm_STFTmag_fweighted(yobs, x, "linear", nfft, logmag=True)
    out["norm_plain"] = ref_ops.apply_filter_and_norm_STFTmag(X, Y, H)
    out["norm_filter"] = ref_ops.apply_norm_filter(H, out["H_G"])
    # gradient of the fit loss wrt (fc, A) and wrt H
    fcg = fc.clone().requires_grad_(True)
    Ag = A.clone().requires_grad_(True)
    Hh = ref_ops.design_filter(fcg, Ag, f)
    Hh.retain_grad()
    nrm = ref_ops.apply_filter_and_norm_STFTmag_fweighted(X, Y, Hh, "sqrt")
    g1, g2, g3 = torch.autograd.grad(nrm, (fcg, Ag, Hh))
    out["fit_gfc"], out["fit_gA"], out["fit_gH"] = g1, g2, g3
    # rec-guidance operator part: grad wrt x of sum_b ||y - A x||
    xg = x.clone().requires_grad_(True)
    nb = torch.linalg.norm(yobs - ref_ops.apply_filter(xg, H, nfft), dim=1, ord=2)
    (gg,) = torch.autograd.grad(nb.sum(), xg)
    out["rg_norms"], out["rg_grad"] = nb.detach(), gg
    np.savez_compressed(os.path.join(HERE, f"operator_{tag}.npz"),
                        **{k: (v.detach().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in out.items()})
    print("operator", tag, "ok")


def gen_fit_and_sampler():
    B, T, nfft, sr = 2, 4096, 1024, 22050
    args = make_args(nfft=nfft, sr=sr, audio_len=T, T=4, max_iter=100)
    torch.manual_seed(0)
    model = ToyDenoiser()
    diff = EDM(args)
    sampler = BlindSampler(model, diff, args, rid=False)
    x = piano_like(B, T, sr, 11)
    f = torch.fft.rfftfreq(nfft, d=1 / sr)
    y = ref_ops.apply_filter(x, ref_ops.design_filter(torch.tensor([1000.0]), torch.tensor([-20.0]), f), nfft)
    out = {"x": x, "y": y, "nfft": nfft, "sr": sr}
    # --- fit_params alone (needs sampler.freqs, normally set in predict_blind_bwe) ---
    sampler.freqs = f
    p0 = torch.Tensor([args.tester.blind_bwe.initial_conditions.fc, args.tester.blind_bwe.initial_conditions.A])
    xden = x + 0.003 * torch.randn(B, T)
    out["fit_xden"] = xden
    out["fit_p0"] = p0.clone()
    for iters in (1, 5, 100):
        args.tester.blind_bwe.optimization.max_iter = iters
        p = sampler.fit_params(xden.clone(), y.clone(), p0.clone())
        out[f"fit_p_{iters}"] = p.detach().clone()
    args.tester.blind_bwe.optimization.max_iter = 100
    # K = 7 formal variant (conf/tester/blind_bwe_formal_1000.yaml:140-141), loose init
    p0f = torch.Tensor([[200, 225, 250, 275, 300, 325, 350], [-15, -20, -25, -30, -40, -50, -55]])
    out["fit7_p0"] = p0f.clone()
    out["fit7_p"] = sampler.fit_params(xden.clone(), y.clone(), p0f.clone()).detach().clone()
    # --- schedule ---
    t = diff.create_schedule_from_initial_t(0.2, 35)
    out["sched35"] = t
    out["gamma35"] = diff.get_gamma(t)
    out["sched_full"] = diff.create_schedule(35)
    # --- full blind sampler, 4 steps, toy denoiser ---
    args.tester.blind_bwe.optimization.max_iter = 20
    torch.manual_seed(42)
    xs, ps = sampler.predict_blind_bwe(y.clone(), rid=False)
    out["sampler_x"], out["sampler_params"] = xs, ps
    np.savez_compressed(os.path.join(HERE, "fit_sampler.npz"),
                        **{k: (v.detach().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in out.items()})
    print("fit+sampler ok", ps)


def gen_fir():
    """Classical FIR observation model (utils/bandwidth_extension.py:43-95)."""
    import utils.bandwidth_extension as ref_bwe
    torch.manual_seed(9)
    x = piano_like(2, 5000, 22050, 21) + 0.01 * torch.randn(2, 5000)
    out = {"x": x}
    for tag, taps in (("lpf500", ref_bwe.get_FIR_lowpass(500, 1000, 1, 22050)),
                      ("hpf499", ref_bwe.get_FIR_high_pass(500, 1000, 1, 22050))):
        xg = x.clone().requires_grad_(True)
        y = ref_bwe.apply_low_pass_firwin(xg, taps)
        r = torch.randn(y.shape)
        (gx,) = torch.autograd.grad((y * r).sum(), xg)
        out["taps_" + tag], out["y_" + tag], out["r_" + tag], out["gx_" + tag] = taps, y, r, gx
    np.savez_compressed(os.path.join(HERE, "fir.npz"),
                        **{k: (v.detach().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in out.items()})
    print("fir ok")


if __name__ == "__main__":
    torch.set_num_threads(8)
    gen_operator(1024, 5000, 2, 3, "n1024")
    gen_operator(4096, 9001, 1, 4, "n4096")
    gen_fit_and_sampler()
    gen_fir()
