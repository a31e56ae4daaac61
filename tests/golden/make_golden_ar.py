#!/usr/bin/env python
"""Golden vectors for the non-blind / autoregressive sampling methods, produced by the UNMODIFIED
reference sampler (testing/blind_bwe_sampler.py: predict_bwe_AR :259-303, predict_bwe :306-364,
predict :406-497) with the toy denoiser.  Needs BABE_REFERENCE set to a checkout of eloimoliner/BABE:

    python tests/golden/make_golden_ar.py        ->  tests/golden/sampler_ar.npz
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as mg                             # noqa: E402  (imports the reference)


def main():
    B, T, nfft, sr = 2, 4096, 1024, 22050
    args = mg.make_args(nfft=nfft, sr=sr, audio_len=T, T=4, max_iter=20)
    torch.manual_seed(0)
    model = mg.ToyDenoiser()
    sampler = mg.BlindSampler(model, mg.EDM(args), args, rid=False)
    x = mg.piano_like(B, T, sr, 31)
    f = torch.fft.rfftfreq(nfft, d=1 / sr)
    filt = torch.tensor([[800.0, 2000.0], [-15.0, -30.0]])
    ylpf = mg.ref_ops.apply_filter(x, mg.ref_ops.design_filter(filt[0], filt[1], f), nfft)
    mask = torch.ones(B, T)
    mask[:, 1200:] = 0                               # head known from the previous segment
    y_masked = x * mask
    out = {"x": x, "ylpf": ylpf, "mask": mask, "y_masked": y_masked, "filt": filt, "nfft": nfft, "sr": sr}
    torch.manual_seed(77)
    out["x_ar"] = sampler.predict_bwe_AR(ylpf.clone(), y_masked.clone(), filt.clone(), "fc_A", mask=mask.clone())
    # plain non-blind run with the same known filter (no mask); fresh sampler: predict_bwe_AR leaves
    # self.data_consistency = True behind
    sampler2 = mg.BlindSampler(model, mg.EDM(args), args, rid=False)
    torch.manual_seed(78)
    out["x_bwe"] = sampler2.predict_bwe(ylpf.clone(), filt.clone(), "fc_A")
    np.savez_compressed(os.path.join(HERE, "sampler_ar.npz"),
                        **{k: (v.detach().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in out.items()})
    print("wrote sampler_ar.npz", float(out["x_ar"].std()), float(out["x_bwe"].std()))


if __name__ == "__main__":
    main()
