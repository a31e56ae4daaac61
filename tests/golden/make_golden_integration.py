#!/usr/bin/env python
"""Integration golden (SURVEY section 4, integration row): the UNMODIFIED reference sampler
(testing/blind_bwe_sampler.py:619-769, BlindSampler.predict_blind_bwe) driving the UNMODIFIED reference network
(networks/cqtdiff+.py:583-845, Unet_CQT_oct_with_attention) -- the network running on the oracle CQT
(oracle/nsgt.py behind the ``cqt_nsgt_pytorch`` import name, upstream being unavailable offline).

Small configuration: 3 octaves x 8 bins, T = 4096 samples, NFFT 1024, 2 sampler steps, 5 fit iterations,
torch.manual_seed(0) network init (zero-initialised gates scaled so that they matter), torch.manual_seed(42) sampling.
Needs BABE_REFERENCE set to a checkout of eloimoliner/BABE:   python tests/golden/make_golden_integration.py  ->  integration.npz
"""
import importlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
import make_golden as mg                                              # noqa: E402  (reference imports + stubs)
from make_golden import BlindSampler, EDM, ref_ops, piano_like      # noqa: E402
from make_golden_tf import Recorder, _np                             # noqa: E402
from oracle.cqt_shim import OracleCQT                                # noqa: E402

AUDIO_LEN, SR, NFFT = 4096, 22050, 1024


def small_args():
    from babe_b200.sampler import make_args
    args = make_args(sample_rate=SR, audio_len=AUDIO_LEN, num_octs=3, bins_per_oct=8, NFFT=NFFT, T=2, max_iter=5)
    args.network.Ns = [8, 8, 16]
    args.network.Ss = [2, 2, 2]
    args.network.num_dils = [1, 2, 2]
    args.network.attention_layers = [0, 0, 0, 0]
    args.network.emb_dim = 32
    return args


def reference_network(args):
    shim = types.ModuleType("cqt_nsgt_pytorch")
    shim.CQT_nsgt = OracleCQT
    sys.modules["cqt_nsgt_pytorch"] = shim
    mod = importlib.import_module("networks.cqtdiff+")
    torch.manual_seed(0)
    net = mod.Unet_CQT_oct_with_attention(args, torch.device("cpu"))
    with torch.no_grad():                      # the gates are zero-initialised: make the residual branches count
        for n, p in net.named_parameters():
            if ".gate." in n and n.endswith("weight"):
                p.mul_(1e6)
    return net


if __name__ == "__main__":
    torch.set_num_threads(8)
    args = small_args()
    net = reference_network(args)
    for p in net.parameters():
        p.requires_grad_(False)
    x = piano_like(2, AUDIO_LEN, SR, 31)
    f = torch.fft.rfftfreq(NFFT, d=1 / SR)
    y = ref_ops.apply_filter(x, ref_ops.design_filter(torch.tensor([1000.0]), torch.tensor([-20.0]), f), NFFT)
    sampler = BlindSampler(net, EDM(args), args, rid=True)
    torch.manual_seed(42)
    with Recorder(sampler) as rec:
        xs, ps, den, t, filt = sampler.predict_blind_bwe(y.clone(), rid=True)
    out = {"y": y, "x": xs, "params": ps, "x_den": den, "t": t, "filters": filt, "draws": torch.stack(rec.draws),
           "x_in": torch.stack(rec.x_in), "x_hat": torch.stack(rec.x_hat), "x_out": torch.stack(rec.x_in[1:] + [xs]),
           "p_in": torch.stack(rec.p_in), "p_out": torch.stack(rec.p_out)}
    # one plain network evaluation as well (pins CQT + U-Net + preconditioning without the sampler around it)
    g = torch.Generator().manual_seed(5)
    xin = torch.randn(2, AUDIO_LEN, generator=g) * 0.1
    sig = torch.tensor([[-0.5], [0.3]])
    out["net_in"], out["net_sigma"], out["net_out"] = xin, sig, net(xin, sig)
    np.savez_compressed(os.path.join(HERE, "integration.npz"), **_np(out))
    print("integration ok", {k: tuple(np.asarray(v).shape) for k, v in _np(out).items()})
