"""CPU: the in-repo CQTDiff+ restatement (babe_b200/denoiser.py) against the
reference network file, both running on the oracle CQT.  Needs BABE_REFERENCE set to a checkout of
eloimoliner/BABE; skipped elsewhere (tests/test_integration_cpu.py checks the network's output against the
reference's stored output everywhere)."""
import importlib
import os
import sys
import types

import pytest
import torch

from conftest import rel_l2
from oracle.cqt_shim import OracleCQT

REF = os.environ.get("BABE_REFERENCE", "")
pytestmark = pytest.mark.skipif(not os.path.isdir(REF), reason="BABE_REFERENCE (reference checkout) not set")


def _small_args():
    from babe_b200.sampler import make_args
    args = make_args(sample_rate=22050, audio_len=4096, num_octs=3, bins_per_oct=8)
    args.network.Ns = [8, 8, 16]
    args.network.Ss = [2, 2, 2]
    args.network.num_dils = [1, 2, 2]
    args.network.attention_layers = [0, 0, 0, 0]
    args.network.emb_dim = 32
    return args


def _reference_net_class():
    saved = sys.modules.get("cqt_nsgt_pytorch")
    shim = types.ModuleType("cqt_nsgt_pytorch")
    shim.CQT_nsgt = OracleCQT
    sys.modules["cqt_nsgt_pytorch"] = shim
    sys.path.insert(0, REF)
    try:
        mod = importlib.import_module("networks.cqtdiff+")
    finally:
        sys.path.remove(REF)
        if saved is not None:
            sys.modules["cqt_nsgt_pytorch"] = saved
        else:
            del sys.modules["cqt_nsgt_pytorch"]
    return mod.Unet_CQT_oct_with_attention


def test_same_init_same_keys_same_output():
    from babe_b200.denoiser import CQTDiffPlus
    args = _small_args()
    Ref = _reference_net_class()
    torch.manual_seed(0)
    ref = Ref(args, torch.device("cpu"))
    torch.manual_seed(0)
    mine = CQTDiffPlus(args, "cpu", cqt=OracleCQT(3, 8, fs=22050, audio_len=4096))
    sr, sm = ref.state_dict(), mine.state_dict()
    assert list(sr.keys()) == list(sm.keys())
    for k in sr:
        assert torch.equal(sr[k], sm[k]), k            # identical random init under one seed
    mine.load_state_dict(sr)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 4096, generator=g) * 0.1
    sigma = torch.tensor([[-0.5], [0.3]])
    # make the zero-initialised gates matter
    with torch.no_grad():
        for n, p in mine.named_parameters():
            if ".gate." in n and n.endswith("weight"):
                p.mul_(1e6)
        ref.load_state_dict(mine.state_dict())
    yr, ym = ref(x, sigma), mine(x, sigma)
    assert ym.shape == x.shape
    assert rel_l2(ym.detach(), yr.detach()) < 1e-5
    # and its input gradient
    xr, xm = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    (gr,) = torch.autograd.grad(ref(xr, sigma).pow(2).sum(), xr)
    (gm,) = torch.autograd.grad(mine(xm, sigma).pow(2).sum(), xm)
    assert rel_l2(gm, gr) < 1e-5
