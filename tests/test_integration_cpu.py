"""CPU: integration row of SURVEY section 4, against the golden the unmodified reference sampler + unmodified
reference network produced (tests/golden/integration.npz).

* the in-repo denoiser restatement (babe_b200.denoiser.CQTDiffPlus on the oracle CQT) gives the reference network's
  output, and the test-local restatement of the loop (tests/parity_loop.py) on it and on the oracle operators
  reproduces the reference run -- which validates the helper that the GPU tests run on the CUDA drop-ins through
  babe_b200.install();
* with BABE_REFERENCE set to a checkout of eloimoliner/BABE: the UNMODIFIED reference sampler on the denoiser
  restatement, and the loop restatement on the reference's OWN operator module, reproduce the same golden;
* the three Hydra callable strings resolve through babe_b200.callables (and through the reference's own dnnlib) to
  classes with the constructor signatures the reference uses (utils/setup.py:49,55; testing/blind_bwe_tester.py:214).
"""
import os
import sys
import types

import numpy as np
import pytest
import torch

from conftest import rel_l2

REF = os.environ.get("BABE_REFERENCE", "")
needs_ref = pytest.mark.skipif(not os.path.isdir(REF), reason="BABE_REFERENCE (reference checkout) not set")


def _small(golden):
    from babe_b200.sampler import make_args
    args = make_args(sample_rate=22050, audio_len=4096, num_octs=3, bins_per_oct=8, NFFT=1024, T=2, max_iter=5)
    args.network.Ns, args.network.Ss, args.network.num_dils = [8, 8, 16], [2, 2, 2], [1, 2, 2]
    args.network.attention_layers, args.network.emb_dim = [0, 0, 0, 0], 32
    return args, golden("integration.npz")


def _my_network(args, device="cpu", cqt=None):
    from babe_b200.denoiser import CQTDiffPlus
    torch.manual_seed(0)
    net = CQTDiffPlus(args, device, cqt=cqt)
    with torch.no_grad():
        for n, p in net.named_parameters():
            if ".gate." in n and n.endswith("weight"):
                p.mul_(1e6)
    for p in net.parameters():
        p.requires_grad_(False)
    return net


def _ref_modules():
    sys.path.insert(0, REF)
    for name in ("plotly", "plotly.express"):
        sys.modules.setdefault(name, types.ModuleType(name))
    import utils.blind_bwe_utils as ref_ops
    from testing.blind_bwe_sampler import BlindSampler
    from diff_params.edm import EDM
    return ref_ops, BlindSampler, EDM


def test_denoiser_restatement_matches_reference_network(golden):
    from oracle.cqt_shim import OracleCQT
    args, g = _small(golden)
    net = _my_network(args, cqt=OracleCQT(3, 8, fs=22050, audio_len=4096))
    assert rel_l2(net(torch.from_numpy(g["net_in"]), torch.from_numpy(g["net_sigma"])), g["net_out"]) < 1e-5


def test_parity_loop_helper_on_oracle_operators(golden):
    import parity_loop
    from babe_b200.edm import EDM
    from oracle import stft_filter as osf
    from oracle.cqt_shim import OracleCQT
    args, g = _small(golden)
    net = _my_network(args, cqt=OracleCQT(3, 8, fs=22050, audio_len=4096))
    torch.manual_seed(42)
    trace = []
    x, p = parity_loop.predict_blind_bwe(osf, net, EDM(args), args, torch.from_numpy(g["y"]).clone(), trace=trace)
    assert rel_l2(x, g["x"]) < 2e-5 and rel_l2(p, g["params"]) < 2e-5
    assert len(trace) == g["x_out"].shape[0]
    for i, (xi, pi, di) in enumerate(trace):
        assert rel_l2(xi, g["x_out"][i]) < 2e-5 and rel_l2(di, g["x_den"][i]) < 2e-5


@needs_ref
def test_reference_sampler_on_denoiser_restatement(golden):
    from oracle.cqt_shim import OracleCQT
    args, g = _small(golden)
    ref_ops, BlindSampler, EDM = _ref_modules()
    net = _my_network(args, cqt=OracleCQT(3, 8, fs=22050, audio_len=4096))
    assert rel_l2(net(torch.from_numpy(g["net_in"]), torch.from_numpy(g["net_sigma"])), g["net_out"]) < 1e-5
    s = BlindSampler(net, EDM(args), args, rid=True)
    torch.manual_seed(42)
    x, p, den, t, filt = s.predict_blind_bwe(torch.from_numpy(g["y"]).clone(), rid=True)
    assert rel_l2(x, g["x"]) < 1e-5 and rel_l2(p, g["params"]) < 1e-5 and rel_l2(den, g["x_den"]) < 1e-5


@needs_ref
def test_parity_loop_helper_on_reference_operators(golden):
    import parity_loop
    from oracle.cqt_shim import OracleCQT
    args, g = _small(golden)
    ref_ops, BlindSampler, EDM = _ref_modules()
    net = _my_network(args, cqt=OracleCQT(3, 8, fs=22050, audio_len=4096))
    torch.manual_seed(42)
    trace = []
    x, p = parity_loop.predict_blind_bwe(ref_ops, net, EDM(args), args, torch.from_numpy(g["y"]).clone(), trace=trace)
    assert rel_l2(x, g["x"]) < 2e-5 and rel_l2(p, g["params"]) < 2e-5
    for i, (xi, pi, di) in enumerate(trace):
        assert rel_l2(xi, g["x_out"][i]) < 2e-5 and rel_l2(di, g["x_den"][i]) < 2e-5


def test_callable_strings_resolve(golden):
    from babe_b200 import callables
    from toy_model import ToyDenoiser
    args, g = _small(golden)
    diff = callables.call_func_by_name(func_name=args.diff_params.callable, args=args)                # utils/setup.py:49
    smp = callables.call_func_by_name(func_name=args.tester.sampler_callable, model=ToyDenoiser(), diff_params=diff,
                                      args=args, rid=True)                                # blind_bwe_tester.py:214
    assert type(diff).__name__ == "EDM" and type(smp).__name__ == "BlindSamplerFused"
    net_cls = callables.get_obj_by_name(args.network.callable)                                       # utils/setup.py:55
    import inspect
    assert list(inspect.signature(net_cls.__init__).parameters)[1:3] == ["args", "device"]
    for m in ("predict_blind_bwe", "predict_bwe", "predict_bwe_AR", "predict_unconditional"):
        assert callable(getattr(smp, m))
    if os.path.isdir(REF):          # the reference's own resolver finds the same objects
        sys.path.insert(0, REF)
        sys.modules.setdefault("requests", types.ModuleType("requests"))
        try:
            from utils.dnnlib import util as ref_util
        except Exception as e:                                   # noqa: BLE001
            pytest.skip(f"reference dnnlib not importable here: {e!r}")
        assert ref_util.get_obj_by_name(args.tester.sampler_callable) is type(smp)
        assert ref_util.get_obj_by_name(args.network.callable) is net_cls
        assert ref_util.get_obj_by_name(args.diff_params.callable) is type(diff)
