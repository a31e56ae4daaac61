"""CPU: babe_b200.edm.EDM against the reference class diff_params/edm.py: the sampler's schedules against the
values the reference produced (tests/golden/fit_sampler.npz), and -- with BABE_REFERENCE set to a checkout of
eloimoliner/BABE -- schedules, preconditioning, training-side members under the same seeds."""
import importlib
import os
import sys
import types

import numpy as np
import pytest
import torch

from conftest import rel_l2
from toy_model import ToyDenoiser

REF = os.environ.get("BABE_REFERENCE", "")
needs_ref = pytest.mark.skipif(not os.path.isdir(REF), reason="BABE_REFERENCE (reference checkout) not set")


def test_sampler_schedules_match_reference_golden(golden):
    """The schedule and gamma of the sampler's EDM (tester block applied, as the reference sampler does) are
    bit-identical to the reference's (tests/golden/make_golden.py)."""
    from babe_b200 import edm, sampler
    g = golden("fit_sampler.npz")
    args = sampler.make_args(sample_rate=int(g["sr"]), audio_len=g["x"].shape[1], T=4, NFFT=int(g["nfft"]))
    diff = sampler.BlindSamplerFused(ToyDenoiser(), edm.EDM(args), args).diff_params
    t = diff.create_schedule_from_initial_t(0.2, 35)
    assert np.array_equal(t.numpy(), g["sched35"])
    assert np.array_equal(diff.get_gamma(t).numpy(), g["gamma35"])
    assert np.array_equal(diff.create_schedule(35).numpy(), g["sched_full"])


def _pair():
    from babe_b200 import edm, sampler
    for name in ("plotly", "plotly.express"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.path.insert(0, REF)
    try:
        ref = importlib.import_module("diff_params.edm")
    finally:
        sys.path.remove(REF)
    args = sampler.make_args(sample_rate=22050, audio_len=4096)
    args.net = sampler._ns(use_cqt_DC_correction=True)
    return edm.EDM(args), ref.EDM(args)


@needs_ref
def test_schedules_and_preconditioning():
    mine, ref = _pair()
    for n in (4, 35):
        assert rel_l2(mine.create_schedule(n), ref.create_schedule(n)) < 1e-7
        assert rel_l2(mine.create_schedule_from_initial_t(0.2, n), ref.create_schedule_from_initial_t(0.2, n)) < 1e-7
        t = ref.create_schedule(n)
        assert torch.equal(mine.get_gamma(t), ref.get_gamma(t))
    s = torch.tensor([[0.01], [0.3], [5.0]])
    for f in ("cskip", "cout", "cin", "cnoise", "lambda_w"):
        assert rel_l2(getattr(mine, f)(s), getattr(ref, f)(s)) < 1e-7


@needs_ref
def test_training_side_members():
    mine, ref = _pair()
    np.random.seed(3)
    a = mine.sample_ptrain(16)
    np.random.seed(3)
    assert np.array_equal(a, ref.sample_ptrain(16))
    torch.manual_seed(4)
    a = mine.sample_ptrain_safe(16)
    torch.manual_seed(4)
    assert torch.equal(a, ref.sample_ptrain_safe(16))
    net = ToyDenoiser()
    x = torch.randn(3, 4096, generator=torch.Generator().manual_seed(5)) * 0.06
    torch.manual_seed(6)
    e1, s1 = mine.loss_fn(net, x)
    torch.manual_seed(6)
    e2, s2 = ref.loss_fn(net, x)
    assert torch.equal(s1, s2) and rel_l2(e1, e2) < 1e-6
