"""CPU: the design helpers / dispatcher of babe_b200.bandwidth_extension against the reference module
(needs BABE_REFERENCE set to a checkout of eloimoliner/BABE; skipped elsewhere) and against closed forms."""
import importlib
import math
import os
import sys
from types import SimpleNamespace as NS

import pytest
import torch

from conftest import rel_l2

REF = os.environ.get("BABE_REFERENCE", "")


def _cfg(kind):
    order = 6 if kind == "cheby1" else 200
    return NS(tester=NS(bandwidth_extension=NS(
        decimate=NS(factor=2),
        filter=NS(type=kind, order=order, fc=1000, beta=1, ripple=0.05, biquad=NS(Q=0.707), resample=NS(fs=2000)))))


def test_biquad_closed_form():
    from babe_b200 import bandwidth_extension as bwe
    b0, b1, b2, a0, a1, a2 = bwe.design_biquad_lpf(1000, 22050, 0.707)
    w0 = 2 * math.pi * 1000 / 22050
    assert abs(float(b1) - (1 - math.cos(w0))) < 1e-6 and abs(float(b0) - float(b1) / 2) < 1e-7
    assert abs(float(a0) - (1 + math.sin(w0) / 2 / 0.707)) < 1e-6
    # unity gain at DC: (b0 + b1 + b2) / (a0 + a1 + a2) = 1
    assert abs(float((b0 + b1 + b2) / (a0 + a1 + a2)) - 1) < 1e-5


def test_decimate_and_dispatch():
    from babe_b200 import bandwidth_extension as bwe
    y = torch.arange(20.0).reshape(2, 10)
    assert torch.equal(bwe.apply_low_pass(y, 3, "decimate"), y[..., 0:-1:3])
    assert bwe.apply_low_pass(y, None, "unknown") is None
    assert bwe.prepare_filter(_cfg("decimate"), 22050) == 2
    assert abs(bwe.prepare_filter(_cfg("resample"), 22050) - 22050 / 2000) < 1e-12


@pytest.mark.skipif(not os.path.isdir(REF), reason="BABE_REFERENCE (reference checkout) not set")
@pytest.mark.parametrize("kind", ["firwin", "firwin_hpf", "cheby1", "biquad", "resample", "decimate"])
def test_prepare_filter_matches_reference(kind):
    from babe_b200 import bandwidth_extension as bwe
    sys.path.insert(0, REF)
    try:
        ref = importlib.import_module("utils.bandwidth_extension")
    finally:
        sys.path.remove(REF)
    a, b = bwe.prepare_filter(_cfg(kind), 22050), ref.prepare_filter(_cfg(kind), 22050)
    if isinstance(b, tuple):
        assert len(a) == len(b)
        for u, v in zip(a, b):
            assert rel_l2(torch.as_tensor(u), torch.as_tensor(v)) < 1e-7
    elif torch.is_tensor(b):
        assert a.shape == b.shape and rel_l2(a, b) < 1e-7
    else:
        assert a == b


@pytest.mark.skipif(not os.path.isdir(REF), reason="BABE_REFERENCE (reference checkout) not set")
def test_iir_models_match_reference():
    """The library-delegated observation models (outside the hand-written path) behave like the reference's."""
    from babe_b200 import bandwidth_extension as bwe
    sys.path.insert(0, REF)
    try:
        ref = importlib.import_module("utils.bandwidth_extension")
    finally:
        sys.path.remove(REF)
    y = torch.randn(2, 2000, generator=torch.Generator().manual_seed(0)) * 0.05
    for kind in ("cheby1", "biquad", "resample"):
        f = ref.prepare_filter(_cfg(kind), 22050)
        out, want = bwe.apply_low_pass(y, f, kind), ref.apply_low_pass(y, f, kind)
        assert torch.isfinite(want).all()
        assert rel_l2(out, want) < 1e-6
