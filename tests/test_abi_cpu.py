"""CPU: the C-ABI library loads and exports every symbol include/babe_b200.h
declares (no compute calls -- there is no GPU here)."""
import ctypes
import os

import numpy as np
import pytest

from babe_b200 import _lib, build


@pytest.fixture(scope="module")
def handle():
    build.build()
    return _lib.lib()


def test_header_symbols_exported(handle):
    names = _lib.header_symbols()
    assert len(names) >= 10
    for n in names:
        assert hasattr(handle, n), f"{n} declared in include/babe_b200.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature in babe_b200/_lib.py"
    for n in _lib.SIGNATURES:
        assert n in names, f"{n} bound in _lib.py but not declared in the header"


def test_version_and_errors(handle):
    assert handle.babe_version() >= 100
    assert handle.babe_stft_supported(4096) == 1
    assert handle.babe_stft_supported(1000) == 0
    # argument validation happens before any CUDA call
    rc = handle.babe_stft_tables_host(1000, None, None)
    assert rc == _lib.BABE_EUNSUPPORTED
    assert b"unsupported" in handle.babe_last_error().lower()
    with pytest.raises(_lib.BabeError):
        _lib.check(rc, "tables")


def test_kernel_selection_rejects_removed_values(handle):
    """The A/B setters accept only the implementations the library still has; a rejected value changes nothing."""
    for setter, v in [("babe_set_cqt_variant", 0), ("babe_set_cqt_variant", 1), ("babe_set_cqt_band_variant", 0),
                      ("babe_set_cqt_band_variant", 3), ("babe_set_fit_variant", 1)]:
        assert getattr(handle, setter)(v) == _lib.BABE_EBADARG, (setter, v)
    assert handle.babe_get_cqt_variant() == 2


def test_host_tables(handle):
    for nfft in (512, 1024, 2048, 4096):
        win = np.empty(nfft, np.float32)
        tw = np.empty(2 * nfft, np.float32)
        assert handle.babe_stft_tables_host(nfft, win.ctypes.data, tw.ctypes.data) == 0
        n = np.arange(nfft)
        assert np.allclose(win, 0.54 - 0.46 * np.cos(2 * np.pi * n / nfft), atol=1e-7)
        c = tw[0::2] + 1j * tw[1::2]
        assert np.allclose(np.abs(c), 1.0, atol=1e-6)
        assert np.allclose(c, np.exp(-2j * np.pi * n / nfft), atol=1e-6)


def test_no_cpu_fallback():
    """Product ops must refuse CPU tensors instead of silently computing."""
    import torch
    from babe_b200 import blind_bwe_utils as bu
    x = torch.zeros(1, 2048)
    H = torch.ones(513)
    with pytest.raises(_lib.BabeError):
        bu.apply_filter(x, H, 1024)
