"""ctypes binding of libbabe_b200.so (the C ABI in include/babe_b200.h).

There is NO fallback: if the shared library is missing or a call fails the
caller gets an exception.  Build it with ``python -m babe_b200.build``.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_longlong, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BABE_B200_LIB") or os.path.join(_HERE, "libbabe_b200.so")

BABE_OK, BABE_EBADARG, BABE_EUNSUPPORTED, BABE_ECUDA = 0, -1, -2, -3
MAX_BREAKPOINTS = 16


class BabeError(RuntimeError):
    pass


class FitConfig(ctypes.Structure):
    """``babe_fit_config`` of include/babe_b200.h."""
    _fields_ = [("mu_fc", c_float), ("mu_A", c_float), ("fcmin", c_float), ("fcmax", c_float),
                ("Amin", c_float), ("Amax", c_float), ("tol_fc", c_float), ("tol_A", c_float),
                ("max_iter", c_int), ("clamp_fc", c_int), ("clamp_A", c_int),
                ("only_negative_A", c_int)]


MAX_FACTORS = 12
MAX_OCTAVES = 16


class FftFactors(ctypes.Structure):
    """``babe_fft_factors`` of include/babe_b200.h."""
    _fields_ = [("n", c_int), ("nf", c_int), ("radix", c_int * MAX_FACTORS)]


class CqtPlan(ctypes.Structure):
    """``babe_cqt_plan`` of include/babe_b200.h (field order matters)."""
    _fields_ = [("Ls", c_int), ("Nc", c_int), ("f1", FftFactors), ("f2", FftFactors),
                ("roots1", c_void_p), ("roots2", c_void_p), ("tw_nc", c_void_p), ("tw_ls", c_void_p),
                ("numocts", c_int), ("binsoct", c_int), ("M", c_int * MAX_OCTAVES),
                ("fm", FftFactors * MAX_OCTAVES), ("rootsm", c_void_p * MAX_OCTAVES),
                ("band_p", c_void_p), ("band_lg", c_void_p), ("band_off", c_void_p),
                ("sum_lg", c_int), ("bin_jlo", c_void_p), ("bin_jhi", c_void_p), ("bin_src", c_void_p)]


# name -> (restype, argtypes); every symbol include/babe_b200.h declares
SIGNATURES = {
    "babe_last_error": (c_char_p, []),
    "babe_version": (c_int, []),
    "babe_sm_count": (c_int, []),
    "babe_stft_supported": (c_int, [c_int]),
    "babe_set_fused_variant": (c_int, [c_int]),
    "babe_get_fused_variant": (c_int, []),
    "babe_set_cqt_variant": (c_int, [c_int]),
    "babe_get_cqt_variant": (c_int, []),
    "babe_set_cqt_band_variant": (c_int, [c_int]),
    "babe_set_cqt_pdl": (c_int, [c_int]),
    "babe_set_fit_variant": (c_int, [c_int]),
    "babe_stft_tables_host": (c_int, [c_int, c_void_p, c_void_p]),
    "babe_design_filter": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                   c_void_p, c_void_p, c_void_p]),
    "babe_design_filter_vjp": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "babe_apply_filter_workspace": (c_size_t, [c_int, c_int, c_int]),
    "babe_apply_filter": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p,
                                  c_void_p]),
    "babe_apply_filter_rows": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_int, c_int,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p,
                                       c_void_p]),
    "babe_apply_filter_rows_known": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                             c_void_p, c_void_p, c_void_p, c_int, c_int,
                                             c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p,
                                             c_void_p, c_void_p]),
    "babe_stft": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                          c_int, c_void_p, c_void_p]),
    "babe_istft": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                           c_void_p, c_int, c_void_p]),
    "babe_fir_filter": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
                                c_void_p]),
    "babe_gn_slices": (c_int, [c_int, c_int, c_int, c_longlong]),
    "babe_net_chunks": (c_int, [c_longlong]),
    "babe_gn_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_longlong, c_int,
                              c_void_p]),
    "babe_gn_film_gelu": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                  c_longlong, c_float, c_void_p]),
    "babe_gate_residual": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_longlong,
                                   c_float, c_void_p]),
    "babe_gate_residual_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_int, c_int, c_int, c_longlong, c_float, c_void_p]),
    "babe_gn_film_gelu_bwd_reduce": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_void_p, c_int, c_int, c_int, c_longlong, c_float,
                                             c_void_p]),
    "babe_gn_film_gelu_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_longlong, c_float,
                                      c_float, c_void_p]),
    "babe_resample2": (c_int, [c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p, c_int, c_void_p]),
    "babe_stft_stats_workspace": (c_size_t, [c_int, c_int, c_int]),
    "babe_stft_stats": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "babe_stft_stats_rows_workspace": (c_size_t, [c_int, c_int, c_int]),
    "babe_stft_stats_rows": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_size_t, c_void_p]),
    "babe_stft_stats_groups_workspace": (c_size_t, [c_int, c_int, c_int]),
    "babe_stft_stats_groups": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                       c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "babe_spec_mag_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                    c_void_p, c_void_p]),
    "babe_spec_mag_grad": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                   c_void_p, c_void_p, c_void_p]),
    "babe_spec_dist_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "babe_spec_dist_grad": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                    c_void_p, c_void_p, c_void_p]),
    "babe_fit_params": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int,
                                POINTER(FitConfig), c_void_p, c_void_p]),
    "babe_fit_params_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int,
                                     POINTER(FitConfig), c_void_p, c_void_p]),
    "babe_cqt_workspace": (c_size_t, [POINTER(CqtPlan), c_int]),
    "babe_rfft": (c_int, [POINTER(CqtPlan), c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_size_t,
                          c_void_p]),
    "babe_irfft": (c_int, [POINTER(CqtPlan), c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_size_t,
                           c_void_p]),
    "babe_spectral_filter": (c_int, [POINTER(CqtPlan), c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                     c_size_t, c_void_p]),
    "babe_cqt_analysis": (c_int, [POINTER(CqtPlan), c_void_p, POINTER(c_void_p), c_int, c_int,
                                  c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "babe_cqt_synthesis": (c_int, [POINTER(CqtPlan), POINTER(c_void_p), c_int, c_void_p, c_int,
                                   c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "babe_row_noise": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p,
                               c_float, c_void_p]),
}

_lib = None


def header_symbols():
    """Function names declared in include/babe_b200.h (parsed, for the tests)."""
    import re
    path = os.path.join(os.path.dirname(_HERE), "include", "babe_b200.h")
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(babe_[a-z0-9_]+)\s*\(", text)))


def lib():
    """Load (once) and return the ctypes handle; raise if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BabeError(
                f"{LIB_PATH} is missing: the CUDA extension is not built "
                "(run `python -m babe_b200.build`); there is no CPU fallback")
        h = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)
            fn.restype = res
            fn.argtypes = args
        _lib = h
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().babe_last_error()
        msg = msg.decode() if msg else ""
        kind = {BABE_EBADARG: "bad argument", BABE_EUNSUPPORTED: "unsupported",
                BABE_ECUDA: "CUDA error"}.get(rc, f"error {rc}")
        raise BabeError(f"{what}: {kind}: {msg}")
