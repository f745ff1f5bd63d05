"""ctypes binding of libgpemu.so (the C ABI declared in include/gpemu.h).

There is deliberately no fallback: if the CUDA library is missing or no sm_100 device is present every
prediction call raises.  The library is built in-tree (``make`` / ``__graft_entry__.build()``) so the
``.so`` next to this file is the one that gets loaded.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgpemu.so")

WANT_MU, WANT_VAR, WANT_DERIV, WANT_HESS, HOST_PTRS = 0x01, 0x02, 0x04, 0x08, 0x100
WANT_FWD, WANT_DERIV_FULL = 0x10, 0x20
OPT_SYMMETRIC_VARIANCE = 0x1
F32_FAST_TF32 = 0x200
F32_FORCE_3X = 0x400
MAX_TRAIN, MAX_INPUTS = 16384, 256
TRAIN_MAX_M = 1024
SOLVE_SPECTRA = 0x1000
SOLVE_MAX_D = 32
SOLVE_CONVERGED, SOLVE_MAX_ITER, SOLVE_STALLED, SOLVE_NONFINITE = 0, 1, 2, 3
SOLVE_DEFAULT_MAX_ITER = 50
SEARCH_MAX_K = 16
SEARCH_PW_MAX_E_BANDS, SEARCH_PW_MAX_E_SPECTRA = 48, 12

# every symbol include/gpemu.h declares (tests/test_abi.py checks the header against this list and the .so)
SYMBOLS = (
    "gpe_last_error", "gpe_version", "gpe_device_count", "gpe_model_create", "gpe_model_create_ex", "gpe_model_destroy",
    "gpe_predict", "gpe_model_plan", "gpe_predict_f32", "gpe_predict_wrap", "gpe_multi_create", "gpe_multi_predict", "gpe_multi_predict_device",
    "gpe_multi_destroy", "gpe_multi_bank_create", "gpe_multi_bank_predict", "gpe_multi_bank_cost",
    "gpe_bank_create", "gpe_bank_destroy", "gpe_bank_predict", "gpe_bank_predict_ex",
    "gpe_bank_cost", "gpe_bank_cost_host", "gpe_bank_forward_cost", "gpe_bank_forward_cost_host",
    "gpe_multi_bank_forward_cost", "gpe_bank_cost_ex", "gpe_bank_cost_host_ex", "gpe_bank_forward_cost_ex",
    "gpe_bank_forward_cost_host_ex", "gpe_multi_bank_cost_ex", "gpe_multi_bank_forward_cost_ex", "gpe_bank_project", "gpe_bank_forward", "gpe_measure_fp64_peaks", "gpe_launch_count",
    "gpe_trainer_create", "gpe_trainer_eval", "gpe_trainer_destroy", "gpe_bank_solve", "gpe_multi_bank_solve",
    "gpe_bank_search", "gpe_multi_bank_search",
    "gpe_bank_cost_pw", "gpe_bank_solve_pw", "gpe_bank_search_pw", "gpe_multi_bank_cost_pw", "gpe_multi_bank_solve_pw",
    "gpe_multi_bank_search_pw", "gpe_bank_solve_series", "gpe_multi_bank_solve_series",
)


class SolveOpts(C.Structure):
    """``gpe_solve_opts`` of include/gpemu.h."""
    _fields_ = [("max_iter", C.c_int), ("ftol", C.c_double), ("xtol", C.c_double), ("gtol", C.c_double),
                ("lambda0", C.c_double), ("lower", C.c_void_p), ("upper", C.c_void_p), ("prior_mean", C.c_void_p),
                ("prior_ld", C.c_int64), ("prior_prec", C.c_void_p)]


class GpemuError(RuntimeError):
    """A libgpemu call returned a negative status."""


_lib = None


def load():
    """Load libgpemu.so once and declare the prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GpemuError(
            f"{LIB_PATH} not found: build it with `make` (or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "gp_emulator_b200 has no CPU fallback for prediction.")
    lib = C.CDLL(LIB_PATH)
    dp = C.c_void_p  # all array arguments are raw addresses (host or device)
    lib.gpe_last_error.restype = C.c_char_p
    lib.gpe_last_error.argtypes = []
    lib.gpe_version.restype = C.c_int
    lib.gpe_device_count.restype = C.c_int
    lib.gpe_launch_count.restype = C.c_int64
    lib.gpe_model_create.restype = C.c_int
    lib.gpe_model_create.argtypes = [C.c_int, C.c_int, C.c_int, dp, dp, dp, dp, C.POINTER(C.c_void_p)]
    lib.gpe_model_create_ex.restype = C.c_int
    lib.gpe_model_create_ex.argtypes = [C.c_int, C.c_int, C.c_int, dp, dp, dp, dp, C.c_uint, C.POINTER(C.c_void_p)]
    lib.gpe_model_destroy.restype = C.c_int
    lib.gpe_model_destroy.argtypes = [C.c_void_p]
    lib.gpe_predict.restype = C.c_int
    lib.gpe_predict.argtypes = [C.c_void_p, dp, C.c_int64, dp, dp, dp, dp, C.c_uint, C.c_void_p]
    lib.gpe_model_plan.restype = C.c_int
    lib.gpe_model_plan.argtypes = [C.c_void_p, C.c_int64, C.c_char_p, C.c_int]
    lib.gpe_predict_f32.restype = C.c_int
    lib.gpe_predict_f32.argtypes = [C.c_void_p, dp, C.c_int64, dp, dp, dp, C.c_uint, C.c_void_p]
    lib.gpe_multi_create.restype = C.c_int
    lib.gpe_multi_create.argtypes = [C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int, dp, dp, dp, dp, C.c_uint,
                                     C.POINTER(C.c_void_p)]
    lib.gpe_multi_predict.restype = C.c_int
    lib.gpe_multi_predict.argtypes = [C.c_void_p, dp, C.c_int64, dp, dp, dp, dp, C.c_uint]
    lib.gpe_multi_destroy.restype = C.c_int
    lib.gpe_multi_destroy.argtypes = [C.c_void_p]
    pp = C.POINTER(C.c_void_p)   # arrays of per-device pointers
    lib.gpe_multi_predict_device.restype = C.c_int
    lib.gpe_multi_predict_device.argtypes = [C.c_void_p, pp, C.POINTER(C.c_int64), pp, pp, pp, pp, C.c_uint, pp]
    lib.gpe_multi_bank_create.restype = C.c_int
    lib.gpe_multi_bank_create.argtypes = [C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, dp, dp, dp, dp, dp, C.c_int,
                                          C.POINTER(C.c_void_p)]
    lib.gpe_multi_bank_predict.restype = C.c_int
    lib.gpe_multi_bank_predict.argtypes = [C.c_void_p, dp, C.c_int64, dp, dp, dp, dp, dp, dp, C.c_uint]
    lib.gpe_multi_bank_cost.restype = C.c_int
    lib.gpe_multi_bank_cost.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, dp, dp]
    lib.gpe_bank_predict_ex.restype = C.c_int
    lib.gpe_bank_predict_ex.argtypes = [C.c_void_p, dp, C.c_int64, dp, dp, dp, dp, dp, dp, C.c_uint, C.c_void_p]
    lib.gpe_bank_cost_host.restype = C.c_int
    lib.gpe_bank_cost_host.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, dp, dp]
    lib.gpe_predict_wrap.restype = C.c_int
    lib.gpe_predict_wrap.argtypes = [dp, dp, dp, dp, dp, dp, dp, dp, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.gpe_bank_create.restype = C.c_int
    lib.gpe_bank_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, dp, dp, dp, dp, dp, C.c_int,
                                    C.POINTER(C.c_void_p)]
    lib.gpe_bank_destroy.restype = C.c_int
    lib.gpe_bank_destroy.argtypes = [C.c_void_p]
    lib.gpe_bank_predict.restype = C.c_int
    lib.gpe_bank_predict.argtypes = [C.c_void_p, dp, C.c_int64, dp, dp, dp, dp, C.c_uint, C.c_void_p]
    lib.gpe_bank_cost.restype = C.c_int
    lib.gpe_bank_cost.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, dp, dp, C.c_void_p]
    lib.gpe_bank_forward_cost.restype = C.c_int
    lib.gpe_bank_forward_cost.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, dp, dp, C.c_void_p]
    lib.gpe_bank_forward_cost_host.restype = C.c_int
    lib.gpe_bank_forward_cost_host.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, dp, dp]
    lib.gpe_multi_bank_forward_cost.restype = C.c_int
    lib.gpe_multi_bank_forward_cost.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, dp, dp]
    for name in ("gpe_bank_cost_ex", "gpe_bank_forward_cost_ex"):
        getattr(lib, name).restype = C.c_int
        getattr(lib, name).argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, dp, dp, dp, C.c_void_p]
    for name in ("gpe_bank_cost_host_ex", "gpe_bank_forward_cost_host_ex", "gpe_multi_bank_cost_ex",
                 "gpe_multi_bank_forward_cost_ex"):
        getattr(lib, name).restype = C.c_int
        getattr(lib, name).argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, dp, dp, dp]
    so = C.POINTER(SolveOpts)
    lib.gpe_bank_solve.restype = C.c_int
    lib.gpe_bank_solve.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, so, dp, dp, dp, dp, dp, dp, C.c_uint,
                                   C.c_void_p]
    lib.gpe_multi_bank_solve.restype = C.c_int
    lib.gpe_multi_bank_solve.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, so, dp, dp, dp, dp, dp, dp, C.c_uint]
    lib.gpe_bank_search.restype = C.c_int
    lib.gpe_bank_search.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, C.c_int64, dp, C.c_int, dp, dp, C.c_uint,
                                    C.c_void_p]
    lib.gpe_multi_bank_search.restype = C.c_int
    lib.gpe_multi_bank_search.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, C.c_int64, dp, C.c_int, dp, dp, C.c_uint]
    # per-point weights: the same arguments plus weights_ld after weights (the cost calls also take flags)
    lib.gpe_bank_cost_pw.restype = C.c_int
    lib.gpe_bank_cost_pw.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, C.c_int64, dp, dp, dp, C.c_uint, C.c_void_p]
    lib.gpe_multi_bank_cost_pw.restype = C.c_int
    lib.gpe_multi_bank_cost_pw.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, C.c_int64, dp, dp, dp, C.c_uint]
    lib.gpe_bank_solve_pw.restype = C.c_int
    lib.gpe_bank_solve_pw.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, C.c_int64, so, dp, dp, dp, dp, dp, dp,
                                      C.c_uint, C.c_void_p]
    lib.gpe_multi_bank_solve_pw.restype = C.c_int
    lib.gpe_multi_bank_solve_pw.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, dp, C.c_int64, so, dp, dp, dp, dp, dp, dp,
                                            C.c_uint]
    lib.gpe_bank_search_pw.restype = C.c_int
    lib.gpe_bank_search_pw.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, C.c_int64, dp, C.c_int64, C.c_int, dp, dp,
                                       C.c_uint, C.c_void_p]
    lib.gpe_multi_bank_search_pw.restype = C.c_int
    lib.gpe_multi_bank_search_pw.argtypes = [C.c_void_p, dp, C.c_int64, dp, C.c_int64, C.c_int64, dp, C.c_int64, C.c_int, dp,
                                             dp, C.c_uint]
    # time series: (S, T) after the handle, smooth_prec and coupling after opts
    lib.gpe_bank_solve_series.restype = C.c_int
    lib.gpe_bank_solve_series.argtypes = [C.c_void_p, C.c_int64, C.c_int64, dp, dp, C.c_int64, dp, C.c_int64, so, dp, dp, dp, dp,
                                          dp, dp, dp, dp, C.c_uint, C.c_void_p]
    lib.gpe_multi_bank_solve_series.restype = C.c_int
    lib.gpe_multi_bank_solve_series.argtypes = [C.c_void_p, C.c_int64, C.c_int64, dp, dp, C.c_int64, dp, C.c_int64, so, dp, dp,
                                                dp, dp, dp, dp, dp, dp, C.c_uint]
    lib.gpe_bank_project.restype = C.c_int
    lib.gpe_bank_project.argtypes = [C.c_void_p, dp, dp, C.c_int64, dp, dp, C.c_void_p]
    lib.gpe_bank_forward.restype = C.c_int
    lib.gpe_bank_forward.argtypes = [C.c_void_p, dp, C.c_int64, dp, dp]
    lib.gpe_measure_fp64_peaks.restype = C.c_int
    lib.gpe_measure_fp64_peaks.argtypes = [C.c_int, dp]
    lib.gpe_trainer_create.restype = C.c_int
    lib.gpe_trainer_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, dp, dp, C.POINTER(C.c_void_p)]
    lib.gpe_trainer_eval.restype = C.c_int
    lib.gpe_trainer_eval.argtypes = [C.c_void_p, C.c_int, dp, dp, dp, dp, dp]
    lib.gpe_trainer_destroy.restype = C.c_int
    lib.gpe_trainer_destroy.argtypes = [C.c_void_p]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().gpe_last_error().decode("utf-8", "replace")
        raise GpemuError(f"libgpemu error {rc}: {msg}")


def f64c(a):
    """float64, C-contiguous numpy view/copy of ``a``."""
    return np.ascontiguousarray(a, dtype=np.float64)


def addr(a):
    """Raw address of a numpy array, a torch tensor, or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.__array_interface__["data"][0]   # (a.ctypes.data builds a helper object: 2.6 us against 0.5 us)
    return a.data_ptr()  # torch tensor


def measure_fp64_peaks(device=0):
    """Live FP64 pipe peaks of ``device`` (dict); the roofline denominators bench.py reports against."""
    out = np.zeros(9)
    check(load().gpe_measure_fp64_peaks(int(device), out.ctypes.data))
    keys = ("dfma_tflops", "dmma_tflops", "mixed_tflops", "mixed_dfma_tflops", "mixed_dmma_tflops",
            "gpe_exp_gps", "cuda_exp_gps", "sm_mhz_fp64_load", "sms")
    return dict(zip(keys, out.tolist()))
