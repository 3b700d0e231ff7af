"""ctypes view of include/mcmc_gpu.h and the loader of libmcmcgpu.so.

There is no CPU fallback: if the CUDA extension has not been built, or no
CUDA device is present, every entry point of the package raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# MCMC_GPU_LIB selects another build of the same library (kernel-variant experiments)
LIB_PATH = os.environ.get("MCMC_GPU_LIB") or os.path.join(_HERE, "libmcmcgpu.so")

MG_OK, MG_EINVAL, MG_EFAIL, MG_ECUDA, MG_ENOMEM = 0, 1, 2, 3, 4

# log-density kinds
FN_ZERO, FN_CONST, FN_BOX_CLOSED, FN_BOX_OPEN, FN_GAUSS_DIAG, FN_GAUSS_CORR = 0, 1, 2, 3, 4, 5
FN_GAUSS_DATA, FN_CAUCHY_DATA, FN_SHELL, FN_GAUSS_MIX = 6, 7, 8, 9
# proposal kinds
PROP_BOX, PROP_WRAP, PROP_INDEP_GAUSS, PROP_LEFT_BIASED, PROP_ONE_SIDED, PROP_MIXTURE, PROP_DE = 0, 1, 2, 3, 4, 5, 6
# into-model proposal kinds
INTO_INTERP, INTO_INDEP_GAUSS = 0, 1
LAYOUT_STEP_MAJOR, LAYOUT_CHAIN_MAJOR = 0, 1

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_int64_p = C.POINTER(C.c_int64)
c_uint8_p = C.POINTER(C.c_uint8)


class mg_logfn(C.Structure):
    _fields_ = [("kind", C.c_int32), ("dim", C.c_int32), ("scale", C.c_double),
                ("params", c_double_p), ("nparams", C.c_int64)]


class mg_proposal(C.Structure):
    _fields_ = [("kind", C.c_int32), ("dim", C.c_int32), ("params", c_double_p), ("nparams", C.c_int64)]


class mg_mcmc_cfg(C.Structure):
    _fields_ = [("nchains", C.c_int64), ("dim", C.c_int32), ("layout", C.c_int32), ("nbin", C.c_int64),
                ("nskip", C.c_int64), ("n", C.c_int64), ("chain_offset", C.c_uint64),
                ("x0_shared", C.c_int32), ("reserved", C.c_int32)]


class mg_into(C.Structure):
    _fields_ = [("kind", C.c_int32), ("nstop", C.c_int32), ("tree", C.c_void_p), ("params", c_double_p),
                ("nparams", C.c_int64)]


class mg_rj_model(C.Structure):
    _fields_ = [("like", mg_logfn), ("prior", mg_logfn), ("prop", mg_proposal), ("into", mg_into),
                ("p", C.c_double)]


class mg_rjmcmc_cfg(C.Structure):
    _fields_ = [("nchains", C.c_int64), ("nbin", C.c_int64), ("nskip", C.c_int64), ("n", C.c_int64),
                ("chain_offset", C.c_uint64), ("layout", C.c_int32), ("reserved", C.c_int32)]


class mg_nested_cfg(C.Structure):
    _fields_ = [("dim", C.c_int32), ("nlive", C.c_int32), ("nmcmc", C.c_int32), ("batch", C.c_int32),
                ("epsrel", C.c_double), ("mode_hopping_frac", C.c_double), ("max_points", C.c_int64)]


class mg_diag_cfg(C.Structure):
    _fields_ = [("n", C.c_int64), ("nchains", C.c_int64), ("dim", C.c_int32), ("maxlag", C.c_int32),
                ("split", C.c_int32), ("reserved", C.c_int32)]


class mg_tempered_cfg(C.Structure):
    _fields_ = [("nladders", C.c_int64), ("ntemps", C.c_int32), ("dim", C.c_int32), ("nbin", C.c_int64),
                ("nsteps", C.c_int64), ("swap_every", C.c_int64), ("ladder_offset", C.c_uint64),
                ("x0_shared", C.c_int32), ("reserved", C.c_int32)]


class mg_tempered_out(C.Structure):
    _fields_ = [("log_z_ss", C.c_double), ("log_z_ss_err", C.c_double), ("log_z_ti", C.c_double),
                ("log_z_ti_err", C.c_double), ("mean_ll", c_double_p), ("mean_ll_err", c_double_p),
                ("accept", c_int64_p), ("swaps_accepted", c_int64_p), ("swaps_tried", c_int64_p),
                ("final", c_double_p), ("ladder_mean_ll", c_double_p)]


TEMPERED_MAX_T = 32  # MG_TEMPERED_MAX_T
DIAG_MAXLAG = 256   # MG_DIAG_MAXLAG
QUANT_MAX = 64      # MG_QUANT_MAX


def as_f64(a, shape=None) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def ptr(a: np.ndarray | None, typ=c_double_p):
    if a is None:
        return typ()
    return a.ctypes.data_as(typ)


class InvalidArgument(ValueError):
    """OCaml Invalid_argument (MG_EINVAL)."""


class Failure(RuntimeError):
    """OCaml Failure (MG_EFAIL / MG_ECUDA / MG_ENOMEM)."""


_lib = None


def load_library() -> C.CDLL:
    """Load libmcmcgpu.so; fail loudly if it was not built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA extension first "
            "(python -c 'import __graft_entry__ as g; g.build()' or make -C mcmc_ocaml_b200/csrc). "
            "There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.mg_last_error.restype = C.c_char_p
    lib.mg_last_error.argtypes = [C.c_void_p]
    lib.mg_ctx_get_epoch.restype = C.c_uint64
    lib.mg_ctx_get_epoch.argtypes = [C.c_void_p]
    lib.mg_ctx_get_stream.restype = C.c_void_p
    lib.mg_ctx_get_stream.argtypes = [C.c_void_p]
    lib.mg_ctx_launch_count.restype = C.c_int64
    lib.mg_ctx_launch_count.argtypes = [C.c_void_p]
    lib.mg_ctx_last_kernel_ms.restype = C.c_double
    lib.mg_ctx_last_kernel_ms.argtypes = [C.c_void_p]
    lib.mg_ctx_create.argtypes = [C.c_int, C.c_uint64, C.POINTER(C.c_void_p)]
    lib.mg_ctx_destroy.argtypes = [C.c_void_p]
    lib.mg_ctx_destroy.restype = None
    lib.mg_ctx_set_seed.argtypes = [C.c_void_p, C.c_uint64]
    lib.mg_ctx_set_epoch.argtypes = [C.c_void_p, C.c_uint64]
    lib.mg_ctx_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    for name in ("mg_bounds_volume", "mg_nested_log_total_error"):
        if hasattr(lib, name):
            getattr(lib, name).restype = C.c_double
    if hasattr(lib, "mg_bounds_volume"):
        lib.mg_bounds_volume.argtypes = [c_double_p, c_double_p, C.c_int32]
    if hasattr(lib, "mg_nested_log_total_error"):
        lib.mg_nested_log_total_error.argtypes = [C.c_double, C.c_double, C.c_int32]
    if hasattr(lib, "mg_kdtree_destroy"):
        lib.mg_kdtree_destroy.restype = None
        lib.mg_kdtree_destroy.argtypes = [C.c_void_p]
    if hasattr(lib, "mg_ellipse_tree_destroy"):
        lib.mg_ellipse_tree_destroy.restype = None
        lib.mg_ellipse_tree_destroy.argtypes = [C.c_void_p]
        lib.mg_ellipse_tree_info.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.mg_ellipse_tree_export.argtypes = [C.c_void_p] + [C.c_void_p] * 10
    for name in ("mg_stats_quantiles_dev", "mg_stats_quantiles", "mg_stats_order_statistics_dev", "mg_comm_quantiles"):
        fn = getattr(lib, name)
        fn.restype = C.c_int
        items = c_int64_p if name == "mg_stats_order_statistics_dev" else c_double_p
        fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, items, C.c_int32, c_double_p]
    for name, first in (("mg_evidence_tempered", C.c_void_p), ("mg_evidence_tempered_sharded", C.c_void_p)):
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = [first, C.POINTER(mg_logfn), C.POINTER(mg_logfn), C.POINTER(mg_proposal), c_double_p,
                       C.POINTER(mg_tempered_cfg), c_double_p, C.POINTER(mg_tempered_out)]
    _lib = lib
    return lib


def declared_symbols() -> list[str]:
    """Every function include/mcmc_gpu.h declares (used by the CPU tests)."""
    import re
    hdr = os.path.join(os.path.dirname(_HERE), "include", "mcmc_gpu.h")
    text = open(hdr).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mg_[a-z0-9_]+)\s*\(", text)))
