"""ctypes binding of ``libklhr_sm100.so`` (declarations: ``include/klhr_sm100.h``).

The library is built in-tree by ``klhr_b200/csrc/Makefile`` (``__graft_entry__.build()``).
There is NO CPU fallback: if the shared object is missing or a CUDA device is absent, the
callers raise.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libklhr_sm100.so"

KLHR_F64, KLHR_F32 = 0, 1
FAMILY_GAUSS, FAMILY_SINH = 0, 1
MAX_NODES = 32
ABI_VERSION = 4

MODEL_IDS = {"normal": 0, "ill-normal": 1, "funnel": 2, "corr-normal": 3, "ar1": 4, "arK": 5,
             "rosenbrock": 6, "earnings": 7, "eight_schools_noncentered": 8, "eight_schools_centered": 9,
             "logistic_regression": 10, "arma11": 11}
# targets compiled from user CUDA source (klhr_b200/cuda_model.py); not a Stan program name, so not in MODEL_IDS
MODEL_USER = 12


class ModelDesc(C.Structure):
    _fields_ = [("id", C.c_int32), ("dim", C.c_int32), ("i0", C.c_int32), ("i1", C.c_int32),
                ("s0", C.c_double), ("s1", C.c_double), ("data0", C.c_void_p), ("data1", C.c_void_p)]


class FitDesc(C.Structure):
    _fields_ = [("family", C.c_int32), ("n_nodes", C.c_int32), ("n1", C.c_int32), ("n2", C.c_int32),
                ("nb", C.c_int32), ("flags", C.c_int32), ("kmax", C.c_int32), ("overrelax_K", C.c_int32),
                ("initscale", C.c_double), ("tol", C.c_double), ("scale_clip", C.c_double),
                ("gtol1", C.c_double), ("gtol2", C.c_double),
                ("step_cap", C.c_double), ("c1", C.c_double), ("basin", C.c_double), ("grad_clip", C.c_double),
                ("x", C.c_double * MAX_NODES), ("w", C.c_double * MAX_NODES)]


class DirectionDesc(C.Structure):
    _fields_ = [("mean_cols", C.c_void_p), ("sd", C.c_void_p), ("cdf", C.c_void_p),
                ("n_cols", C.c_int32), ("n_zero_cols", C.c_int32)]


class TraceDesc(C.Structure):
    _fields_ = [("eta", C.c_void_p), ("zp", C.c_void_p), ("r", C.c_void_p), ("accept", C.c_void_p),
                ("evals", C.c_void_p), ("rho", C.c_void_p), ("z_init", C.c_void_p),
                ("z_prop", C.c_void_p), ("u", C.c_void_p), ("init4", C.c_void_p), ("or_r", C.c_void_p),
                ("or_v", C.c_void_p), ("slice_u", C.c_void_p), ("slice_n", C.c_void_p)]


class SliceDesc(C.Structure):
    _fields_ = [("w", C.c_double), ("lower", C.c_double), ("upper", C.c_double), ("tol", C.c_double),
                ("cap", C.c_int32), ("reserved", C.c_int32)]


class AccumDesc(C.Structure):
    _fields_ = [("shift", C.c_void_p), ("pooled_s1", C.c_void_p), ("pooled_s2", C.c_void_p),
                ("chain_s1", C.c_void_p), ("chain_s2", C.c_void_p), ("accept_count", C.c_void_p),
                ("evals_total", C.c_void_p), ("draws", C.c_void_p), ("thin", C.c_int32),
                ("skip_accum_last", C.c_int32), ("thin_offset", C.c_int64)]




class UserTable(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("sizeof_step_args", C.c_int32), ("sizeof_slice_args", C.c_int32),
                ("sizeof_mh_args", C.c_int32), ("sizeof_kl_args", C.c_int32), ("sizeof_model_params", C.c_int32),
                ("step", C.c_void_p), ("chain", C.c_void_p), ("eval", C.c_void_p), ("kl", C.c_void_p),
                ("mh", C.c_void_p), ("slice", C.c_void_p)]


EXPORTS = {
    "klhr_abi_version": (C.c_int, []),
    "klhr_last_error": (C.c_size_t, [C.c_char_p, C.c_size_t]),
    "klhr_model_eval": (C.c_int, [C.POINTER(ModelDesc), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int64, C.c_void_p]),
    "klhr_step_replay": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(FitDesc), C.c_int, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.POINTER(TraceDesc), C.c_int64, C.c_void_p]),
    "klhr_run": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(FitDesc), C.POINTER(DirectionDesc), C.c_int,
                           C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_uint64,
                           C.POINTER(AccumDesc), C.POINTER(TraceDesc), C.c_void_p]),
    "klhr_mh_run": (C.c_int, [C.POINTER(ModelDesc), C.c_int, C.c_void_p, C.c_double, C.c_int64, C.c_int64, C.c_int64,
                              C.c_int32, C.c_uint64, C.POINTER(AccumDesc), C.POINTER(TraceDesc), C.c_void_p]),
    "klhr_slice_run": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(SliceDesc), C.POINTER(DirectionDesc), C.c_int,
                                 C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_uint64,
                                 C.POINTER(AccumDesc), C.POINTER(TraceDesc), C.c_void_p]),
    "klhr_slice_replay": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(SliceDesc), C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(TraceDesc), C.c_int64,
                                    C.c_void_p]),
    "klhr_kl_eval": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(FitDesc), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "klhr_math_eval": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "klhr_outer_accumulate": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "klhr_outer_scratch_doubles": (C.c_int64, [C.c_int64, C.c_int32]),
    "klhr_outer_reduce": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "klhr_corr_pack_cholesky": (C.c_int64, [C.c_void_p, C.c_int32, C.c_void_p]),
    "klhr_philox_eval": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "klhr_peak_probe": (C.c_int64, [C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "klhr_user_register": (C.c_int, [C.POINTER(UserTable)]),
    "klhr_launch_info": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(FitDesc), C.c_int, C.c_int, C.c_int,
                                   C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
}

_lib = None


class KLHRLibraryError(RuntimeError):
    pass


def load():
    """Load the shared object (once) and type its exports.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("KLHR_SM100_LIB", LIB_PATH))
    if not path.exists():
        raise KLHRLibraryError(
            f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C klhr_b200/csrc`.  klhr_b200 has no CPU fallback.")
    lib = C.CDLL(str(path))
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.klhr_abi_version() != ABI_VERSION:
        raise KLHRLibraryError("libklhr_sm100.so ABI version mismatch")
    _lib = lib
    return lib


def last_error() -> str:
    buf = C.create_string_buffer(512)
    load().klhr_last_error(buf, 512)
    return buf.value.decode("utf-8", "replace")


def check(code: int, what: str):
    if code != 0:
        raise KLHRLibraryError(f"{what} failed with code {code}: {last_error()}")
