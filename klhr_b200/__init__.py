"""klhr_b200 -- B200-native KL Hit-and-Run (the hot path of roualdes/klhr).

Public surface mirrors the reference: ``BSModel`` (reference bsmodel.py), ``KLHR``
(klhr.py), ``KLHRSINH`` (klhr_sinh.py), plus the comparison samplers ``SUBKLHRSINH``
(sub_klhr_sinh.py), ``Slice`` (slice.py) and ``MH`` (mh.py).  Everything numeric runs in hand-written sm_100a
CUDA kernels behind the C ABI of ``libklhr_sm100.so`` (include/klhr_sm100.h); there is no
CPU fallback.
"""
from .bsmodel import BSModel
from .cuda_model import CudaModel
from .engine import (FitConfig, Direction, Trace, SliceConfig, step_replay, run, slice_replay, slice_run, kl_eval,
                     outer_accumulate, outer_scratch, outer_reduce, launch_info, gauss_hermite)

__all__ = ["BSModel", "CudaModel", "FitConfig", "Direction", "Trace", "step_replay", "run", "outer_accumulate", "outer_scratch", "outer_reduce",
           "launch_info", "gauss_hermite", "SliceConfig", "slice_replay", "slice_run", "kl_eval"]

try:  # samplers (import kept soft only so that partial checkouts still expose the engine)
    from .klhr import KLHR
    from .klhr_sinh import KLHRSINH
    from .sub_klhr_sinh import SUBKLHRSINH
    from .mh import MH
    from .slice import Slice
    __all__ += ["KLHR", "KLHRSINH", "SUBKLHRSINH", "MH", "Slice"]
except ImportError:  # pragma: no cover
    pass
