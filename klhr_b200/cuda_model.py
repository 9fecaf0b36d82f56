"""``CudaModel``: sample a target written as one CUDA device function, without changing the library.

The user writes a struct with one templated device function (README, "Your own target")::

    struct Target {
        template <typename T, typename X, typename Data>
        __device__ static T log_density(const X& x, const Data& d);
    };

``CudaModel`` compiles it with nvcc into a shared library that instantiates every kernel of the library for
``UserModel<double, Target>`` and ``UserModel<float, Target>`` (``csrc/klhr_user.cuh``), registers the library's
launcher table with ``libklhr_sm100.so`` and then has the ``BSModel`` surface: the samplers and the engine run it like a
built-in target.  Line derivatives come from forward-mode Taylor arithmetic (``csrc/klhr_ad.cuh``).

Compiled libraries are cached in ``klhr_b200/_user_cache`` (or ``$KLHR_USER_CACHE``), keyed by a hash of the user
source, the target name, the sorted data keys, the library's device headers and the compiler flags -- not by the data
values, so one build serves every data set with the same keys.  On a hit nvcc is not called.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import re
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import torch

from . import _lib
from .bsmodel import BSModel

_HERE = Path(__file__).resolve().parent
_CSRC = _HERE / "csrc"
_INCLUDE = _HERE.parent / "include"
DEFAULT_CACHE = _HERE / "_user_cache"
# the Makefile's flags (csrc/Makefile NVFLAGS) plus -shared; hidden visibility keeps two user libraries' kernels apart
NVFLAGS = ["-O3", "-std=c++17", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
           "-Xptxas", "-v", "--expt-relaxed-constexpr", "-shared", "-Xcompiler", "-fvisibility=hidden"]

_IDENT = re.compile(r"^[A-Za-z_][A-Za-z0-9_]*$")
_LOADED = {}          # library path -> (CDLL, slot): each library is loaded and registered once per process


class CudaModelBuildError(RuntimeError):
    """nvcc rejected the user target; the message carries nvcc's diagnostic."""


def cache_dir() -> Path:
    return Path(os.environ.get("KLHR_USER_CACHE", DEFAULT_CACHE))


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"),
              str(Path(os.environ.get("CUDA_HOME", "/usr/local/cuda")) / "bin" / "nvcc")):
        if c and Path(c).exists():
            return c
    raise CudaModelBuildError("nvcc not found (set NVCC or CUDA_HOME): a user target that is not in the cache "
                              "must be compiled")


def cache_key(source: str, target: str, keys) -> str:
    """Hash of what the compiled library depends on: the source, the target name, the sorted data keys, the device
    headers of the library and the flags."""
    h = hashlib.sha256()
    for part in (source, target, "\0".join(sorted(keys)), " ".join(NVFLAGS)):
        h.update(part.encode())
        h.update(b"\0")
    for p in sorted(_CSRC.glob("*.cuh")) + sorted(_INCLUDE.glob("*.h")):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    return h.hexdigest()[:32]


def translation_unit(cuda_file, target: str, keys) -> str:
    """The generated translation unit: the library, the field constants, the user's file, the instantiations."""
    names = sorted(keys)
    fields = ", ".join(f"{k} = {i}" for i, k in enumerate(names))
    return (f'#include "{_CSRC / "klhr_user.cuh"}"\n'
            f"namespace field {{ enum : int {{ {fields} }}; }}\n"
            f'#include "{Path(cuda_file).resolve()}"\n'
            f"KLHR_DEFINE_USER_TARGET(::{target})\n")


def build_library(cuda_file, target: str = "Target", keys=()) -> Path:
    """Path of the compiled library of ``target`` in ``cuda_file`` for data with these keys; compiled on a miss.
    The library is written to a temporary file and renamed into place, so processes that build at once do not
    corrupt the cache.  The ptxas log is kept next to it."""
    if not _IDENT.match(target):
        raise ValueError(f"target must be a C++ identifier, got {target!r}")
    for k in keys:
        if not _IDENT.match(k):
            raise ValueError(f"data key {k!r} is not a C++ identifier (it becomes field::{k})")
    source = Path(cuda_file).read_text()
    key = cache_key(source, target, keys)
    root = cache_dir()
    lib = root / f"libklhr_user_{key}.so"
    if lib.exists():
        return lib
    root.mkdir(parents=True, exist_ok=True)
    fd, tmp = tempfile.mkstemp(dir=root, prefix=f".{key}.", suffix=".tmp")
    os.close(fd)
    cu = Path(tmp).with_suffix(".cu")
    try:
        cu.write_text(translation_unit(cuda_file, target, keys))
        r = subprocess.run([_nvcc(), *NVFLAGS, str(cu), "-o", tmp], capture_output=True, text=True)
        if r.returncode != 0:
            raise CudaModelBuildError(f"nvcc failed to compile {target} of {cuda_file}:\n{r.stderr}{r.stdout}")
        (root / f"libklhr_user_{key}.ptxas.log").write_text(r.stderr)
        os.replace(tmp, lib)
    finally:
        cu.unlink(missing_ok=True)
        Path(tmp).unlink(missing_ok=True)
    return lib


def register(lib_path: Path) -> int:
    """Load a user target library with ctypes, check its launcher table and register it; the registry slot."""
    lib_path = Path(lib_path).resolve()
    if str(lib_path) not in _LOADED:
        ulib = C.CDLL(str(lib_path))
        fn = ulib.klhr_user_table
        fn.restype = C.POINTER(_lib.UserTable)
        fn.argtypes = []
        table = fn()
        if not table or table.contents.abi_version != _lib.ABI_VERSION:
            raise _lib.KLHRLibraryError(f"{lib_path}: launcher table missing or built for another ABI version")
        slot = _lib.load().klhr_user_register(table)
        if slot < 0:
            raise _lib.KLHRLibraryError(f"klhr_user_register failed with code {slot}: {_lib.last_error()}")
        _LOADED[str(lib_path)] = (ulib, slot)
    return _LOADED[str(lib_path)][1]


def pack_data(data: dict):
    """(reals, table, keys) of a data dict, validated: every value an int, a finite real, or a (nested) array of them.
    reals: every field flattened in C order, concatenated in sorted-key order (fp64; converted to the arithmetic type
    on the device); table: int64 header (offset into reals, length, offset into table or -1) per field, then the values
    of the integer fields (csrc/klhr_user.cuh)."""
    keys = sorted(data)
    parts, ints, header = [], [], []
    off, ioff = 0, 3 * len(keys)
    for k in keys:
        v = data[k]
        if not _IDENT.match(k):
            raise ValueError(f"data key {k!r} is not a C++ identifier (it becomes field::{k})")
        try:
            a = np.asarray(v)
        except ValueError as e:                       # ragged nesting (NumPy >= 1.24 raises)
            raise ValueError(f"data[{k!r}]: not a rectangular array ({e})") from None
        if a.dtype == np.bool_ or isinstance(v, bool):
            raise ValueError(f"data[{k!r}]: booleans are not data; give 0 / 1 integers")
        if a.dtype.kind not in "iuf":
            raise ValueError(f"data[{k!r}]: must be an int, a real or an array of them, got dtype {a.dtype}")
        if a.dtype.kind == "f" and not np.all(np.isfinite(a)):
            raise ValueError(f"data[{k!r}]: must be finite (no NaN or inf)")
        flat = a.reshape(-1)
        header += [off, flat.size, ioff if a.dtype.kind in "iu" else -1]
        if a.dtype.kind in "iu":
            ints.append(flat.astype(np.int64))
            ioff += flat.size
        parts.append(flat.astype(np.float64))
        off += flat.size
    reals = np.concatenate(parts) if parts else np.zeros(0)
    table = np.concatenate([np.asarray(header, dtype=np.int64)] + ints)
    return reals, table, keys


class CudaModel(BSModel):
    """A target written as a CUDA device function, with the ``BSModel`` surface.

    ``cuda_file``: the user's source; ``target``: the struct in it; ``data``: the data block (keys become
    ``field::<key>``); ``dim``: the number of unconstrained parameters; ``constrain`` / ``unconstrain``: optional
    callables between the unconstrained and constrained scales (identity by default); ``parameter_names``: optional."""

    def __init__(self, cuda_file, data, dim, target="Target", parameter_names=None, constrain=None,
                 unconstrain=None, device=None):
        dim = int(dim)
        if dim <= 0:
            raise ValueError(f"dim must be positive, got {dim}")
        reals, table, keys = pack_data(dict(data))
        self._stan_file = str(cuda_file)
        self._data_file = ""
        self.name = f"user:{Path(cuda_file).stem}:{target}"
        self.data = dict(data)
        self.device = torch.device(device) if device is not None else torch.device("cuda", 0)
        self._cache = {}
        self.library = build_library(cuda_file, target, keys)
        slot = register(self.library)
        self._host = dict(dim=dim, i0=slot, i1=len(keys), s0=0.0, s1=0.0, data0=reals, data1=table)
        if parameter_names is not None and len(parameter_names) != dim:
            raise ValueError(f"parameter_names has {len(parameter_names)} names for dim = {dim}")
        self._names = list(parameter_names) if parameter_names is not None else None
        self._constrain, self._unconstrain = constrain, unconstrain

    def descriptor(self, dtype=torch.float64, device=None):
        device = torch.device(device) if device is not None else self.device
        key = (dtype, str(device))
        if key not in self._cache:
            h = self._host
            # one element at least, so that the buffers have an address even when every field is empty
            buf = torch.zeros(max(1, h["data0"].size), dtype=torch.float64)
            buf[:h["data0"].size] = torch.as_tensor(h["data0"])
            buf = buf.to(device=device, dtype=dtype).contiguous()
            buf1 = torch.as_tensor(h["data1"], dtype=torch.int64).to(device=device).contiguous()
            desc = _lib.ModelDesc(id=_lib.MODEL_USER, dim=h["dim"], i0=h["i0"], i1=h["i1"], s0=0.0, s1=0.0,
                                  data0=buf.data_ptr(), data1=buf1.data_ptr() if h["i1"] > 0 else None)
            self._cache[key] = (desc, buf, buf1)
        return self._cache[key][0]

    def constrain(self, theta):
        out = theta.clone() if torch.is_tensor(theta) else np.array(theta, dtype=np.float64)
        return self._constrain(out) if self._constrain is not None else out

    def unconstrain(self, theta):
        out = theta.clone() if torch.is_tensor(theta) else np.array(theta, dtype=np.float64)
        return self._unconstrain(out) if self._unconstrain is not None else out

    def parameter_names(self):
        return list(self._names) if self._names is not None else [f"theta.{i + 1}" for i in range(self.dim())]
