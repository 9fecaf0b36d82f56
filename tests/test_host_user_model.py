"""CudaModel on the CPU: compile errors, the build cache key, data validation, and the checks klhr_user_register makes on
a launcher table (no GPU needed)."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

from klhr_b200 import _lib, cuda_model
from klhr_b200.cuda_model import CudaModel, CudaModelBuildError, build_library, cache_key, pack_data

ROOT = Path(__file__).resolve().parent.parent
TARGETS = ROOT / "tests" / "user_targets"
TRIO_DATA = {"nu": 5.0, "s": [1.0], "a": 3.0, "b": 2.0, "alpha": 2.0, "beta": 3.0}


def test_compile_error_raises_with_nvccs_diagnostic(tmp_path, monkeypatch):
    monkeypatch.setenv("KLHR_USER_CACHE", str(tmp_path / "cache"))
    bad = tmp_path / "bad_target.cuh"
    bad.write_text("struct Target {\n    template <typename T, typename X, typename Data>\n"
                   "    __device__ static T log_density(const X& x, const Data& d) { return x[0] +; }\n};\n")
    with pytest.raises(CudaModelBuildError) as e:
        build_library(bad, "Target", [])
    msg = str(e.value)
    assert "bad_target.cuh(3)" in msg and "error" in msg, msg
    assert not list((tmp_path / "cache").glob("*.so")) and not list((tmp_path / "cache").glob(".*tmp"))


def test_cache_key_follows_source_and_keys_not_values():
    src = (TARGETS / "trio.cuh").read_text()
    keys = sorted(TRIO_DATA)
    k0 = cache_key(src, "Target", keys)
    assert cache_key(src, "Target", list(reversed(keys))) == k0                 # sorted
    assert cache_key(src + "\n// edit\n", "Target", keys) != k0
    assert cache_key(src, "Target", keys + ["extra"]) != k0
    assert cache_key(src, "Other", keys) != k0
    r1, t1, _ = pack_data(TRIO_DATA)
    r2, t2, _ = pack_data(dict(TRIO_DATA, nu=7.0, s=[2.5]))
    assert not np.array_equal(r1, r2) and np.array_equal(t1, t2)              # values live in the buffers only


def test_cache_hit_calls_no_compiler(monkeypatch):
    path = build_library(TARGETS / "trio.cuh", "Target", sorted(TRIO_DATA))  # prebuilt by __graft_entry__.build()

    def no_nvcc(*a, **k):
        raise AssertionError("nvcc called on a cache hit")
    monkeypatch.setattr(cuda_model.subprocess, "run", no_nvcc)
    m = CudaModel(TARGETS / "trio.cuh", TRIO_DATA, dim=3, device="cpu")
    m2 = CudaModel(TARGETS / "trio.cuh", dict(TRIO_DATA, nu=9.0), dim=3, device="cpu")
    assert m.library == m2.library == path
    assert m.descriptor is not None and m._host["i0"] == m2._host["i0"] >= 0
    assert m.dim() == 3 and m.parameter_names() == ["theta.1", "theta.2", "theta.3"]


def test_data_layout():
    reals, table, keys = pack_data({"n": 3, "x": [[1.0, 2.0], [3.0, 4.0]], "k": [4, 5]})
    assert keys == ["k", "n", "x"]
    assert np.array_equal(reals, [4, 5, 3, 1, 2, 3, 4])
    assert np.array_equal(table[:9], [0, 2, 9, 2, 1, 11, 3, 4, -1]) and np.array_equal(table[9:], [4, 5, 3])


@pytest.mark.parametrize("key,value", [("flag", True), ("flags", [True, False]), ("x", float("nan")),
                                       ("x", [1.0, float("inf")]), ("x", [[1.0, 2.0], [3.0]]), ("x", "abc"),
                                       ("x", None), ("x", [1.0, "a"]), ("x", 1 + 2j)])
def test_malformed_data_is_refused_by_key(key, value):
    with pytest.raises(ValueError, match=repr(key)):
        pack_data({"ok": 1.0, key: value})


def test_bad_key_and_target_are_refused():
    with pytest.raises(ValueError, match="not a C\\+\\+ identifier"):
        pack_data({"1x": 1.0})
    with pytest.raises(ValueError, match="target"):
        build_library(TARGETS / "trio.cuh", "Tar get", [])
    with pytest.raises(ValueError, match="dim"):
        CudaModel(TARGETS / "trio.cuh", TRIO_DATA, dim=0)


def _table(**kw):
    lib = _lib.load()
    t = _lib.UserTable(abi_version=_lib.ABI_VERSION)
    for f in ("step", "chain", "eval", "kl", "mh", "slice"):
        setattr(t, f, C.cast(lib.klhr_abi_version, C.c_void_p).value)          # never called: registration only
    for f in ("sizeof_step_args", "sizeof_slice_args", "sizeof_mh_args", "sizeof_kl_args", "sizeof_model_params"):
        setattr(t, f, getattr(_real_table(), f))
    for k, v in kw.items():
        setattr(t, k, v)
    return t


def _real_table():
    ulib = C.CDLL(str(build_library(TARGETS / "trio.cuh", "Target", sorted(TRIO_DATA))))
    fn = ulib.klhr_user_table
    fn.restype = C.POINTER(_lib.UserTable)
    return fn().contents


def test_register_refuses_bad_tables():
    lib = _lib.load()
    assert lib.klhr_user_register(None) == -1 and "table is NULL" in _lib.last_error()
    for kw, msg in [(dict(abi_version=3), "ABI version"), (dict(sizeof_step_args=8), "layout"),
                    (dict(sizeof_model_params=0), "layout"), (dict(mh=None), "launcher")]:
        assert lib.klhr_user_register(C.byref(_table(**kw))) < 0
        assert msg in _lib.last_error(), (kw, _lib.last_error())
    real = _real_table()
    s1 = lib.klhr_user_register(C.byref(real))
    assert s1 >= 0 and lib.klhr_user_register(C.byref(real)) == s1             # same table, same slot


def test_user_descriptor_refusals_without_a_gpu():
    lib = _lib.load()
    md = _lib.ModelDesc(id=_lib.MODEL_USER, dim=3, i0=63, i1=0, s0=0.0, s1=0.0, data0=None, data1=None)
    assert lib.klhr_model_eval(C.byref(md), _lib.KLHR_F64, None, None, None, 0, None) == -5
    assert "registered slot" in _lib.last_error()


def test_user_table_layout_matches_header():
    src = '#include <stdio.h>\n#include "klhr_user.h"\nint main(){printf("%zu\\n", sizeof(klhr_user_table_t));return 0;}'
    exe = ROOT / "build" / "user_abi_probe"
    exe.parent.mkdir(exist_ok=True)
    (exe.parent / "user_abi_probe.c").write_text(src)
    subprocess.run(["gcc", "-I", str(ROOT / "include"), str(exe.parent / "user_abi_probe.c"), "-o", str(exe)], check=True)
    size = int(subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout)
    assert size == C.sizeof(_lib.UserTable)
