"""Every built-in Stan target on the host, without a GPU: the model ids of the C header against the Python map, and for
each program on small data its dimension, parameter names, descriptor fields, data buffers and transforms."""
import re
from pathlib import Path

import numpy as np
import pytest
import torch

import klhr_b200 as kb
from klhr_b200 import _lib

ROOT = Path(__file__).resolve().parent.parent


def header_model_ids():
    text = (ROOT / "include" / "klhr_sm100.h").read_text()
    return {k: int(v) for k, v in re.findall(r"\bKLHR_MODEL_(\w+)\s*=\s*(\d+)", text)}


def test_model_ids_match_the_header():
    ids = header_model_ids()
    user = ids["USER"]
    assert sorted(_lib.MODEL_IDS.values()) == list(range(user))
    assert _lib.MODEL_USER == user and ids["COUNT"] == user + 1
    assert sorted(v for k, v in ids.items() if k not in ("USER", "COUNT")) == list(range(user))


def test_every_model_id_has_a_target_record():
    from klhr_b200.bsmodel import _TARGETS
    assert set(_TARGETS) == set(_lib.MODEL_IDS)


ARK_Y = [1.0, 2.0, 0.5, -1.0, 3.0, 2.5]
ES = {"J": 3, "y": [28.0, 8.0, -3.0], "sigma": [15.0, 10.0, 16.0]}
ES_DATA0 = np.array(ES["y"] + [1.0 / 225.0, 1.0 / 100.0, 1.0 / 256.0])


def ark_stats(y, K):
    """[X'X | X'y | y'y] of the AR(K) regression, with rows [1, y_t, .., y_{t+K-1}] and targets y_{t+K}."""
    rows = [[1.0] + y[t:t + K] for t in range(len(y) - K)]
    targets = y[K:]
    G = [sum(r[i] * r[j] for r in rows) for i in range(K + 1) for j in range(K + 1)]
    c = [sum(r[i] * yt for r, yt in zip(rows, targets)) for i in range(K + 1)]
    return np.array(G + c + [sum(yt * yt for yt in targets)])


# name: data, dim, (i0, i1, s0, s1), data0 on the host (None: no buffer), whether the descriptor keeps data0 in fp64 for
# every dtype, the parameter names, and the constrained-scale transforms as (index, "exp" | "tanh_half")
CASES = {
    "normal": ({"D": 3}, 3, (0, 0, 0.0, 0.0), None, False, ["y.1", "y.2", "y.3"], []),
    "ill-normal": ({"D": 4}, 4, (0, 0, 0.0, 0.0), np.array([4.0, 1.0, 4.0 / 9.0, 0.25]), False,
                   ["y.1", "y.2", "y.3", "y.4"], []),
    "funnel": ({"D": 3}, 4, (3, 0, 0.0, 0.0), None, False, ["double_log_sigma", "alpha.1", "alpha.2", "alpha.3"], []),
    "corr-normal": ({"N": 4, "rho": 0.5}, 4, (0, 0, 0.0, 0.0),
                    np.array([[4, -2, 0, 0], [-2, 5, -2, 0], [0, -2, 5, -2], [0, 0, -2, 4]]).reshape(-1) / 3.0, False,
                    ["y.1", "y.2", "y.3", "y.4"], []),
    "ar1": ({"N": 5}, 5, (0, 0, 0.9, 1.0 / 0.19), None, False, ["y.1", "y.2", "y.3", "y.4", "y.5"], []),
    "arK": ({"K": 2, "T": 6, "y": ARK_Y}, 4, (2, 4, 0.0, 0.0), ark_stats(ARK_Y, 2), True,
            ["alpha", "beta.1", "beta.2", "sigma"], [(3, "exp")]),
    "rosenbrock": ({"D": 2}, 4, (2, 0, 0.0, 0.0), None, False, ["v.1", "v.2", "theta.1", "theta.2"], []),
    "earnings": ({"N": 3, "earn": [10.0, 20.0, 30.0], "height": [60.0, 65.0, 70.0]}, 4, (0, 0, 0.0, 0.0),
                 np.array([3.0, 60.0, 195.0, 1400.0, 4000.0, 12725.0]), True, ["beta.1", "beta.2", "sigma", "s"],
                 [(2, "exp"), (3, "exp")]),
    "eight_schools_noncentered": (ES, 5, (3, 0, 0.0, 0.0), ES_DATA0, False,
                                  ["theta_trans.1", "theta_trans.2", "theta_trans.3", "mu", "tau"], [(4, "exp")]),
    "eight_schools_centered": (ES, 5, (3, 0, 0.0, 0.0), ES_DATA0, False,
                               ["mu", "tau", "theta.1", "theta.2", "theta.3"], [(1, "exp")]),
    "logistic_regression": ({"N": 3, "K": 2, "x": [[0.5, -1.0], [1.5, 2.0], [-0.5, 0.0]], "y": [1, 0, 1]}, 3,
                            (3, 2, 0.0, 0.0),
                            np.array([1, 0.5, -1, 1, 1.5, 2, 1, -0.5, 0, 1, 0, 1], dtype=np.float64), False,
                            ["alpha", "beta.1", "beta.2"], []),
    "arma11": ({"T": 3, "y": [0.1, -0.4, 1.2]}, 4, (3, 0, 0.0, 0.0), np.array([0.1, -0.4, 1.2]), False,
               ["mu", "phi", "theta", "sigma"], [(1, "tanh_half"), (2, "tanh_half"), (3, "exp")]),
}


def test_cases_cover_every_model():
    assert set(CASES) == set(_lib.MODEL_IDS)


def model(name, data=None):
    return kb.BSModel(stan_file=f"stan/{name}.stan", data=CASES[name][0] if data is None else data, device="cpu")


@pytest.mark.parametrize("name", sorted(CASES))
def test_host_data_and_parameter_names(name):
    _, dim, (i0, i1, s0, s1), data0, _, names, _ = CASES[name]
    m = model(name)
    h = m._host
    assert m.dim() == dim and m.parameter_names() == names
    assert (h["i0"], h["i1"]) == (i0, i1)
    assert np.isclose(h["s0"], s0, rtol=1e-15, atol=0) and np.isclose(h["s1"], s1, rtol=1e-14, atol=0)
    if data0 is None:
        assert h["data0"] is None
    else:
        assert h["data0"].dtype == np.float64 and h["data0"].shape == data0.shape
        assert np.allclose(h["data0"], data0, rtol=1e-15, atol=1e-15)
    assert h.get("data1") is None


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_descriptor(name, dtype):
    _, dim, (i0, i1, s0, s1), data0, keeps_fp64, _, _ = CASES[name]
    m = model(name)
    d = m.descriptor(dtype)
    assert (d.id, d.dim, d.i0, d.i1, d.s0, d.s1) == (_lib.MODEL_IDS[name], dim, i0, i1, m._host["s0"], m._host["s1"])
    assert d.data1 is None
    _, buf, buf1 = m._cache[(dtype, "cpu")]
    assert buf1 is None
    if data0 is None:
        assert d.data0 is None and buf is None
        return
    assert d.data0 == buf.data_ptr() and buf.device.type == "cpu" and buf.is_contiguous()
    assert buf.dtype == (torch.float64 if keeps_fp64 else dtype)
    assert torch.equal(buf, torch.as_tensor(m._host["data0"]).to(buf.dtype))


@pytest.mark.parametrize("N", [128, 256])
def test_corr_normal_packs_the_cholesky_factor_at_the_dense_sizes(N):
    """data1 is the packed lower Cholesky factor of P (fp64, klhr_corr_pack_cholesky), passed with fp64 descriptors
    only: unpacked, it is lower triangular and L L' = P."""
    m = model("corr-normal", {"N": N, "rho": 0.5})
    h = m._host
    T = N // 8
    assert h["data1"].dtype == np.float64 and h["data1"].shape == (64 * T * (T + 1) // 2,)
    L = np.zeros((N, N))
    o = iter(h["data1"])
    for nt in range(T):
        for p in range(nt, T):
            for lane in range(32):
                r8, k4 = lane >> 2, lane & 3
                L[8 * p + k4, 8 * nt + r8] = next(o)
                L[8 * p + 4 + k4, 8 * nt + r8] = next(o)
    P = h["data0"].reshape(N, N)
    assert np.array_equal(L, np.tril(L)) and np.allclose(L @ L.T, P, rtol=0, atol=1e-12)
    d64 = m.descriptor(torch.float64)
    assert d64.data1 == m._cache[(torch.float64, "cpu")][2].data_ptr()
    assert torch.equal(m._cache[(torch.float64, "cpu")][2], torch.as_tensor(h["data1"]))
    assert m.descriptor(torch.float32).data1 is None


def transformed(x, spec, inverse, lib):
    """The closed forms: exp / log, and tanh(x / 2) / 2 atanh(x)."""
    out = x.clone() if lib is torch else x.copy()
    for k, kind in spec:
        if kind == "exp":
            out[..., k] = lib.log(x[..., k]) if inverse else lib.exp(x[..., k])
        else:
            atanh = torch.atanh if lib is torch else np.arctanh
            out[..., k] = 2.0 * atanh(x[..., k]) if inverse else lib.tanh(0.5 * x[..., k])
    return out


@pytest.mark.parametrize("name", sorted(CASES))
def test_constrain_and_unconstrain(name):
    spec = CASES[name][6]
    m = model(name)
    D = m.dim()
    x = np.linspace(-0.9, 0.8, 2 * D).reshape(2, D)
    c = m.constrain(x)
    assert c.dtype == np.float64 and np.array_equal(c, transformed(x, spec, False, np))
    assert np.array_equal(m.constrain(x[0]), c[0]) and np.array_equal(m.constrain(x[0].tolist()), c[0])
    u = m.unconstrain(c)
    assert np.array_equal(u, transformed(c, spec, True, np)) and np.allclose(u, x, rtol=1e-14, atol=1e-15)
    xt = torch.as_tensor(x)
    ct = m.constrain(xt)
    assert torch.is_tensor(ct) and torch.equal(ct, transformed(xt, spec, False, torch))
    ut = m.unconstrain(ct)
    assert torch.equal(ut, transformed(ct, spec, True, torch)) and torch.allclose(ut, xt, rtol=1e-14, atol=1e-15)
    assert torch.equal(xt, torch.as_tensor(x)) and ct.data_ptr() != xt.data_ptr()      # the input is not modified
