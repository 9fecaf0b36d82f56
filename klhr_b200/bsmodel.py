"""Model boundary: ``BSModel`` with the surface of reference ``bsmodel.py:5-55``.

The reference wraps ``bridgestan.StanModel`` (a Stan program compiled to a C++ ``.so`` and
called through ctypes once per evaluation).  Here the Stan program is selected by the stem of
``stan_file`` and evaluated by hand-written CUDA device functions
(``csrc/klhr_models.cuh``); ``data_file`` is the same JSON the reference passes to Stan.

    dim()                          bsmodel.py:42-43
    log_density(theta)             bsmodel.py:15-21   -inf instead of an exception
    log_density_gradient(theta)    bsmodel.py:23-30   (-inf, zeros) instead of an exception
    constrain / unconstrain / parameter_names          bsmodel.py:48-55

``theta`` may be a NumPy vector ``(D,)`` (returns Python floats / NumPy arrays like the
reference) or a batch ``(B, D)`` as a NumPy array or CUDA tensor (returns tensors on the
device).  An unknown Stan program is an explicit error -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import json
from pathlib import Path
from typing import Callable, NamedTuple

import numpy as np
import torch

from . import _lib

_DTYPES = {torch.float64: _lib.KLHR_F64, torch.float32: _lib.KLHR_F32}


def _dtype_code(dtype):
    try:
        return _DTYPES[dtype]
    except KeyError:
        raise TypeError(f"klhr_b200 computes in float64 or float32, not {dtype}") from None


def _eight_schools_data(d):
    """(J, y, sigma) of the eight-schools data block, validated: J >= 1, y and sigma of length J, sigma > 0 and finite."""
    try:
        J = int(d["J"])
        y = np.asarray(d["y"], dtype=np.float64)
        sigma = np.asarray(d["sigma"], dtype=np.float64)
    except (KeyError, TypeError) as e:
        raise ValueError(f"eight schools: data needs J, y[J] and sigma[J] ({e})") from None
    if J < 1 or J != d["J"]:
        raise ValueError(f"eight schools: J must be an integer >= 1, got {d['J']!r}")
    if y.shape != (J,) or sigma.shape != (J,):
        raise ValueError(f"eight schools: y and sigma must have length J = {J}, got {y.shape} and {sigma.shape}")
    if not np.all(np.isfinite(y)):
        raise ValueError("eight schools: y must be finite")
    if not np.all(np.isfinite(sigma) & (sigma > 0)):
        raise ValueError("eight schools: sigma must be positive and finite")
    return J, y, sigma


def _int_at_least(d, key, lo, what):
    v = d[key]
    if isinstance(v, bool) or not isinstance(v, (int, np.integer, float, np.floating)) or v != int(v) or v < lo:
        raise ValueError(f"{what}: {key} must be an integer >= {lo}, got {v!r}")
    return int(v)


def _logistic_regression_data(d):
    """(N, K, X, y) of the logistic-regression data block, validated: integers N >= 0 and K >= 1, x finite of shape
    (N, K), y of length N with every entry 0 or 1.  X = [1 | x] is the N x (K + 1) design."""
    what = "logistic regression"
    try:
        N = _int_at_least(d, "N", 0, what)
        K = _int_at_least(d, "K", 1, what)
        x = np.asarray(d["x"], dtype=np.float64)
        y = np.asarray(d["y"], dtype=np.float64)
    except KeyError as e:
        raise ValueError(f"{what}: data needs N, K, x[N, K] and y[N] ({e})") from None
    except (TypeError, ValueError) as e:
        raise ValueError(f"{what}: x and y must be numeric arrays ({e})") from None
    if N == 0 and x.size == 0:
        x = x.reshape(0, K)
    if x.shape != (N, K):
        raise ValueError(f"{what}: x must have shape (N, K) = ({N}, {K}), got {x.shape}")
    if not np.all(np.isfinite(x)):
        raise ValueError(f"{what}: x must be finite")
    if y.shape != (N,):
        raise ValueError(f"{what}: y must have length N = {N}, got shape {y.shape}")
    if not np.all((y == 0) | (y == 1)):
        raise ValueError(f"{what}: every y must be 0 or 1")
    X = np.concatenate([np.ones((N, 1)), x], axis=1)
    return N, K, X, y


def _arma11_data(d):
    """(T, y) of the ARMA(1,1) data block, validated: an integer T >= 1 and y finite of length T."""
    what = "arma11"
    try:
        T = _int_at_least(d, "T", 1, what)
        y = np.asarray(d["y"], dtype=np.float64)
    except KeyError as e:
        raise ValueError(f"{what}: data needs T and y[T] ({e})") from None
    except (TypeError, ValueError) as e:
        raise ValueError(f"{what}: y must be a numeric array ({e})") from None
    if y.shape != (T,):
        raise ValueError(f"{what}: y must have length T = {T}, got shape {y.shape}")
    if not np.all(np.isfinite(y)):
        raise ValueError(f"{what}: y must be finite")
    return T, y


# ---------------------------------------------------------------------- one record per Stan program
# prepare: the data block -> the descriptor fields that differ from the defaults (the program's "transformed data");
# names: the host fields -> the parameter names; fp64_data: data0 holds sufficient statistics that stay fp64 whatever
# the arithmetic type (klhr_models.cuh); transforms: (index or slice, kind) of every coordinate whose constrained value
# is exp(u) ("exp") or tanh(u / 2) ("tanh_half").
class _Target(NamedTuple):
    prepare: Callable[[dict], dict]
    names: Callable[[dict], list]
    fp64_data: bool = False
    transforms: tuple = ()


def _y_names(h):
    return [f"y.{i + 1}" for i in range(h["dim"])]


def _ill_normal(d):                                  # stan/ill-normal.stan:4-6
    D = int(d["D"])
    s = np.arange(1, D + 1, dtype=np.float64) / np.sqrt(float(D))
    return dict(dim=D, data0=1.0 / (s * s))


def _corr_normal(d):                                 # stan/corr-normal.stan:5-13
    N, rho = int(d["N"]), float(d["rho"])
    idx = np.arange(N)
    Sigma = rho ** np.abs(idx[:, None] - idx[None, :])
    P = np.linalg.inv(Sigma)
    P = 0.5 * (P + P.T)
    h = dict(dim=N, data0=P.reshape(-1))
    if N in (128, 256):
        # P = L L' (fp64): the dense kernels work with V = L' rho and w = L' theta (csrc/klhr_densek.cuh); L goes
        # to the device packed in the order the tensor warps consume it (klhr_corr_pack_cholesky)
        L = np.ascontiguousarray(np.tril(np.linalg.cholesky(P)), dtype=np.float64)
        lib = _lib.load()
        n = lib.klhr_corr_pack_cholesky(None, N, None)
        packed = np.empty(int(n), dtype=np.float64)
        if lib.klhr_corr_pack_cholesky(L.ctypes.data, N, packed.ctypes.data) != n:
            raise _lib.KLHRLibraryError(f"klhr_corr_pack_cholesky failed: {_lib.last_error()}")
        h["data1"] = packed
    return h


def _ar1(d):                                         # stan/ar1.stan:4-7
    alpha = 0.9
    return dict(dim=int(d["N"]), s0=alpha, s1=1.0 / (1.0 - alpha * alpha))


def _ark(d):                                         # stan/arK.stan:1-20, sufficient statistics
    K, T = int(d["K"]), int(d["T"])
    y = np.asarray(d["y"], dtype=np.float64)
    if y.shape != (T,):
        raise ValueError("arK: len(y) must equal T")
    nobs = T - K
    X = np.empty((nobs, K + 1))
    X[:, 0] = 1.0
    for k in range(K):
        X[:, 1 + k] = y[k:k + nobs]
    yt = y[K:]
    pack = np.concatenate([(X.T @ X).reshape(-1), X.T @ yt, [yt @ yt]])
    return dict(dim=K + 2, i0=K, i1=nobs, data0=pack)


def _earnings(d):                                    # stan/earnings.stan:1-17, sufficient statistics
    e = np.asarray(d["earn"], dtype=np.float64)
    ht = np.asarray(d["height"], dtype=np.float64)
    if e.shape != (int(d["N"]),) or ht.shape != e.shape:
        raise ValueError("earnings: earn and height must have length N")
    return dict(dim=4, data0=np.array([float(len(e)), e.sum(), ht.sum(), e @ e, e @ ht, ht @ ht]))


def _eight_schools(d):                               # posteriordb eight_schools_{noncentered,centered}
    J, y, sigma = _eight_schools_data(d)
    return dict(dim=J + 2, i0=J, data0=np.concatenate([y, 1.0 / (sigma * sigma)]))


def _logistic_regression(d):                         # y ~ bernoulli_logit(alpha + x * beta)
    N, K, X, y = _logistic_regression_data(d)
    return dict(dim=K + 1, i0=N, i1=K, data0=np.concatenate([X.reshape(-1), y]))


def _arma11(d):                                      # posteriordb arma11, ARMA(1,1)
    T, y = _arma11_data(d)
    return dict(dim=4, i0=T, data0=y)


_TARGETS = {
    "normal": _Target(lambda d: dict(dim=int(d["D"])), _y_names),
    "ill-normal": _Target(_ill_normal, _y_names),
    # stan/funnel.stan:4-7
    "funnel": _Target(lambda d: dict(dim=int(d["D"]) + 1, i0=int(d["D"])),
                      lambda h: ["double_log_sigma"] + [f"alpha.{i + 1}" for i in range(h["i0"])]),
    "corr-normal": _Target(_corr_normal, _y_names),
    "ar1": _Target(_ar1, _y_names),
    # sigma = exp(u), stan/arK.stan:9
    "arK": _Target(_ark, lambda h: ["alpha"] + [f"beta.{i + 1}" for i in range(h["i0"])] + ["sigma"],
                   fp64_data=True, transforms=((-1, "exp"),)),
    # stan/rosenbrock.stan:4-7
    "rosenbrock": _Target(lambda d: dict(dim=2 * int(d["D"]), i0=int(d["D"])),
                          lambda h: ([f"v.{i + 1}" for i in range(h["i0"])] +
                                     [f"theta.{i + 1}" for i in range(h["i0"])])),
    # sigma, s > 0, stan/earnings.stan:9-10
    "earnings": _Target(_earnings, lambda h: ["beta.1", "beta.2", "sigma", "s"],
                        fp64_data=True, transforms=((slice(2, None), "exp"),)),
    # [theta_trans, mu, log tau]
    "eight_schools_noncentered": _Target(
        _eight_schools, lambda h: [f"theta_trans.{j + 1}" for j in range(h["i0"])] + ["mu", "tau"],
        transforms=((-1, "exp"),)),
    # [mu, log tau, theta]
    "eight_schools_centered": _Target(
        _eight_schools, lambda h: ["mu", "tau"] + [f"theta.{j + 1}" for j in range(h["i0"])],
        transforms=((1, "exp"),)),
    "logistic_regression": _Target(_logistic_regression,
                                   lambda h: ["alpha"] + [f"beta.{k + 1}" for k in range(h["i1"])]),
    # [mu, a, b, v]: phi, theta = tanh(a / 2), tanh(b / 2); sigma = exp(v)
    "arma11": _Target(_arma11, lambda h: ["mu", "phi", "theta", "sigma"],
                      transforms=((slice(1, 3), "tanh_half"), (3, "exp"))),
}


class BSModel:
    def __init__(self, stan_file="", data_file="", stepsize=1.0, warn=False, data=None, device=None):
        self._stan_file = stan_file
        self._data_file = data_file
        name = Path(str(stan_file)).stem
        if name not in _lib.MODEL_IDS:
            raise NotImplementedError(
                f"Stan program {name!r} has no device implementation; available: "
                f"{sorted(_lib.MODEL_IDS)} (klhr_b200 has no CPU fallback)")
        if data is None:
            data = json.loads(Path(data_file).read_text()) if str(data_file) else {}
        self.name = name
        self.data = dict(data)
        self.device = torch.device(device) if device is not None else torch.device("cuda", 0)
        self._cache = {}
        self._host = self._prepare_host()

    # ------------------------------------------------------------------ host-side "transformed data"
    def _prepare_host(self):
        h = dict(i0=0, i1=0, s0=0.0, s1=0.0, data0=None, data1=None)
        h.update(_TARGETS[self.name].prepare(self.data))
        return h

    def dim(self):
        return self._host["dim"]

    # ------------------------------------------------------------------ device descriptor
    def descriptor(self, dtype=torch.float64, device=None):
        """``klhr_model_t`` for the C ABI; the device buffers it points to are cached here."""
        device = torch.device(device) if device is not None else self.device
        key = (dtype, str(device))
        if key not in self._cache:
            h = self._host
            buf = None
            if h["data0"] is not None:
                # sufficient statistics (arK, earnings) stay fp64 whatever the arithmetic type (klhr_models.cuh)
                bt = torch.float64 if _TARGETS[self.name].fp64_data else dtype
                buf = torch.as_tensor(h["data0"], dtype=torch.float64).to(device=device, dtype=bt).contiguous()
            buf1 = None
            if h.get("data1") is not None and dtype == torch.float64:
                buf1 = torch.as_tensor(h["data1"], dtype=torch.float64).to(device=device).contiguous()
            desc = _lib.ModelDesc(id=_lib.MODEL_IDS[self.name], dim=h["dim"], i0=h["i0"], i1=h["i1"],
                                  s0=h["s0"], s1=h["s1"],
                                  data0=buf.data_ptr() if buf is not None else None,
                                  data1=buf1.data_ptr() if buf1 is not None else None)
            self._cache[key] = (desc, buf, buf1)
        return self._cache[key][0]

    # ------------------------------------------------------------------ evaluation
    def _eval(self, theta, want_grad):
        lib = _lib.load()
        single = False
        as_numpy = not torch.is_tensor(theta)
        if as_numpy:
            theta = torch.as_tensor(np.asarray(theta, dtype=np.float64))
        if theta.dim() == 1:
            single = True
            theta = theta[None, :]
        if theta.shape[-1] != self.dim():
            raise ValueError(f"theta has {theta.shape[-1]} columns, model has {self.dim()} parameters")
        dtype = theta.dtype if theta.dtype in _DTYPES else torch.float64
        dev = theta.device if theta.is_cuda else self.device
        th = theta.to(device=dev, dtype=dtype).contiguous()
        B = th.shape[0]
        lp = torch.empty(B, dtype=dtype, device=dev)
        grad = torch.empty_like(th) if want_grad else None
        desc = self.descriptor(dtype, dev)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.klhr_model_eval(C.byref(desc), _dtype_code(dtype), th.data_ptr(), lp.data_ptr(),
                                           grad.data_ptr() if want_grad else None, B, stream),
                       "klhr_model_eval")
        if as_numpy:
            lp_h = lp.cpu().numpy()
            g_h = grad.cpu().numpy() if want_grad else None
            if single:
                return (float(lp_h[0]), g_h[0]) if want_grad else float(lp_h[0])
            return (lp_h, g_h) if want_grad else lp_h
        if single:
            return (lp[0], grad[0]) if want_grad else lp[0]
        return (lp, grad) if want_grad else lp

    def log_density(self, theta, **kws):
        return self._eval(theta, False)

    def log_density_gradient(self, theta, **kws):
        return self._eval(theta, True)

    # ------------------------------------------------------------------ transforms / names
    def _transform(self, theta, inverse):
        out = theta.clone() if torch.is_tensor(theta) else np.array(theta, dtype=np.float64)
        xp = torch if torch.is_tensor(out) else np
        for k, kind in _TARGETS[self.name].transforms:
            u = out[..., k]
            if kind == "exp":
                out[..., k] = xp.log(u) if inverse else xp.exp(u)
            else:                                    # "tanh_half"
                out[..., k] = 2.0 * xp.arctanh(u) if inverse else xp.tanh(0.5 * u)
        return out

    def constrain(self, theta):
        return self._transform(theta, inverse=False)

    def unconstrain(self, theta):
        return self._transform(theta, inverse=True)

    def parameter_names(self):
        return _TARGETS[self.name].names(self._host)

    def Hamiltonian(self, theta, rho):               # bsmodel.py:45-46
        return -self.log_density(theta) + 0.5 * (rho * rho).sum(-1)
