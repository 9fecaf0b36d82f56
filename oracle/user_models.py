"""NumPy fp64 restatements of the user-written targets of ``tests/user_targets`` that have no built-in counterpart:
``trio`` (with its exact moments) and the AD ``probe`` (each primitive with its analytic first and second
derivative).  The restatements of built-in targets there are checked against the existing oracles (hier, glm, ts).

TEST INFRASTRUCTURE (see oracle/__init__.py).

trio: K Student-t(nu) coordinates t_k with scales s_k, u = log sigma with sigma ~ Gamma(a, b), z = logit p with
p ~ Beta(alpha, beta), on the unconstrained scale with the Jacobians:

    lp = sum_k -(nu + 1)/2 log1p((t_k / s_k)^2 / nu) + a u - b e^u + alpha log sigma(z) + beta log sigma(-z).

u and z are exactly log-Gamma and logit-Beta variates: E[u] = psi(a) - log b, Var u = psi'(a), E[z] = psi(alpha) -
psi(beta), Var z = psi'(alpha) + psi'(beta); Var t_k = s_k^2 nu / (nu - 2) (nu > 2).
"""
from __future__ import annotations

import numpy as np
from scipy.special import digamma, expit, polygamma

from .stan_models import StanModelBase


def _log_sigmoid(z):
    """log sigma(z) = -softplus(-z) = -(max(-z, 0) + log1p(e^-|z|))."""
    return -(np.maximum(-z, 0.0) + np.log1p(np.exp(-np.abs(z))))


class Trio(StanModelBase):
    name = "trio"

    def __init__(self, nu, s, a, b, alpha, beta):
        self.nu, self.s = float(nu), np.asarray(s, dtype=np.float64).reshape(-1)
        self.a, self.b, self.alpha, self.beta = float(a), float(b), float(alpha), float(beta)
        self.K = len(self.s)

    @classmethod
    def from_data(cls, d):
        return cls(d["nu"], d["s"], d["a"], d["b"], d["alpha"], d["beta"])

    def dim(self):
        return self.K + 2

    def lp_grad(self, theta):
        theta = np.asarray(theta, dtype=np.float64)
        K, nu = self.K, self.nu
        t, u, z = theta[..., :K], theta[..., K], theta[..., K + 1]
        with np.errstate(all="ignore"):
            r = t / self.s
            eu = np.exp(u)
            lp = (-0.5 * (nu + 1) * np.log1p(r * r / nu)).sum(-1) + self.a * u - self.b * eu \
                + self.alpha * _log_sigmoid(z) + self.beta * _log_sigmoid(-z)
            g = np.empty_like(theta)
            g[..., :K] = -(nu + 1) * r / (self.s * (nu + r * r))
            g[..., K] = self.a - self.b * eu
            g[..., K + 1] = self.alpha * expit(-z) - self.beta * expit(z)
        return lp, g

    def dir2(self, theta, rho):
        theta = np.asarray(theta, dtype=np.float64)
        K, nu = self.K, self.nu
        t, u, z = theta[..., :K], theta[..., K], theta[..., K + 1]
        with np.errstate(all="ignore"):
            r = t / self.s
            htt = -(nu + 1) / self.s ** 2 * (nu - r * r) / (nu + r * r) ** 2
            hu = -self.b * np.exp(u)
            hz = -(self.alpha + self.beta) * expit(z) * expit(-z)
            return (htt * rho[..., :K] ** 2).sum(-1) + hu * rho[..., K] ** 2 + hz * rho[..., K + 1] ** 2

    def moments(self):
        """Exact posterior mean and variance of every unconstrained coordinate."""
        mean = np.concatenate([np.zeros(self.K), [digamma(self.a) - np.log(self.b), digamma(self.alpha) - digamma(self.beta)]])
        var = np.concatenate([self.s ** 2 * self.nu / (self.nu - 2),
                              [polygamma(1, self.a), polygamma(1, self.alpha) + polygamma(1, self.beta)]])
        return mean, var


class UserBSModel:
    """``oracle/bsmodel.py:BSModel`` surface for a model above (-inf / zero gradient on failure)."""

    def __init__(self, model: StanModelBase):
        self.model = model

    def dim(self):
        return self.model.dim()

    def log_density(self, theta, **kws):
        ld = float(self.model.lp(np.asarray(theta, dtype=np.float64)))
        return ld if np.isfinite(ld) else -np.inf

    def log_density_gradient(self, theta, **kws):
        theta = np.asarray(theta, dtype=np.float64)
        ld, g = self.model.lp_grad(theta)
        if not (np.isfinite(ld) and np.all(np.isfinite(g))):
            return -np.inf, np.zeros_like(theta)
        return float(ld), g


# ------------------------------------------------------------------ probe: one primitive per coordinate
def _tanh_jet(x):
    e = np.exp(-2.0 * np.abs(x))
    t = np.sign(x) * (1.0 - e) / (1.0 + e)
    q = 4.0 * e / (1.0 + e) ** 2
    return t, q, -2.0 * t * q


def _softplus_jet(x):
    e = np.exp(-np.abs(x))
    sg = np.where(x >= 0, 1.0 / (1.0 + e), e / (1.0 + e))
    return np.maximum(x, 0.0) + np.log1p(e), sg, e / (1.0 + e) ** 2


def _log_inv_logit_jet(x):
    sp, sg, sg1 = _softplus_jet(-x)
    return -sp, sg, -sg1


# (name, f, f', f'') of coordinate k of tests/user_targets/probe.cuh, in its order
PROBE = [
    ("exp", lambda x: (np.exp(x), np.exp(x), np.exp(x))),
    ("log", lambda x: (np.log(x), 1.0 / x, -1.0 / x ** 2)),
    ("log1p", lambda x: (np.log1p(x), 1.0 / (1.0 + x), -1.0 / (1.0 + x) ** 2)),
    ("expm1", lambda x: (np.expm1(x), np.exp(x), np.exp(x))),
    ("sqrt", lambda x: (np.sqrt(x), 0.5 / np.sqrt(x), -0.25 / (x * np.sqrt(x)))),
    ("square", lambda x: (x * x, 2.0 * x, np.full_like(x, 2.0))),
    ("pow2.5", lambda x: (x ** 2.5, 2.5 * x ** 1.5, 3.75 * x ** 0.5)),
    ("tanh", _tanh_jet),
    ("log1p_exp", _softplus_jet),
    ("log_inv_logit", _log_inv_logit_jet),
    ("fabs", lambda x: (np.abs(x), np.sign(x), np.zeros_like(x))),
    ("reciprocal", lambda x: (1.0 / x, -1.0 / x ** 2, 2.0 / x ** 3)),
]
PROBE_DIM = len(PROBE)
# a point where every primitive is finite (the t = 0 end of each probed line)
PROBE_BASE = np.array([0.0, 1.0, 0.0, 0.0, 1.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0, 1.0])


def probe_jet(k, x):
    """(f_k, f_k', f_k'') of primitive k at the points x (fp64, analytic)."""
    with np.errstate(all="ignore"):
        return tuple(np.asarray(v, dtype=np.float64) for v in PROBE[k][1](np.asarray(x, dtype=np.float64)))
