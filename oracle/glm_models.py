"""NumPy fp64 restatement of Bayesian logistic regression, with ``lp_grad`` / ``dir2`` like ``oracle/stan_models.py``
and the line restriction the device model evaluates, plus the named synthetic data sets the tests and the bench use.

TEST INFRASTRUCTURE (see oracle/__init__.py).  BridgeStan conventions ``propto=True``: with X = [1 | x] and
theta = [alpha, beta_1..K],

    lp(theta) = -|theta|^2 / 12.5 + sum_i (y_i eta_i - softplus(eta_i)),   eta = X theta,

softplus formed as max(z, 0) + log1p(e^-|z|), finite for every finite z.  ``GLMBSModel`` wraps the model with the
surface of ``oracle/bsmodel.py`` (``log_density``, ``log_density_gradient``: -inf / zero gradient on failure), which
the bit-exact port of the reference (``oracle/ref_port.py``) evaluates.  The data sets are generated from fixed seeds.
"""
from __future__ import annotations

import numpy as np

from .hier_models import _softplus
from .stan_models import StanModelBase

PRIOR_VAR = 6.25                       # alpha, beta ~ normal(0, 2.5)


class LogisticRegression(StanModelBase):
    """y ~ bernoulli_logit(alpha + x * beta); alpha, beta ~ normal(0, 2.5).  Unconstrained [alpha, beta_1..K]."""
    name = "logistic_regression"

    def __init__(self, x, y):
        self.x = np.asarray(x, dtype=np.float64)          # (N, K)
        self.y = np.asarray(y, dtype=np.float64)
        self.N, self.K = self.x.shape
        assert self.K >= 1 and self.y.shape == (self.N,)
        self.X = np.concatenate([np.ones((self.N, 1)), self.x], axis=1)

    def dim(self):
        return self.K + 1

    def lp_grad(self, theta):
        theta = np.asarray(theta, dtype=np.float64)
        with np.errstate(all="ignore"):
            eta = theta @ self.X.T
            sp, sg, _ = _softplus(eta)
            lp = -np.sum(theta * theta, axis=-1) / (2 * PRIOR_VAR) + np.sum(self.y * eta - sp, axis=-1)
            g = -theta / PRIOR_VAR + (self.y - sg) @ self.X
        return lp, g

    def dir2(self, theta, rho):
        theta, rho = np.asarray(theta, dtype=np.float64), np.asarray(rho, dtype=np.float64)
        with np.errstate(all="ignore"):
            eta = theta @ self.X.T
            b = rho @ self.X.T
            _, _, sg1 = _softplus(eta)
            return -np.sum(b * b * sg1, axis=-1) - np.sum(rho * rho, axis=-1) / PRIOR_VAR

    def terms_scale(self, theta):
        """sum_i |y_i eta_i - softplus(eta_i)| + |theta|^2 / 12.5: the magnitude of what lp sums."""
        theta = np.asarray(theta, dtype=np.float64)
        eta = theta @ self.X.T
        return np.sum(np.abs(self.y * eta - _softplus(eta)[0]), axis=-1) + np.sum(theta * theta, -1) / (2 * PRIOR_VAR)

    def line(self, theta, rho, t):
        """(l(t) - l(0), l'(t), l''(t)) along theta + t rho from a = X theta and b = X rho, as the device model forms
        them (klhr_models.cuh LogisticRegression)."""
        t = np.asarray(t, dtype=np.float64)
        a, b = theta @ self.X.T, rho @ self.X.T
        tr, rr = np.sum(theta * rho, -1), np.sum(rho * rho, -1)
        eta = a + t[..., None] * b
        sp, sg, sg1 = _softplus(eta)
        l0 = np.sum(self.y * a - _softplus(a)[0], -1)
        l = np.sum(self.y * eta - sp, -1) - l0 - t * (2 * tr + t * rr) / (2 * PRIOR_VAR)
        l1 = np.sum(b * (self.y - sg), -1) - (tr + t * rr) / PRIOR_VAR
        l2 = -np.sum(b * b * sg1, -1) - rr / PRIOR_VAR
        return l, l1, l2


def synthetic(N, K, seed, corr=0.0, alpha=0.0, beta=None, scale=1.0, separated=False):
    """Data dict {N, K, x, y}: rows of x ~ N(0, scale^2 C) with C_jk = corr^|j-k|, y ~ bernoulli_logit(alpha + x beta).
    ``separated``: y = 1 exactly where x beta > 0, so no finite maximum-likelihood estimate exists."""
    rng = np.random.default_rng(seed)
    idx = np.arange(K)
    L = np.linalg.cholesky(corr ** np.abs(idx[:, None] - idx[None, :]))
    x = scale * rng.normal(size=(N, K)) @ L.T
    beta = np.ones(K) if beta is None else np.asarray(beta, dtype=np.float64)
    eta = alpha + x @ beta
    if separated:
        y = (x @ beta > 0).astype(int)
    else:
        y = (rng.random(N) < 1.0 / (1.0 + np.exp(-eta))).astype(int)
    return {"N": N, "K": K, "x": x.tolist(), "y": y.tolist()}


# N = 200, K = 2, covariates correlated 0.6: a posterior close to a Gaussian, D = 3
MODERATE = synthetic(200, 2, seed=101, corr=0.6, alpha=0.3, beta=[1.0, -0.5])
# N = 40, K = 1, separated: the likelihood keeps rising along beta -> +inf; the posterior of beta is strongly skewed and
# held in by the prior alone, D = 2
SEPARATED = synthetic(40, 1, seed=102, beta=[1.0], separated=True)
# N = 1000, K = 24 (D = 25): beyond the chain kernel's thread-per-chain D-phase
WIDE = synthetic(1000, 24, seed=103, scale=0.3, beta=np.random.default_rng(104).normal(size=24) * 0.5)
EMPTY = {"N": 0, "K": 2, "x": [], "y": []}                # N = 0: the posterior is the prior N(0, 6.25 I)


def make_glm_model(name: str, data: dict) -> StanModelBase:
    if name != "logistic_regression":
        raise ValueError(f"unknown GLM {name!r}; known: ('logistic_regression',)")
    K = int(data["K"])
    x = np.asarray(data["x"], dtype=np.float64).reshape(int(data["N"]), K)
    return LogisticRegression(x, data["y"])


class GLMBSModel:
    """``oracle/bsmodel.py:BSModel`` surface for logistic regression."""

    def __init__(self, name: str, data: dict):
        self.name = name
        self.model = make_glm_model(name, data)

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
