"""NumPy fp64 restatement of ARMA(1,1) (posteriordb ``arma11``, the Stan User's Guide ARMA(1,1)), with ``lp_grad`` /
``dir2`` like ``oracle/stan_models.py`` and the line restriction the device model evaluates, plus a seeded simulator
and the named data sets the tests and the bench use.

TEST INFRASTRUCTURE (see oracle/__init__.py).  BridgeStan conventions ``propto=True, jacobian=True``.  Unconstrained
[mu, a, b, v] with phi = tanh(a / 2), theta = tanh(b / 2), sigma = e^v:

    lp = -mu^2/200 - phi^2/8 - theta^2/8 - softplus(2v - log 25) + (1 - T) v - e^{-2v} sum_t err_t^2 / 2 + J(a) + J(b)
    err_1 = y_1 - mu (1 + phi),  err_t = y_t - mu - phi y_{t-1} - theta err_{t-1},
    J(u) = log 2 - |u| - 2 log1p(e^-|u|)   (log d phi / du, finite for every finite u).

``TSBSModel`` wraps the model with the surface of ``oracle/bsmodel.py`` (``log_density``, ``log_density_gradient``:
-inf / zero gradient on failure), which the bit-exact port of the reference (``oracle/ref_port.py``) evaluates.
"""
from __future__ import annotations

import numpy as np

from .hier_models import LOG25, _softplus
from .stan_models import StanModelBase

LN2 = float(np.log(2.0))


def bounded(u):
    """(phi, q, J) of phi = tanh(u / 2): q = d phi / du = (1 - phi^2) / 2 and J = log q, all from e^-|u|."""
    with np.errstate(all="ignore"):
        e = np.exp(-np.abs(u))
        p = (1.0 - e) / (1.0 + e)
        return np.where(u < 0, -p, p), 2.0 * e / (1.0 + e) ** 2, LN2 - np.abs(u) - 2.0 * np.log1p(e)


class Arma11(StanModelBase):
    """posteriordb arma11: mu ~ normal(0, 10); phi, theta ~ normal(0, 2) on (-1, 1); sigma ~ cauchy(0, 5) on
    (0, inf); err ~ normal(0, sigma).  Unconstrained [mu, a, b, v]."""
    name = "arma11"

    def __init__(self, y):
        self.y = np.asarray(y, dtype=np.float64)
        assert self.y.ndim == 1 and len(self.y) >= 1
        self.T = len(self.y)

    def dim(self):
        return 4

    def _rest(self, mu, v, A, B):
        """Every term of lp but the likelihood sum, and the softplus of the Cauchy term."""
        sp = _softplus(2.0 * v - LOG25)
        return -mu * mu / 200.0 - (A[0] ** 2 + B[0] ** 2) / 8.0 - sp[0] + (1 - self.T) * v + A[2] + B[2], sp

    def lp_grad(self, theta):
        """lp and its gradient from forward-mode tangents of err_t in mu, a and b (three extra recurrences)."""
        theta = np.asarray(theta, dtype=np.float64)
        mu, a, b, v = (theta[..., k] for k in range(4))
        y = self.y
        with np.errstate(all="ignore"):
            A, B = bounded(a), bounded(b)
            ph, th = A[0], B[0]
            e = y[0] - mu * (1.0 + ph)
            gm, ga, gb = -(1.0 + ph), -mu * A[1], np.zeros_like(e)
            E0, Sm, Sa, Sb = e * e, e * gm, e * ga, np.zeros_like(e)
            for t in range(1, self.T):
                n = (y[t] - mu) - ph * y[t - 1] - th * e
                gb = -B[1] * e - th * gb
                gm = -1.0 - th * gm
                ga = -A[1] * y[t - 1] - th * ga
                e = n
                E0, Sm, Sa, Sb = E0 + e * e, Sm + e * gm, Sa + e * ga, Sb + e * gb
            em2 = np.exp(-2.0 * v)
            rest, sp = self._rest(mu, v, A, B)
            lp = rest - 0.5 * em2 * E0
            g = np.empty_like(theta)
            g[..., 0] = -mu / 100.0 - em2 * Sm
            g[..., 1] = -ph * A[1] / 4.0 - ph - em2 * Sa
            g[..., 2] = -th * B[1] / 4.0 - th - em2 * Sb
            g[..., 3] = -2.0 * sp[1] + (1 - self.T) + em2 * E0
        return lp, g

    def jet(self, theta, rho, t):
        """(l(t), l'(t), l''(t)) of l(t) = lp(theta + t rho), not differenced: the recursion carrying err_t and its
        first two t-derivatives, as the device model forms it (klhr_models.cuh Arma11)."""
        theta, rho = np.asarray(theta, dtype=np.float64), np.asarray(rho, dtype=np.float64)
        t = np.asarray(t, dtype=np.float64)
        (m0, a0, b0, v0), (rm, ra, rb, rv) = (theta[..., k] for k in range(4)), (rho[..., k] for k in range(4))
        y = self.y
        with np.errstate(all="ignore"):
            mu, v = m0 + t * rm, v0 + t * rv
            A, B = bounded(a0 + t * ra), bounded(b0 + t * rb)
            ph, ph1, ph2 = A[0], ra * A[1], -ra * ra * A[0] * A[1]
            th, th1, th2 = B[0], rb * B[1], -rb * rb * B[0] * B[1]
            e = y[0] - mu * (1.0 + ph)
            e1 = -rm * (1.0 + ph) - mu * ph1
            e2 = -2.0 * rm * ph1 - mu * ph2
            E0, E1, E2 = e * e, e * e1, e1 * e1 + e * e2
            for k in range(1, self.T):
                n = (y[k] - mu) - ph * y[k - 1] - th * e
                n1 = -rm - ph1 * y[k - 1] - th1 * e - th * e1
                n2 = -ph2 * y[k - 1] - th2 * e - 2.0 * th1 * e1 - th * e2
                e, e1, e2 = n, n1, n2
                E0, E1, E2 = E0 + e * e, E1 + e * e1, E2 + e1 * e1 + e * e2
            em2 = np.exp(-2.0 * v)
            rest, sp = self._rest(mu, v, A, B)
            l = rest - 0.5 * em2 * E0
            l1 = (-mu * rm / 100.0 - (ph * ph1 + th * th1) / 4.0 - 2.0 * rv * sp[1] + (1 - self.T) * rv
                  - em2 * (E1 - rv * E0) - ra * ph - rb * th)
            l2 = (-rm * rm / 100.0 - (ph1 * ph1 + ph * ph2 + th1 * th1 + th * th2) / 4.0 - 4.0 * rv * rv * sp[2]
                  - em2 * (2.0 * rv * rv * E0 - 4.0 * rv * E1 + E2) - ra * ra * A[1] - rb * rb * B[1])
        return l, l1, l2

    def dir2(self, theta, rho):
        return self.jet(theta, rho, np.zeros(np.shape(theta)[:-1]))[2]

    def line(self, theta, rho, t):
        """(l(t) - l(0), l'(t), l''(t)) along theta + t rho (vectorised over chains)."""
        l, l1, l2 = self.jet(theta, rho, t)
        return l - self.jet(theta, rho, np.zeros_like(np.asarray(t, dtype=np.float64)))[0], l1, l2

    def error_scales(self, theta):
        """(lp scale, gradient scales (..., 4)) that bound the rounding error of lp and its gradient: in a precision
        with unit roundoff u, |error| <= (T + 18) u x scale.

        With a_t = |y_t| + |mu| + |phi y_{t-1}| + |theta| a_{t-1} (a bound on |err_t| and on every partial sum of
        the step that forms it) the rounding error of err_t obeys d_t <= 8 u a_t + |theta| d_{t-1}, so
        d_t <= 8 u b_t with b_t = a_t + |theta| b_{t-1}.  The error of e^{-2v} sum err^2 / 2 is then at most
        e^{-2v} (16 u sum a_t b_t + (T + 2) u sum a_t^2) / 2 <= (T + 18) u e^{-2v} sum a_t b_t / 2; each of the other
        terms is formed to a few ulp of its magnitude.  The tangents get the same treatment with their own magnitude
        recursions (the one of b driven by b_{t-1}, which bounds err_{t-1} with its error), and every product
        err_t g_t by b_t times the tangent's accumulated magnitude."""
        theta = np.asarray(theta, dtype=np.float64)
        mu, a, b, v = (theta[..., k] for k in range(4))
        y = np.abs(self.y)
        with np.errstate(all="ignore"):
            A, B = bounded(a), bounded(b)
            ap, tp, am = np.abs(A[0]), np.abs(B[0]), np.abs(mu)
            at = y[0] + am * (1.0 + ap)
            bt = at
            tm, ta, tb = 1.0 + ap, am * A[1], np.zeros_like(at)          # tangent magnitudes ...
            um, ua, ub = tm, ta, tb                                          # ... and their accumulations
            Sab, Sm, Sa, Sb = at * bt, bt * um, bt * ua, np.zeros_like(at)
            for t in range(1, self.T):
                tb = B[1] * bt + tp * tb
                tm = 1.0 + tp * tm
                ta = A[1] * y[t - 1] + tp * ta
                at = y[t] + am + ap * y[t - 1] + tp * at
                bt = at + tp * bt
                um, ua, ub = tm + tp * um, ta + tp * ua, tb + tp * ub
                Sab, Sm, Sa, Sb = Sab + at * bt, Sm + bt * um, Sa + bt * ua, Sb + bt * ub
            em2 = np.exp(-2.0 * v)
            sp = _softplus(2.0 * v - LOG25)[0]
            lp = (mu * mu / 200.0 + (A[0] ** 2 + B[0] ** 2) / 8.0 + np.abs(sp) + np.abs((1 - self.T) * v)
                  + 0.5 * em2 * Sab + np.abs(A[2]) + np.abs(B[2]))
            g = np.empty_like(theta)
            g[..., 0] = am / 100.0 + em2 * Sm
            g[..., 1] = ap * A[1] / 4.0 + ap + em2 * Sa
            g[..., 2] = tp * B[1] / 4.0 + tp + em2 * Sb
            g[..., 3] = 2.0 + abs(1 - self.T) + em2 * Sab
        return lp, g

    def terms_scale(self, theta):
        """The magnitude of what lp sums, as ``error_scales`` bounds it."""
        return self.error_scales(theta)[0]


def simulate(T, mu, phi, theta, sigma, seed):
    """Data dict {T, y} of y_t = mu + phi (y_{t-1} - mu) + theta e_{t-1} + e_t, e_t ~ normal(0, sigma), started from
    y_0 := mu, e_0 := 0 (seeded)."""
    rng = np.random.default_rng(seed)
    e = rng.normal(size=T) * sigma
    y = np.empty(T)
    yp, ep = mu, 0.0
    for t in range(T):
        y[t] = mu + phi * (yp - mu) + theta * ep + e[t]
        yp, ep = y[t], e[t]
    return {"T": T, "y": y.tolist()}


# T = 200 from mu = 1, phi = 0.6, theta = 0.3, sigma = 1: a posterior close to a Gaussian
MODERATE = simulate(200, 1.0, 0.6, 0.3, 1.0, seed=201)
# T = 100 of white noise: the AR and MA roots cancel along phi ~ -theta, a ridge in (a, b) held in by the priors
RIDGE = simulate(100, 0.0, 0.0, 0.0, 1.0, seed=202)
# T = 1: theta does not enter the likelihood, so its posterior is exactly its prior
SINGLE = {"T": 1, "y": [0.7]}
# T = 10 000 (the bench's largest series and one replay case)
LONG = simulate(10_000, 1.0, 0.6, 0.3, 1.0, seed=203)


def make_ts_model(name: str, data: dict) -> StanModelBase:
    if name != "arma11":
        raise ValueError(f"unknown time-series model {name!r}; known: ('arma11',)")
    assert int(data["T"]) == len(data["y"])
    return Arma11(data["y"])


class TSBSModel:
    """``oracle/bsmodel.py:BSModel`` surface for ARMA(1,1)."""

    def __init__(self, name: str, data: dict):
        self.name = name
        self.model = make_ts_model(name, data)

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
