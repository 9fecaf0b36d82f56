"""NumPy fp64 restatement of the two eight-schools programs (posteriordb ``eight_schools_noncentered`` and
``eight_schools_centered``), with ``lp_grad`` / ``dir2`` like ``oracle/stan_models.py`` and the O(1) line restriction
the device models are built on.

TEST INFRASTRUCTURE (see oracle/__init__.py).  BridgeStan conventions ``propto=True, jacobian=True``: constants are
dropped and tau is sampled as u = log tau with its log-Jacobian u.  ``make_hier_model`` builds a model from the
program's stem and JSON data; ``HierBSModel`` wraps one with the surface of ``oracle/bsmodel.py`` (``log_density``,
``log_density_gradient``: -inf / zero gradient on failure), which the bit-exact port of the reference
(``oracle/ref_port.py``) evaluates.
"""
from __future__ import annotations

import numpy as np

from .stan_models import StanModelBase


def _softplus(z):
    """log(1 + e^z) without overflow; with the logistic sigma(z) and sigma (1 - sigma)."""
    q = np.exp(-np.abs(z))
    sp = np.maximum(z, 0.0) + np.log1p(q)
    sg = np.where(z >= 0, 1.0 / (1.0 + q), q / (1.0 + q))
    return sp, sg, q / (1.0 + q) ** 2


LOG25 = float(np.log(25.0))
EIGHT_SCHOOLS_DATA = {"J": 8, "y": [28.0, 8.0, -3.0, 7.0, -1.0, 1.0, 18.0, 12.0],
                      "sigma": [15.0, 10.0, 16.0, 11.0, 9.0, 11.0, 10.0, 18.0]}


class _EightSchools(StanModelBase):
    def __init__(self, J, y, sigma):
        self.J = int(J)
        self.y = np.asarray(y, dtype=np.float64)
        self.sigma = np.asarray(sigma, dtype=np.float64)
        assert self.J >= 1 and self.y.shape == (self.J,) and self.sigma.shape == (self.J,)
        self.w = 1.0 / (self.sigma * self.sigma)

    def dim(self):
        return self.J + 2


class EightSchoolsNC(_EightSchools):
    """posteriordb eight_schools_noncentered: theta = theta_trans * tau + mu; theta_trans ~ normal(0, 1);
    y ~ normal(theta, sigma); mu ~ normal(0, 5); tau ~ cauchy(0, 5).

    Unconstrained [tt_1..tt_J, mu, u = log tau]:
    lp = -1/2 sum tt^2 - 1/2 sum w (y - mu - e^u tt)^2 - mu^2/50 - log1p(e^{2u}/25) + u,  w = 1/sigma^2,
    the Cauchy term as softplus(2u - log 25)."""
    name = "eight_schools_noncentered"

    def lp_grad(self, theta):
        theta = np.asarray(theta, dtype=np.float64)
        tt, mu, u = theta[..., :self.J], theta[..., self.J], theta[..., self.J + 1]
        with np.errstate(all="ignore"):
            E = np.exp(u)
            res = self.y - mu[..., None] - E[..., None] * tt
            sp, sg, _ = _softplus(2.0 * u - LOG25)
            lp = (-0.5 * np.sum(tt * tt, axis=-1) - 0.5 * np.sum(self.w * res * res, axis=-1) - mu * mu / 50.0
                  - sp + u)
            g = np.empty_like(theta)
            g[..., :self.J] = -tt + E[..., None] * self.w * res
            g[..., self.J] = np.sum(self.w * res, axis=-1) - mu / 25.0
            g[..., self.J + 1] = E * np.sum(self.w * res * tt, axis=-1) - 2.0 * sg + 1.0
        return lp, g

    def dir2(self, theta, rho):
        theta, rho = np.asarray(theta, dtype=np.float64), np.asarray(rho, dtype=np.float64)
        J = self.J
        tt, mu, u = theta[..., :J], theta[..., J], theta[..., J + 1]
        rt, rm, ru = rho[..., :J], rho[..., J], rho[..., J + 1]
        with np.errstate(all="ignore"):
            E = np.exp(u)[..., None]
            # residual e(y) = y - mu - e^u tt along the line: e' = -rm - E (ru tt + rt), e'' = -E (ru^2 tt + 2 ru rt)
            res = self.y - mu[..., None] - E * tt
            e1 = -rm[..., None] - E * (ru[..., None] * tt + rt)
            e2 = -E * (ru[..., None] ** 2 * tt + 2.0 * ru[..., None] * rt)
            _, _, sg1 = _softplus(2.0 * u - LOG25)
            return (-np.sum(rt * rt, axis=-1) - np.sum(self.w * (e1 * e1 + res * e2), axis=-1) - rm * rm / 25.0
                    - 4.0 * ru * ru * sg1)

    def line_sums(self, theta, rho):
        """The 13 sums of the O(1) line restriction (klhr_models.cuh EightSchoolsNC)."""
        J = self.J
        a, m0, r, rm = theta[..., :J], theta[..., J], rho[..., :J], rho[..., J]
        c = self.y - m0[..., None]
        W = lambda f: np.sum(self.w * f, axis=-1)
        return dict(W1=W(np.ones_like(c)), Wc=W(c), Wc2=W(c * c), Wa=W(a), Wr=W(r), Wca=W(c * a), Wcr=W(c * r),
                    Wa2=W(a * a), War=W(a * r), Wr2=W(r * r), a2=np.sum(a * a, -1), ar=np.sum(a * r, -1),
                    r2=np.sum(r * r, -1))

    def line_from_sums(self, theta, rho, t):
        """l(t) = lp(theta + t rho) from the 13 sums, the Cauchy term as a softplus."""
        S = self.line_sums(theta, rho)
        J = self.J
        m0, rm, u0, ru = theta[..., J], rho[..., J], theta[..., J + 1], rho[..., J + 1]
        mu, u = m0 + t * rm, u0 + t * ru
        with np.errstate(all="ignore"):
            E = np.exp(u)
            Pd = S["Wc2"] - 2 * t * rm * S["Wc"] + t * t * rm * rm * S["W1"]
            Qd = S["Wca"] + t * (S["Wcr"] - rm * S["Wa"]) - t * t * rm * S["Wr"]
            Sd = S["Wa2"] + 2 * t * S["War"] + t * t * S["Wr2"]
            N = S["a2"] + 2 * t * S["ar"] + t * t * S["r2"]
            return -0.5 * N - 0.5 * (Pd - 2 * E * Qd + E * E * Sd) - mu * mu / 50.0 - _softplus(2 * u - LOG25)[0] + u


class EightSchoolsC(_EightSchools):
    """posteriordb eight_schools_centered: mu ~ normal(0, 5); tau ~ cauchy(0, 5); theta ~ normal(mu, tau);
    y ~ normal(theta, sigma).

    Unconstrained [mu, u = log tau, theta_1..theta_J]:
    lp = -mu^2/50 - log1p(e^{2u}/25) + (1 - J) u - 1/2 e^{-2u} sum (theta - mu)^2 - 1/2 sum w (y - theta)^2."""
    name = "eight_schools_centered"

    def lp_grad(self, theta):
        theta = np.asarray(theta, dtype=np.float64)
        mu, u, th = theta[..., 0], theta[..., 1], theta[..., 2:]
        with np.errstate(all="ignore"):
            em2 = np.exp(-2.0 * u)
            d = th - mu[..., None]
            e = self.y - th
            sd2 = np.sum(d * d, axis=-1)
            sp, sg, _ = _softplus(2.0 * u - LOG25)
            lp = (-mu * mu / 50.0 - sp + (1 - self.J) * u - 0.5 * em2 * sd2
                  - 0.5 * np.sum(self.w * e * e, axis=-1))
            g = np.empty_like(theta)
            g[..., 0] = -mu / 25.0 + em2 * np.sum(d, axis=-1)
            g[..., 1] = -2.0 * sg + (1 - self.J) + em2 * sd2
            g[..., 2:] = -em2[..., None] * d + self.w * e
        return lp, g

    def dir2(self, theta, rho):
        theta, rho = np.asarray(theta, dtype=np.float64), np.asarray(rho, dtype=np.float64)
        mu, u, th = theta[..., 0], theta[..., 1], theta[..., 2:]
        rm, ru, rt = rho[..., 0], rho[..., 1], rho[..., 2:]
        with np.errstate(all="ignore"):
            em2 = np.exp(-2.0 * u)
            d = th - mu[..., None]
            dr = rt - rm[..., None]
            A, A1, A2 = np.sum(d * d, -1), 2.0 * np.sum(d * dr, -1), 2.0 * np.sum(dr * dr, -1)
            _, _, sg1 = _softplus(2.0 * u - LOG25)
            return (-rm * rm / 25.0 - 4.0 * ru * ru * sg1 - 0.5 * em2 * (4.0 * ru * ru * A - 4.0 * ru * A1 + A2)
                    - np.sum(self.w * rt * rt, axis=-1))

    def line_sums(self, theta, rho):
        """The 6 sums of the O(1) line restriction (klhr_models.cuh EightSchoolsC)."""
        a, m0, r, rm = theta[..., 2:], theta[..., 0], rho[..., 2:], rho[..., 0]
        dm, dr, e = a - m0[..., None], r - rm[..., None], self.y - a
        return dict(A0=np.sum(dm * dm, -1), A1=np.sum(dm * dr, -1), A2=np.sum(dr * dr, -1),
                    B0=np.sum(self.w * e * e, -1), B1=np.sum(self.w * e * r, -1), B2=np.sum(self.w * r * r, -1))

    def line_from_sums(self, theta, rho, t):
        """l(t) = lp(theta + t rho) from the 6 sums, the Cauchy term as a softplus."""
        S = self.line_sums(theta, rho)
        mu, u = theta[..., 0] + t * rho[..., 0], theta[..., 1] + t * rho[..., 1]
        with np.errstate(all="ignore"):
            A = S["A0"] + 2 * t * S["A1"] + t * t * S["A2"]
            B = S["B0"] - 2 * t * S["B1"] + t * t * S["B2"]
            return (-mu * mu / 50.0 - _softplus(2 * u - LOG25)[0] + (1 - self.J) * u - 0.5 * np.exp(-2.0 * u) * A
                    - 0.5 * B)


HIER_MODEL_NAMES = ("eight_schools_noncentered", "eight_schools_centered")


def make_hier_model(name: str, data: dict) -> StanModelBase:
    """Build an eight-schools model from the Stan program's stem and its JSON data dict."""
    if name == "eight_schools_noncentered":
        return EightSchoolsNC(data["J"], data["y"], data["sigma"])
    if name == "eight_schools_centered":
        return EightSchoolsC(data["J"], data["y"], data["sigma"])
    raise ValueError(f"unknown hierarchical model {name!r}; known: {HIER_MODEL_NAMES}")


class HierBSModel:
    """``oracle/bsmodel.py:BSModel`` surface for the eight-schools models."""

    def __init__(self, name: str, data: dict):
        self.name = name
        self.model = make_hier_model(name, data)

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
