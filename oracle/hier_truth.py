"""Exact posterior moments of the hierarchical normal model (eight schools), both parametrisations.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Model: y_j ~ normal(theta_j, sigma_j), theta_j ~ normal(mu, tau),
mu ~ normal(0, 5), tau ~ cauchy(0, 5) on tau > 0; u = log tau.  Everything but u integrates in closed form:

    mu | tau, y        ~ normal(m_tau, v_tau),  1 / v_tau = 1/25 + sum_j 1 / (sigma_j^2 + tau^2),
                                                m_tau = v_tau sum_j y_j / (sigma_j^2 + tau^2);
    p(u | y)           ∝ tau / (1 + tau^2 / 25) * sqrt(v_tau) * exp(m_tau^2 / (2 v_tau))
                         * prod_j (sigma_j^2 + tau^2)^(-1/2) * exp(-1/2 sum_j y_j^2 / (sigma_j^2 + tau^2));
    theta_j | mu, tau  ~ normal((1 - lam_j) y_j + lam_j mu, sigma_j^2 tau^2 / (sigma_j^2 + tau^2)),
                         lam_j = sigma_j^2 / (sigma_j^2 + tau^2);
    theta_trans_j = (theta_j - mu) / tau | mu, tau ~ normal(tau (y_j - mu) / (sigma_j^2 + tau^2), lam_j).

So E and Var of every unconstrained coordinate are 1-D integrals over u of conditional moments, done here with the
trapezoidal rule on a uniform grid over the range where log p(u | y) is within ``drop`` of its maximum (the
integrands are smooth and decay exponentially at both ends, where the rule converges geometrically).
"""
from __future__ import annotations

import numpy as np


def _conditionals(u, y, s2):
    """log p(u | y) (unnormalised) and the conditional moments given u = log tau, all shaped (n,) or (n, J)."""
    tau2 = np.exp(2.0 * u)[:, None]
    V = s2[None, :] + tau2                               # sigma^2 + tau^2
    prec = 1.0 / 25.0 + np.sum(1.0 / V, axis=1)
    v = 1.0 / prec
    b = np.sum(y / V, axis=1)
    m = v * b
    logp = (u - np.log1p(tau2[:, 0] / 25.0) + 0.5 * np.log(v) + 0.5 * v * b * b
            - 0.5 * np.sum(np.log(V), axis=1) - 0.5 * np.sum(y * y / V, axis=1))
    lam = s2[None, :] / V
    tau = np.exp(u)[:, None]
    # centered theta_j: E = (1 - lam) y + lam m ; Var = s2 tau2 / V + lam^2 v
    e_th = (1.0 - lam) * y + lam * m[:, None]
    v_th = s2 * tau2 / V + lam * lam * v[:, None]
    # non-centered theta_trans_j: E = tau (y - m) / V ; Var = lam + tau^2 v / V^2
    e_tt = tau * (y - m[:, None]) / V
    v_tt = lam + tau2 * v[:, None] / (V * V)
    return logp, m, v, e_th, v_th, e_tt, v_tt


def _grid(y, s2, n, drop):
    lo, hi = -120.0, 120.0
    coarse = np.linspace(lo, hi, 24001)
    lp = _conditionals(coarse, y, s2)[0]
    keep = coarse[lp > lp.max() - drop]
    h = coarse[1] - coarse[0]
    return np.linspace(keep[0] - 2 * h, keep[-1] + 2 * h, n)


def posterior_moments(y, sigma, n=20001, drop=80.0):
    """Exact posterior means and variances of the unconstrained coordinates.

    Returns dict(noncentered=(mean, var), centered=(mean, var)) in the parameter orders of the two programs:
    [theta_trans_1..J, mu, log tau] and [mu, log tau, theta_1..J]; each mean / var an array of length J + 2."""
    y = np.asarray(y, dtype=np.float64)
    s2 = np.asarray(sigma, dtype=np.float64) ** 2
    u = _grid(y, s2, n, drop)
    logp, m, v, e_th, v_th, e_tt, v_tt = _conditionals(u, y, s2)
    p = np.exp(logp - logp.max())
    wq = np.full(n, u[1] - u[0])
    wq[0] = wq[-1] = 0.5 * (u[1] - u[0])
    p = p * wq
    p /= p.sum()

    def mom(e, var):              # E and Var of X from E[X | u], Var[X | u]
        e = e if e.ndim == 2 else e[:, None]
        var = var if var.ndim == 2 else var[:, None]
        mean = p @ e
        return mean, p @ (var + e * e) - mean * mean

    mu_m, mu_v = mom(m, v)
    u_m, u_v = mom(u, np.zeros_like(u))
    th_m, th_v = mom(e_th, v_th)
    tt_m, tt_v = mom(e_tt, v_tt)
    nc = (np.concatenate([tt_m, mu_m, u_m]), np.concatenate([tt_v, mu_v, u_v]))
    c = (np.concatenate([mu_m, u_m, th_m]), np.concatenate([mu_v, u_v, th_v]))
    return dict(noncentered=nc, centered=c)


def brute_force_mu_u(y, sigma, n_mu=1201, n_u=1201):
    """E and Var of (mu, log tau) by a plain 2-D grid over the marginal density p(mu, u | y) (theta integrated out:
    y_j | mu, tau ~ normal(mu, sigma_j^2 + tau^2)).  An independent check of posterior_moments."""
    y = np.asarray(y, dtype=np.float64)
    s2 = np.asarray(sigma, dtype=np.float64) ** 2
    u = _grid(y, s2, n_u, 40.0)
    mu = np.linspace(-60.0, 60.0, n_mu)
    U, M = np.meshgrid(u, mu, indexing="ij")
    V = s2 + np.exp(2.0 * U)[..., None]
    logp = (-M * M / 50.0 + U - np.log1p(np.exp(2.0 * U) / 25.0)
            - 0.5 * np.sum(np.log(V) + (y - M[..., None]) ** 2 / V, axis=-1))
    p = np.exp(logp - logp.max())
    p /= p.sum()
    out = {}
    for name, X in (("mu", M), ("u", U)):
        e = float(np.sum(p * X))
        out[name] = (e, float(np.sum(p * X * X)) - e * e)
    return out
