"""Exact posterior means and variances of Bayesian logistic regression for D = K + 1 <= 3.

TEST INFRASTRUCTURE (see oracle/__init__.py).  The posterior is smooth and, under the normal(0, 2.5) prior, decays
at least like a Gaussian in every direction.  In Laplace-whitened coordinates z (theta = mode + L z, L L^T the inverse
of the negative Hessian at the mode) it is close to a standard normal, and the tensor-product trapezoidal rule on
[-R, R]^D converges geometrically in the number of points per axis once R covers the mass.  Refining the rule and
widening its range shows the moments converged to < 1e-9 (tests/test_oracle_glm.py).
"""
from __future__ import annotations

import numpy as np

from .glm_models import LogisticRegression


def mode_and_hessian(model: LogisticRegression, iters=100):
    """Posterior mode by Newton's method (lp is strictly concave) and the Hessian of lp there."""
    th = np.zeros(model.dim())
    for _ in range(iters):
        _, g = model.lp_grad(th)
        eta = model.X @ th
        s = 1.0 / (1.0 + np.exp(-eta))
        H = -(model.X.T * (s * (1 - s))) @ model.X - np.eye(model.dim()) / 6.25
        step = np.linalg.solve(H, -g)
        th = th + step
        if np.max(np.abs(step)) < 1e-15 * (1 + np.max(np.abs(th))):
            break
    eta = model.X @ th
    s = 1.0 / (1.0 + np.exp(-eta))
    H = -(model.X.T * (s * (1 - s))) @ model.X - np.eye(model.dim()) / 6.25
    return th, H


def posterior_moments(model: LogisticRegression, n=None, R=None, chunk=1 << 16):
    """(mean, var) of every coordinate of theta = [alpha, beta_1..K] by the n^D-point trapezoidal rule on [-R, R]^D
    in Laplace-whitened coordinates (the end points carry weight ~ e^{-R^2 / 2}; the rule's weights are uniform).
    Defaults: n = 161, R = 15 for D <= 2; n = 81, R = 13 for D = 3 (near-Gaussian posteriors only)."""
    D = model.dim()
    if D > 3:
        raise ValueError("the tensor-product rule is meant for D <= 3")
    n = n or (161 if D <= 2 else 81)
    R = R or (15.0 if D <= 2 else 13.0)
    m, H = mode_and_hessian(model)
    L = np.linalg.cholesky(np.linalg.inv(-H))
    z1 = np.linspace(-R, R, n)
    grids = np.meshgrid(*([z1] * D), indexing="ij")
    Z = np.stack([g.reshape(-1) for g in grids], axis=1)
    lp0 = model.lp(m)
    s0, s1, s2 = 0.0, np.zeros(D), np.zeros(D)
    for c in range(0, Z.shape[0], chunk):
        th = m + Z[c:c + chunk] @ L.T
        w = np.exp(model.lp(th) - lp0)
        s0 += w.sum()
        s1 += w @ th
        s2 += w @ (th * th)
    mean = s1 / s0
    return mean, s2 / s0 - mean * mean


def brute_force_2d(model: LogisticRegression, lo, hi, n=1201):
    """(mean, var) of (alpha, beta) for K = 1 by a plain grid over the box [lo, hi] in the original coordinates: an
    independent check of posterior_moments."""
    assert model.dim() == 2
    a = np.linspace(lo[0], hi[0], n)
    b = np.linspace(lo[1], hi[1], n)
    A, B = np.meshgrid(a, b, indexing="ij")
    th = np.stack([A.reshape(-1), B.reshape(-1)], axis=1)
    lp = model.lp(th)
    p = np.exp(lp - lp.max())
    p /= p.sum()
    mean = p @ th
    return mean, p @ (th * th) - mean * mean
