"""Exact posterior means and variances of ARMA(1,1) (all four unconstrained coordinates [mu, a, b, v]).

TEST INFRASTRUCTURE (see oracle/__init__.py).  The recursion is affine in mu: err_t = e_t - mu g_t with
e_1 = y_1, g_1 = 1 + phi, e_t = y_t - phi y_{t-1} - theta e_{t-1}, g_t = 1 - theta g_{t-1}.  So S0 = sum e^2,
S1 = sum e g and S2 = sum g^2 depend on (a, b) only, and given (a, b, v) mu is Gaussian with precision
P = 1/100 + e^{-2v} S2 and mean m = e^{-2v} S1 / P.  Integrating mu out leaves the weight
exp(P m^2 / 2 - e^{-2v} S0 / 2) / sqrt(P) times the (a, b, v) terms of lp; the moments of mu come from m and
m^2 + 1 / P.  What remains is a trapezoidal rule over (a, b) -- one O(T) recursion per node -- times one over v.

  - (a, b): a coarse grid over [-L, L]^2 locates the mass; the fine grid covers the box where the coarse log-weight
    is within ``cut`` of its maximum, with spacing 1/k of the conditional standard deviations at the coarse mode;
    nodes whose coarse neighbourhood lies below the cut are skipped.
  - v: for T >= 2, per (a, b) node a grid centred on the conditional mode of v with the residual sum of squares at
    the best mu, v* = log(R / (T - 1)) / 2, spacing 1/kv of sd_v = 1 / sqrt(2 (T - 1)) and half-width zv sd_v
    (the trapezoidal rule's error on a smooth peak of width sd_v falls like exp(-2 pi^2 kv^2)); for T = 1 one wide
    grid, since the single residual can be zeroed by mu and v is then held in by its prior alone.
Every grid has uniform weights and negligible mass at its ends.  Refining the rule and widening its range shows the
moments converged to < 1e-8 of each coordinate's posterior sd (tests/test_oracle_ts.py).
"""
from __future__ import annotations

import numpy as np

from .hier_models import LOG25, _softplus
from .ts_models import Arma11, bounded


def _sums(y, a, b):
    """(S0, S1, S2, R, base) at the nodes (a, b), base = -phi^2/8 - theta^2/8 + J(a) + J(b).  R = S0 - S1^2 / S2, the
    residual sum of squares at the best mu, cancels in that form (and S2 can be ~0 where phi rounds to -1): it is
    r22^2 of the 2-column QR factor of the rows (g_t, e_t), kept up to date by Givens rotations (R = 0 for T = 1)."""
    A, B = bounded(a), bounded(b)
    ph, th = A[0], B[0]
    e = np.full_like(a, y[0])
    g = 1.0 + ph
    S0, S1, S2 = e * e, e * g, g * g
    r11, r12, r22 = np.abs(g), np.where(g < 0, -e, e), np.zeros_like(e)
    for t in range(1, len(y)):
        e = y[t] - ph * y[t - 1] - th * e
        g = 1.0 - th * g
        S0, S1, S2 = S0 + e * e, S1 + e * g, S2 + g * g
        rho = np.hypot(r11, g)
        ok = rho > 0
        c = np.where(ok, r11 / np.where(ok, rho, 1.0), 1.0)
        s = np.where(ok, g / np.where(ok, rho, 1.0), 0.0)
        r11, r12, x2 = rho, c * r12 + s * e, c * e - s * r12
        r22 = np.hypot(r22, x2)
    return S0, S1, S2, r22 * r22, -(ph * ph + th * th) / 8.0 + A[2] + B[2]


def _logw(T, S0, S1, S2, R, base, v):
    """log weight of (a, b, v) with mu integrated out (constants dropped), and m, P; v broadcasts against the sums.
    P m^2 / 2 - e^{-2v} S0 / 2 = -e^{-2v} (S0 / 100 + e^{-2v} S2 R) / (2 P), free of cancellation."""
    em2 = np.exp(-2.0 * v)
    P = 0.01 + em2 * S2
    m = em2 * S1 / P
    lw = base - _softplus(2.0 * v - LOG25)[0] + (1 - T) * v - 0.5 * em2 * (0.01 * S0 + em2 * S2 * R) / P - 0.5 * np.log(P)
    return lw, m, P


def _vstar(T, R):
    return 0.5 * np.log(np.maximum(R, 1e-300) / (T - 1))


def _profile(y, a, b):
    """Coarse log-weight at (a, b): the weight at v* (T >= 2) or the maximum over a wide v grid (T = 1)."""
    T = len(y)
    S0, S1, S2, R, base = _sums(y, a, b)
    if T >= 2:
        return _logw(T, S0, S1, S2, R, base, _vstar(T, R))[0]
    v = np.linspace(-40.0, 25.0, 261)
    return _logw(T, S0[..., None], S1[..., None], S2[..., None], R[..., None], base[..., None], v)[0].max(-1)


def posterior_moments(model: Arma11, k=4.0, L=40.0, cut=40.0, kv=2.0, zv=12.0, h0=0.25, max_h=0.25, chunk=1 << 15):
    """(mean, var) of [mu, a, b, v].  k, kv: points per conditional sd in (a, b) and in v; L: half-width of the
    coarse (a, b) box; cut: log-weight below the coarse maximum that is dropped; zv: half-width of the v grid in
    sd_v (T >= 2); h0: coarse spacing; max_h: largest fine (a, b) spacing."""
    y = model.y
    T = len(y)
    # coarse grid: where the mass is
    c = np.arange(-L, L + h0 / 2, h0)
    CA, CB = np.meshgrid(c, c, indexing="ij")
    lc = _profile(y, CA, CB)
    lc = np.where(np.isfinite(lc), lc, -np.inf)
    ref = lc.max()
    i, j = np.unravel_index(np.argmax(lc), lc.shape)
    keep = lc > ref - cut
    dil = keep.copy()                                       # one coarse cell of margin all round
    for di in (-1, 0, 1):
        for dj in (-1, 0, 1):
            dil |= np.roll(np.roll(keep, di, 0), dj, 1)
    ia, ja = np.nonzero(dil.any(1))[0], np.nonzero(dil.any(0))[0]
    lo_a, hi_a = c[max(ia[0] - 1, 0)], c[min(ia[-1] + 1, len(c) - 1)]
    lo_b, hi_b = c[max(ja[0] - 1, 0)], c[min(ja[-1] + 1, len(c) - 1)]
    # conditional sds at the coarse mode from second differences of the profile
    d = 0.02
    a0, b0 = c[i], c[j]
    f = lambda da, db: _profile(y, np.array([a0 + da]), np.array([b0 + db]))[0]
    f0 = f(0, 0)
    sa = 1.0 / np.sqrt(max(-(f(d, 0) - 2 * f0 + f(-d, 0)) / d ** 2, 1e-12))
    sb = 1.0 / np.sqrt(max(-(f(0, d) - 2 * f0 + f(0, -d)) / d ** 2, 1e-12))
    ha, hb = min(sa / k, max_h), min(sb / k, max_h)
    fa = np.arange(lo_a, hi_a + ha / 2, ha)
    fb = np.arange(lo_b, hi_b + hb / 2, hb)
    FA, FB = np.meshgrid(fa, fb, indexing="ij")
    ci = np.clip(np.rint((FA + L) / h0).astype(int), 0, len(c) - 1)
    cj = np.clip(np.rint((FB + L) / h0).astype(int), 0, len(c) - 1)
    sel = dil[ci, cj]
    pa, pb = FA[sel], FB[sel]
    if T >= 2:
        sv = 1.0 / np.sqrt(2.0 * (T - 1))
        hv = sv / kv
        kk = np.arange(-np.ceil(zv * kv), np.ceil(zv * kv) + 1) * hv
    else:
        vg = np.arange(-45.0, 30.0 + 1e-9, 0.5 / kv)
    acc = np.zeros(9)
    for s in range(0, len(pa), chunk):
        a, b = pa[s:s + chunk], pb[s:s + chunk]
        S0, S1, S2, R, base = _sums(y, a, b)
        if T >= 2:
            v = _vstar(T, R)[:, None] + kk[None, :]
        else:
            v = np.broadcast_to(vg[None, :], (len(a), len(vg)))
        lw, m, P = _logw(T, S0[:, None], S1[:, None], S2[:, None], R[:, None], base[:, None], v)
        w = np.exp(lw - ref)
        w = np.where(np.isfinite(w), w, 0.0)
        wn = w.sum(1)
        acc += np.array([wn.sum(), (w * m).sum(), (w * (m * m + 1.0 / P)).sum(), wn @ a, wn @ (a * a), wn @ b,
                         wn @ (b * b), (w * v).sum(), (w * v * v).sum()])
    Z = acc[0]
    mean = np.array([acc[1], acc[3], acc[5], acc[7]]) / Z
    second = np.array([acc[2], acc[4], acc[6], acc[8]]) / Z
    return mean, second - mean * mean


def brute_force_4d(model: Arma11, lo, hi, n=41):
    """(mean, var) of [mu, a, b, v] by a plain n^4 grid over the box [lo, hi] of the original coordinates, lp from the
    model's own recursion: an independent check of posterior_moments, to the grid's resolution."""
    grids = [np.linspace(lo[k], hi[k], n) for k in range(4)]
    G = np.stack([g.reshape(-1) for g in np.meshgrid(*grids, indexing="ij")], axis=1)
    lp = model.lp(G)
    p = np.exp(lp - lp.max())
    p /= p.sum()
    mean = p @ G
    return mean, p @ (G * G) - mean * mean


def prior_b_variance(L=60.0, n=120_001):
    """Variance of b under the pushed-forward theta ~ normal(0, 2) prior on (-1, 1) (mean 0 by symmetry), by a 1-D
    rule: the exact posterior of b when T = 1, where theta does not enter the likelihood."""
    b = np.linspace(-L, L, n)
    th, _, J = bounded(b)
    w = np.exp(-th * th / 8.0 + J)
    return float((w @ (b * b)) / w.sum())
