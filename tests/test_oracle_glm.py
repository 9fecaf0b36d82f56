"""Logistic regression on the CPU: the NumPy oracle's derivatives, the line restriction the device model evaluates
(far beyond the range of a naive log1p(exp(eta))), the exact posterior by quadrature, and the data validation of
BSModel."""
import numpy as np
import pytest

import klhr_b200 as kb
from oracle.glm_models import EMPTY, MODERATE, SEPARATED, WIDE, make_glm_model, synthetic
from oracle.glm_truth import brute_force_2d, posterior_moments

LR = "logistic_regression"


def _points(m, B, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    theta = rng.normal(size=(B, m.dim())) * scale
    rho = rng.normal(size=(B, m.dim()))
    rho /= np.linalg.norm(rho, axis=1, keepdims=True)
    return theta, rho


@pytest.mark.parametrize("data", [MODERATE, SEPARATED, WIDE], ids=["moderate", "separated", "wide"])
def test_lp_grad_and_dir2_against_central_differences(data):
    m = make_glm_model(LR, data)
    theta, rho = _points(m, 8, 1)
    lp, g = m.lp_grad(theta)
    h = 1e-6
    for i in range(m.dim()):
        e = np.zeros(m.dim())
        e[i] = h
        num = (m.lp(theta + e) - m.lp(theta - e)) / (2 * h)
        assert np.allclose(num, g[:, i], rtol=1e-6, atol=1e-6 * (1 + np.abs(lp))), (i, num, g[:, i])
    h = 1e-5
    gp = np.sum(m.lp_grad(theta + h * rho)[1] * rho, axis=-1)
    gm = np.sum(m.lp_grad(theta - h * rho)[1] * rho, axis=-1)
    d2 = m.dir2(theta, rho)
    assert np.allclose((gp - gm) / (2 * h), d2, rtol=1e-6, atol=1e-6 * (1 + np.abs(d2)))


def test_line_identity_up_to_eta_800():
    """l(t) - l(0) from a = X theta, b = X rho equals lp(theta + t rho) - lp(theta), and l', l'' match the directional
    derivatives, at |eta| up to 800, where log1p(exp(eta)) overflows in fp64."""
    m = make_glm_model(LR, MODERATE)
    rng = np.random.default_rng(2)
    for top in (None, 100.0, 800.0):
        theta, rho = _points(m, 64, 3)
        t = rng.normal(size=64)
        eta = np.concatenate([theta @ m.X.T, (theta + t[:, None] * rho) @ m.X.T])
        if top:                        # scale the points so that the largest |eta| is `top`
            f = top / np.abs(eta).max()
            theta, t, eta = theta * f, t * f, eta * f
        l, l1, l2 = m.line(theta, rho, t)
        ref = m.lp(theta + t[:, None] * rho) - m.lp(theta)
        sc = m.terms_scale(theta) + m.terms_scale(theta + t[:, None] * rho)
        assert np.all(np.isfinite(l)) and np.all(np.abs(l - ref) <= 1e-13 * sc)
        pt = theta + t[:, None] * rho
        assert np.allclose(l1, np.sum(m.lp_grad(pt)[1] * rho, -1), rtol=1e-12, atol=1e-12 * sc)
        assert np.allclose(l2, m.dir2(pt, rho), rtol=1e-12, atol=1e-12 * sc)
        if top == 800.0:
            with np.errstate(over="ignore"):
                assert not np.all(np.isfinite(np.log1p(np.exp(eta))))        # the form the model avoids


def test_quadrature_truth_converges():
    for data, fine in ((MODERATE, dict(n=101, R=15.0)), (SEPARATED, dict(n=301, R=20.0))):
        m = make_glm_model(LR, data)
        a, b = posterior_moments(m), posterior_moments(m, **fine)
        assert np.abs(a[0] - b[0]).max() < 1e-9 and np.abs(a[1] - b[1]).max() < 1e-9


def test_quadrature_truth_against_a_2d_grid_on_separated_data():
    m = make_glm_model(LR, SEPARATED)
    mean, var = posterior_moments(m)
    bf_mean, bf_var = brute_force_2d(m, (-6.0, -8.0), (6.0, 22.0))
    assert np.abs(mean - bf_mean).max() < 1e-8 and np.abs(var - bf_var).max() < 1e-8
    # the likelihood alone has no maximum: beta is held in by the prior, its posterior skewed far to the right
    assert mean[1] > 5 and var[1] > 2


def test_quadrature_truth_in_the_prior_limit():
    """N = 0: the posterior is the prior N(0, 6.25 I)."""
    mean, var = posterior_moments(make_glm_model(LR, EMPTY))
    assert np.abs(mean).max() < 1e-12 and np.abs(var - 6.25).max() < 1e-9


def test_quadrature_truth_against_exact_sampling_near_the_prior_limit():
    """Rejection from the prior (accept with probability prod_i p(y_i | theta) <= 1) samples the posterior exactly;
    three nearly uninformative observations keep the acceptance near 1/8."""
    m = make_glm_model(LR, synthetic(3, 1, seed=7, scale=0.01))
    rng = np.random.default_rng(0)
    kept = []
    while sum(len(k) for k in kept) < 200_000:
        th = rng.normal(size=(1_000_000, m.dim())) * 2.5
        loglik = m.lp(th) + np.sum(th * th, -1) / 12.5
        kept.append(th[np.log(rng.random(len(th))) < loglik])
    X = np.concatenate(kept)
    n = len(X)
    mean, var = posterior_moments(m)
    assert np.all(np.abs(X.mean(0) - mean) < 5 * np.sqrt(var / n))
    assert np.all(np.abs(X.var(0) - var) < 5 * var * np.sqrt(3.0 / n))


def test_bsmodel_host_data_and_names():
    m = kb.BSModel(stan_file="logistic_regression.stan", data=MODERATE)
    assert m.dim() == 3 and m.parameter_names() == ["alpha", "beta.1", "beta.2"]
    h = m._host
    X = np.asarray(h["data0"][:600]).reshape(200, 3)
    assert h["i0"] == 200 and h["i1"] == 2 and h["data0"].shape == (800,)
    assert np.array_equal(X[:, 0], np.ones(200)) and np.array_equal(X[:, 1:], np.asarray(MODERATE["x"]))
    assert np.array_equal(h["data0"][600:], MODERATE["y"])
    x = np.array([0.5, -1.0, 2.0])
    assert np.array_equal(m.constrain(x), x) and np.array_equal(m.unconstrain(x), x)
    e = kb.BSModel(stan_file="logistic_regression.stan", data=EMPTY)
    assert e.dim() == 3 and e._host["i0"] == 0 and e._host["data0"].shape == (0,)


@pytest.mark.parametrize("data,what", [
    ({"N": -1, "K": 1, "x": [], "y": []}, "N must be an integer"),
    ({"N": 1.5, "K": 1, "x": [[1.0]], "y": [1]}, "N must be an integer"),
    ({"N": 1, "K": 0, "x": [[]], "y": [1]}, "K must be an integer"),
    ({"N": 1, "K": 2.5, "x": [[1.0, 2.0]], "y": [1]}, "K must be an integer"),
    ({"N": 2, "K": 1, "x": [[1.0], [2.0], [3.0]], "y": [1, 0]}, "shape"),
    ({"N": 2, "K": 2, "x": [[1.0], [2.0]], "y": [1, 0]}, "shape"),
    ({"N": 2, "K": 1, "x": [[1.0], [float("nan")]], "y": [1, 0]}, "finite"),
    ({"N": 2, "K": 1, "x": [[1.0], [float("inf")]], "y": [1, 0]}, "finite"),
    ({"N": 2, "K": 1, "x": [[1.0], [2.0]], "y": [1]}, "length"),
    ({"N": 2, "K": 1, "x": [[1.0], [2.0]], "y": [1, 2]}, "0 or 1"),
    ({"N": 2, "K": 1, "x": [[1.0], [2.0]], "y": [1, 0.5]}, "0 or 1"),
    ({"N": 2, "K": 1, "x": [[1.0], [2.0]]}, "needs"),
])
def test_bsmodel_rejects_bad_data(data, what):
    with pytest.raises(ValueError, match=what):
        kb.BSModel(stan_file="logistic_regression.stan", data=data)


def test_unknown_program_still_raises():
    with pytest.raises(NotImplementedError):
        kb.BSModel(stan_file="garch.stan", data={})
