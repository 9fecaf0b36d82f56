"""ARMA(1,1) on the CPU: the NumPy oracle's derivatives, the line restriction the device model evaluates (far beyond
the range of the naive Jacobian and Cauchy terms), the exact posterior by quadrature, and the data validation of
BSModel."""
import numpy as np
import pytest
import torch

import klhr_b200 as kb
from oracle.ts_models import LONG, MODERATE, RIDGE, SINGLE, bounded, make_ts_model, simulate
from oracle.ts_truth import brute_force_4d, posterior_moments, prior_b_variance

ARMA = "arma11"


def _points(B, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    theta = rng.normal(size=(B, 4)) * scale
    rho = rng.normal(size=(B, 4))
    rho /= np.linalg.norm(rho, axis=1, keepdims=True)
    return theta, rho


@pytest.mark.parametrize("data", [MODERATE, RIDGE, SINGLE], ids=["moderate", "ridge", "single"])
def test_lp_grad_and_dir2_against_central_differences(data):
    m = make_ts_model(ARMA, data)
    theta, rho = _points(8, 1)
    lp, g = m.lp_grad(theta)
    h = 1e-6
    for i in range(4):
        e = np.zeros(4)
        e[i] = h
        num = (m.lp(theta + e) - m.lp(theta - e)) / (2 * h)
        assert np.allclose(num, g[:, i], rtol=1e-6, atol=1e-6 * (1 + np.abs(lp))), (i, num, g[:, i])
    h = 1e-5
    gp = np.sum(m.lp_grad(theta + h * rho)[1] * rho, axis=-1)
    gm = np.sum(m.lp_grad(theta - h * rho)[1] * rho, axis=-1)
    d2 = m.dir2(theta, rho)
    assert np.allclose((gp - gm) / (2 * h), d2, rtol=1e-6, atol=1e-6 * (1 + np.abs(d2)))


def test_line_against_lp_along_random_lines():
    m = make_ts_model(ARMA, MODERATE)
    theta, rho = _points(64, 2)
    t = np.random.default_rng(3).normal(size=64)
    l, l1, l2 = m.line(theta, rho, t)
    pt = theta + t[:, None] * rho
    sc = m.terms_scale(theta) + m.terms_scale(pt)
    assert np.all(np.abs(l - (m.lp(pt) - m.lp(theta))) <= 1e-13 * sc)
    assert np.allclose(l1, np.sum(m.lp_grad(pt)[1] * rho, -1), rtol=1e-12, atol=1e-12 * sc)
    assert np.allclose(l2, m.dir2(pt, rho), rtol=1e-12, atol=1e-12 * sc)
    assert np.array_equal(m.line(theta, rho, np.zeros(64))[0], np.zeros(64))


def test_line_identity_far_out():
    """|a|, |b| up to 40 and |v| up to 300: every term finite, where log(1 - phi^2) is -inf (phi rounds to +-1) and
    log1p(sigma^2 / 25) overflows in fp32 (it does in fp64 from v ~ 355)."""
    m = make_ts_model(ARMA, MODERATE)
    rng = np.random.default_rng(4)
    B = 64
    theta = np.stack([rng.normal(size=B), rng.uniform(-40, 40, B), rng.uniform(-40, 40, B),
                      rng.uniform(-300, 300, B)], axis=1)
    theta[:4, 1:] = [[40.0, -40.0, 300.0], [-40.0, 40.0, -300.0], [39.0, 38.0, 299.0], [-38.5, -39.5, -299.0]]
    rho = rng.normal(size=(B, 4))
    rho /= np.linalg.norm(rho, axis=1, keepdims=True)
    t = rng.normal(size=B)
    pt = theta + t[:, None] * rho
    l, l1, l2 = m.line(theta, rho, t)
    lp, g = m.lp_grad(pt)
    assert np.all(np.isfinite(l)) and np.all(np.isfinite(l1)) and np.all(np.isfinite(l2))
    assert np.all(np.isfinite(lp)) and np.all(np.isfinite(g))
    sc = m.terms_scale(theta) + m.terms_scale(pt)
    assert np.all(np.abs(l - (lp - m.lp(theta))) <= 1e-13 * sc)
    assert np.allclose(l1, np.sum(g * rho, -1), rtol=1e-12, atol=1e-12 * sc)
    with np.errstate(all="ignore"):
        phi = np.tanh(pt[:, 1] / 2)
        assert np.isneginf(np.log(1 - phi * phi)).any()                         # the naive Jacobian
        v32 = pt[:, 3].astype(np.float32)
        assert np.isinf(np.log1p(np.exp(2 * v32) / np.float32(25))).any()       # the naive Cauchy term
    phi, q, J = bounded(np.array([40.0, -40.0]))
    assert np.all(np.abs(phi) == 1.0) and np.all(q > 0) and np.allclose(J, np.log(2) - 40 - 2 * np.log1p(np.exp(-40)))


@pytest.mark.parametrize("data", [MODERATE, RIDGE, SINGLE], ids=["moderate", "ridge", "single"])
def test_quadrature_truth_converges(data):
    """Refining the rule (k, kv) and widening its range (L, cut, zv) moves no moment by 1e-8 of its sd."""
    m = make_ts_model(ARMA, data)
    a = posterior_moments(m)
    b = posterior_moments(m, k=6.0, kv=3.0, zv=16.0, cut=50.0, L=50.0)
    sd = np.sqrt(a[1])
    assert np.all(np.abs(a[0] - b[0]) < 1e-8 * sd) and np.all(np.abs(a[1] - b[1]) < 1e-8 * sd), (a, b)


def test_quadrature_truth_against_a_plain_4d_grid():
    """MODERATE: a plain 33^4 grid over mean +- 10 sd, from lp alone, agrees to its resolution: ~2e-7 sd in the means
    and ~3e-6 in the relative variances (its tails are cut at 10 sd of a skewed posterior)."""
    m = make_ts_model(ARMA, MODERATE)
    mean, var = posterior_moments(m)
    sd = np.sqrt(var)
    bm, bv = brute_force_4d(m, mean - 10 * sd, mean + 10 * sd, n=33)
    assert np.all(np.abs(bm - mean) < 1e-6 * sd) and np.all(np.abs(bv - var) < 1e-5 * var), (bm - mean, bv - var)


def test_quadrature_truth_single_observation_b_is_its_prior():
    """T = 1: theta does not enter the likelihood, so b has mean 0 and the variance of the pushed-forward prior."""
    mean, var = posterior_moments(make_ts_model(ARMA, SINGLE))
    vb = prior_b_variance()
    assert abs(mean[2]) < 1e-10 and abs(var[2] - vb) < 1e-8 * np.sqrt(vb)
    assert abs(vb - 3.12667) < 1e-5


def test_simulator_is_seeded():
    assert simulate(5, 1.0, 0.6, 0.3, 1.0, seed=9) == simulate(5, 1.0, 0.6, 0.3, 1.0, seed=9)
    assert len(LONG["y"]) == LONG["T"] == 10_000 and len(RIDGE["y"]) == 100 and len(MODERATE["y"]) == 200


def test_bsmodel_host_data_names_and_transforms():
    m = kb.BSModel(stan_file="arma11.stan", data=MODERATE)
    assert m.dim() == 4 and m.parameter_names() == ["mu", "phi", "theta", "sigma"]
    h = m._host
    assert h["i0"] == 200 and np.array_equal(h["data0"], np.asarray(MODERATE["y"]))
    x = np.array([0.5, 1.2, -0.7, 0.3])
    c = m.constrain(x)
    assert np.allclose(c, [0.5, np.tanh(0.6), np.tanh(-0.35), np.exp(0.3)], rtol=1e-15)
    assert np.allclose(m.unconstrain(c), x, rtol=1e-14)
    ct = m.constrain(torch.as_tensor(x)).numpy()
    assert np.allclose(ct, c, rtol=1e-15) and np.allclose(m.unconstrain(torch.as_tensor(c)).numpy(), x, rtol=1e-14)


@pytest.mark.parametrize("data,what", [
    ({"T": 0, "y": []}, "T must be an integer"),
    ({"T": 1.5, "y": [1.0]}, "T must be an integer"),
    ({"T": True, "y": [1.0]}, "T must be an integer"),
    ({"T": 2, "y": [1.0]}, "length"),
    ({"T": 2, "y": [1.0, 2.0, 3.0]}, "length"),
    ({"T": 2, "y": [[1.0, 2.0]]}, "length"),
    ({"T": 2, "y": [1.0, float("nan")]}, "finite"),
    ({"T": 2, "y": [1.0, float("inf")]}, "finite"),
    ({"T": 2, "y": ["a", 1.0]}, "numeric"),
    ({"T": 2}, "needs"),
])
def test_bsmodel_rejects_bad_data(data, what):
    with pytest.raises(ValueError, match=what):
        kb.BSModel(stan_file="arma11.stan", data=data)
