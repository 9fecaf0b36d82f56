"""Eight schools (non-centered and centered) on the CPU: the NumPy oracle's derivatives, the O(1) line restriction
the device models are built on, the exact posterior by quadrature, and the data validation of BSModel."""
import numpy as np
import pytest

import klhr_b200 as kb
from oracle.hier_truth import brute_force_mu_u, posterior_moments
from oracle.hier_models import EIGHT_SCHOOLS_DATA, EightSchoolsC, EightSchoolsNC, make_hier_model

NAMES = ("eight_schools_noncentered", "eight_schools_centered")


def _points(m, B, seed, uspread=1.5):
    rng = np.random.default_rng(seed)
    theta = rng.normal(size=(B, m.dim()))
    k = m.J + 1 if isinstance(m, EightSchoolsNC) else 1
    theta[:, k] = rng.normal(size=B) * uspread
    if isinstance(m, EightSchoolsC):
        theta[:, 2:] = theta[:, 2:] * 5 + 4
        theta[:, 0] *= 5
    rho = rng.normal(size=(B, m.dim()))
    rho /= np.linalg.norm(rho, axis=1, keepdims=True)
    return theta, rho, k


@pytest.mark.parametrize("name", NAMES)
def test_lp_grad_against_central_differences(name):
    m = make_hier_model(name, EIGHT_SCHOOLS_DATA)
    theta, _, _ = _points(m, 16, 1)
    lp, g = m.lp_grad(theta)
    h = 1e-6
    for i in range(m.dim()):
        e = np.zeros(m.dim())
        e[i] = h
        num = (m.lp(theta + e) - m.lp(theta - e)) / (2 * h)
        assert np.allclose(num, g[:, i], rtol=1e-6, atol=1e-6 * (1 + np.abs(lp))), (i, num, g[:, i])


@pytest.mark.parametrize("name", NAMES)
def test_dir2_against_differences_of_the_directional_gradient(name):
    m = make_hier_model(name, EIGHT_SCHOOLS_DATA)
    theta, rho, _ = _points(m, 16, 2)
    h = 1e-5
    gp = np.sum(m.lp_grad(theta + h * rho)[1] * rho, axis=-1)
    gm = np.sum(m.lp_grad(theta - h * rho)[1] * rho, axis=-1)
    d2 = m.dir2(theta, rho)
    assert np.allclose((gp - gm) / (2 * h), d2, rtol=1e-6, atol=1e-6 * (1 + np.abs(d2)))


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("J", [1, 8, 30])
def test_line_restriction_from_sums_equals_the_density(name, J):
    """l(t) from the 13 (non-centered) / 6 (centered) sums equals lp(theta + t rho), also at u = +-300 (where
    log1p(e^{2u} / 25) overflows in fp32) and, for the centered form, whose density stays finite there, at u = 400,
    where it overflows in fp64 too and only the softplus form of the Cauchy term is finite."""
    rng = np.random.default_rng(J)
    m = make_hier_model(name, {"J": J, "y": (rng.normal(size=J) * 10).tolist(), "sigma": (5 + 10 * rng.random(J)).tolist()})
    theta, rho, k = _points(m, 64, 3 + J)
    t = rng.normal(size=64)
    ref = m.lp(theta + t[:, None] * rho)
    got = m.line_from_sums(theta, rho, t)
    assert np.allclose(got, ref, rtol=1e-12, atol=1e-10), np.abs(got - ref).max()
    # far from the mode: the line restriction keeps full relative accuracy
    for u in (300.0, -300.0) + ((400.0,) if name == "eight_schools_centered" else ()):
        th = theta.copy()
        th[:, k] = u
        r = rho.copy()
        r[:, k] *= 0.01
        ref = m.lp(th + t[:, None] * r)
        got = m.line_from_sums(th, r, t)
        assert np.all(np.isfinite(ref)) and np.allclose(got, ref, rtol=1e-12, atol=0)
        with np.errstate(over="ignore"):
            naive = -np.log1p(np.exp(2 * (u + t * r[:, k])) / 25.0)
        assert u < 355 or not np.any(np.isfinite(naive))        # the form the model avoids


def test_quadrature_truth_converges_and_matches_a_2d_grid():
    y, s = EIGHT_SCHOOLS_DATA["y"], EIGHT_SCHOOLS_DATA["sigma"]
    a = posterior_moments(y, s, n=20001)
    b = posterior_moments(y, s, n=80001, drop=120.0)
    for k in ("noncentered", "centered"):
        for i in range(2):
            assert np.abs(a[k][i] - b[k][i]).max() < 1e-9
    # the two parametrisations share mu and log tau
    assert np.allclose(a["noncentered"][0][-2:], a["centered"][0][:2], rtol=0, atol=1e-14)
    bf = brute_force_mu_u(y, s)
    mean_c, var_c = a["centered"]
    assert abs(bf["mu"][0] - mean_c[0]) < 1e-6 and abs(bf["mu"][1] - var_c[0]) < 1e-6
    assert abs(bf["u"][0] - mean_c[1]) < 1e-6 and abs(bf["u"][1] - var_c[1]) < 1e-6
    # the classic posterior: E mu = 4.4, E tau of order 3.6 (log tau mean 0.80)
    assert abs(mean_c[0] - 4.3968) < 1e-3 and abs(mean_c[1] - 0.8021) < 1e-3


def test_quadrature_truth_in_the_prior_limit():
    """sigma -> infinity: the posterior is the prior.  log(tau / 5) of a half-Cauchy(0, 5) has density
    1 / (pi cosh v): mean 0, variance pi^2 / 4; mu ~ N(0, 25); theta_trans ~ N(0, 1)."""
    r = posterior_moments([3.0, -1.0, 7.0], [1e30] * 3)
    mean, var = r["noncentered"]
    assert np.allclose(mean, [0, 0, 0, 0, np.log(5.0)], atol=1e-9)
    assert np.allclose(var, [1, 1, 1, 25, np.pi ** 2 / 4], rtol=1e-9)


def test_quadrature_truth_against_a_sampled_posterior():
    """Exact sampling of the joint through the conditionals (u on the quadrature grid, then mu, then theta)."""
    y = np.array(EIGHT_SCHOOLS_DATA["y"])
    s = np.array(EIGHT_SCHOOLS_DATA["sigma"])
    from oracle.hier_truth import _conditionals, _grid
    u = _grid(y, s * s, 20001, 80.0)
    logp, m, v = _conditionals(u, y, s * s)[:3]
    p = np.exp(logp - logp.max())
    p /= p.sum()
    rng = np.random.default_rng(0)
    n = 400_000
    k = rng.choice(len(u), size=n, p=p)
    tau2 = np.exp(2 * u[k])[:, None]
    mu = m[k] + np.sqrt(v[k]) * rng.normal(size=n)
    prec = 1 / s ** 2 + 1 / tau2
    th = (y / s ** 2 + mu[:, None] / tau2) / prec + rng.normal(size=(n, len(y))) / np.sqrt(prec)
    X = np.column_stack([mu, u[k], th])
    mean, var = posterior_moments(y, s)["centered"]
    se = np.sqrt(var / n)
    assert np.all(np.abs(X.mean(0) - mean) < 5 * se)
    # step of the grid: the u draws are on a 0.01-wide lattice, which adds h^2 / 12 to nothing here (same grid)
    assert np.all(np.abs(X.var(0) - var) < 5 * var * np.sqrt(2.0 / n) + 1e-12)


@pytest.mark.parametrize("name", NAMES)
def test_bsmodel_host_data_names_and_transforms(name):
    m = kb.BSModel(stan_file=f"stan/{name}.stan", data=EIGHT_SCHOOLS_DATA)
    assert m.dim() == 10
    h = m._host
    assert h["i0"] == 8 and h["data0"].shape == (16,)
    assert np.array_equal(h["data0"][:8], EIGHT_SCHOOLS_DATA["y"])
    assert np.allclose(h["data0"][8:], 1.0 / np.asarray(EIGHT_SCHOOLS_DATA["sigma"]) ** 2, rtol=0, atol=0)
    names = m.parameter_names()
    k = names.index("tau")
    if name == "eight_schools_noncentered":
        assert names == [f"theta_trans.{j}" for j in range(1, 9)] + ["mu", "tau"]
    else:
        assert names == ["mu", "tau"] + [f"theta.{j}" for j in range(1, 9)]
    x = np.arange(10, dtype=np.float64) * 0.1
    c = m.constrain(x)
    assert c[k] == np.exp(x[k]) and np.array_equal(np.delete(c, k), np.delete(x, k))
    assert np.allclose(m.unconstrain(c), x, rtol=0, atol=1e-15)


@pytest.mark.parametrize("data,what", [
    ({"J": 0, "y": [], "sigma": []}, "J"),
    ({"J": 2.5, "y": [1, 2], "sigma": [1, 1]}, "J"),
    ({"J": 3, "y": [1, 2], "sigma": [1, 1, 1]}, "length"),
    ({"J": 2, "y": [1, 2], "sigma": [1]}, "length"),
    ({"J": 2, "y": [1, 2], "sigma": [1, 0]}, "sigma"),
    ({"J": 2, "y": [1, 2], "sigma": [1, -3]}, "sigma"),
    ({"J": 2, "y": [1, 2], "sigma": [1, float("inf")]}, "sigma"),
    ({"J": 2, "y": [1, 2], "sigma": [1, float("nan")]}, "sigma"),
    ({"J": 2, "y": [1, float("nan")], "sigma": [1, 1]}, "y"),
    ({"J": 2, "y": [1, 2]}, "sigma"),
])
@pytest.mark.parametrize("name", NAMES)
def test_bsmodel_rejects_bad_data(name, data, what):
    with pytest.raises(ValueError, match=what):
        kb.BSModel(stan_file=f"stan/{name}.stan", data=data)
