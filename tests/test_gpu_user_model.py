"""CudaModel on the GPU: the AD primitives against their analytic derivatives, user restatements of three built-in
targets against those targets and the oracle (evaluation, KL objective, step replay on every kernel, free-running
parity), posteriors within 4 MCSE of exact truths with no slack, two user targets in one process, and the refusals of
the C ABI."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest
import torch

import klhr_b200 as kb
from gpu_util import assert_kernel, device, fit_pair, rel_errors, up
from klhr_b200 import _lib
from klhr_b200.diagnostics import chain_summary
from oracle import batched
from oracle import glm_models, glm_truth, hier_truth, ts_models, ts_truth
from oracle.hier_models import EIGHT_SCHOOLS_DATA, make_hier_model
from oracle.user_models import PROBE, PROBE_BASE, PROBE_DIM, Trio, probe_jet

pytestmark = pytest.mark.gpu

F64, F32 = torch.float64, torch.float32
TARGETS = Path(__file__).resolve().parent / "user_targets"
NC = "eight_schools_noncentered"
LOGIT = "logistic_regression"
ARMA = "arma11"
# (user source, built-in Stan name, data, dim, oracle model)
RESTATED = {
    "es_nc": ("eight_schools_noncentered.cuh", NC, EIGHT_SCHOOLS_DATA, 10, lambda d: make_hier_model(NC, d)),
    "logit": ("logistic_regression.cuh", LOGIT, glm_models.MODERATE, 3, lambda d: glm_models.make_glm_model(LOGIT, d)),
    "wide": ("logistic_regression.cuh", LOGIT, glm_models.WIDE, 25, lambda d: glm_models.make_glm_model(LOGIT, d)),
    "arma": ("arma11.cuh", ARMA, ts_models.MODERATE, 4, lambda d: ts_models.make_ts_model(ARMA, d)),
}


def _user(name):
    src, _, data, dim, _ = RESTATED[name]
    return kb.CudaModel(TARGETS / src, data, dim, device=device())


def _builtin(name):
    _, stan, data, _, _ = RESTATED[name]
    return kb.BSModel(stan_file=f"stan/{stan}.stan", data=data, device=device())


def _oracle(name, dtype=F64):
    _, _, data, _, make = RESTATED[name]
    if dtype == F32:            # the oracle on the data the device holds
        data = {k: (np.asarray(v, dtype=np.float32).astype(np.float64).tolist()
                    if isinstance(v, (list, np.ndarray)) and np.asarray(v).dtype.kind == "f" else v)
                for k, v in data.items()}
    return make(data)


def _states(name, B, seed, spread=1.0):
    """Points around the posterior bulk (a few oracle-free anchors) and unit directions."""
    rng = np.random.default_rng(seed)
    D = RESTATED[name][3]
    centre = {"es_nc": np.r_[np.zeros(8), 4.0, 1.0], "arma": np.array([0.5, 1.4, 0.6, 0.0])}.get(name, np.zeros(D))
    x = centre + rng.normal(size=(B, D)) * 0.3 * spread
    rho = rng.normal(size=(B, D))
    rho /= np.linalg.norm(rho, axis=1, keepdims=True)
    return x, rho


def _trio(K):
    data = {"nu": 9.0, "s": list(np.linspace(0.5, 2.0, K)), "a": 3.0, "b": 2.0, "alpha": 2.0, "beta": 3.0}
    return kb.CudaModel(TARGETS / "trio.cuh", data, K + 2, device=device()), Trio.from_data(data)


# ------------------------------------------------------------------ AD primitives
def _probe_args(k, dtype):
    """Arguments over each primitive's range, far ones included.  fp32: where f, f' and f'' are all normal fp32
    numbers (or exactly 0 in both precisions, as softplus far left)."""
    rng = np.random.default_rng(100 + k)
    lg = lambda lo, hi, n=64: 10.0 ** rng.uniform(lo, hi, n)
    f64 = dtype == F64
    name = PROBE[k][0]
    if name in ("exp", "expm1"):
        return rng.uniform(-700, 700, 128) if f64 else rng.uniform(-80, 80, 128)
    if name in ("log", "sqrt"):
        return lg(-150, 300, 128) if f64 else lg(-12, 18 if name == "log" else 24, 128)
    if name == "log1p":
        return np.r_[-1 + lg(-12, 0), lg(-10, 300)] if f64 else np.r_[-1 + lg(-3, 0), lg(-5, 18)]
    if name == "square":
        return np.r_[lg(-100, 150), -lg(-100, 150)] if f64 else np.r_[lg(-15, 18), -lg(-15, 18)]
    if name == "pow2.5":
        return lg(-100, 100, 128) if f64 else lg(-10, 10, 128)
    if name == "tanh":
        return rng.uniform(-400, 400, 128) if f64 else rng.uniform(-40, 40, 128)
    if name in ("log1p_exp", "log_inv_logit"):
        return np.r_[rng.uniform(-40, 40, 64), rng.uniform(-1e5, 1e5, 64)] if f64 else \
            np.r_[rng.uniform(-20, 20, 64), rng.choice([-1, 1], 64) * rng.uniform(200, 1e4, 64)]
    if name == "fabs":
        return np.r_[lg(-100, 100), -lg(-100, 100)] if f64 else np.r_[lg(-30, 30), -lg(-30, 30)]
    return np.r_[lg(-100, 100), -lg(-100, 100)] if f64 else np.r_[lg(-12, 12), -lg(-12, 12)]   # reciprocal


@pytest.mark.parametrize("dtype", [F64, F32], ids=["fp64", "fp32"])
def test_ad_primitives_value_first_and_second_derivative(dtype):
    """Probe target, one-node fit (x = 0, w = 1): theta_k = a / 2, rho = e_k and eta = (a / 2, 0) put the one evaluation
    at theta_k + m = a exactly (a doubling), so kl_eval gives f = -l(m) (up to the rounding of l(0) = f_k(a / 2)),
    g_0 = -f_k'(a) and H_00 = -f_k''(a).  fp64 to 1e-13 relative; fp32 to 1e-5 relative (about 80 units of fp32
    rounding)."""
    tol = 1e-13 if dtype == F64 else 1e-5
    np_t = np.float64 if dtype == F64 else np.float32
    kfit = kb.FitConfig(family="gauss", N=1).for_dtype(dtype)
    for k in range(PROBE_DIM):
        w = np.zeros(PROBE_DIM)
        w[k] = 1.0
        model = kb.CudaModel(TARGETS / "probe.cuh", {"w": w}, PROBE_DIM, device=device())
        half = (_probe_args(k, dtype) / 2).astype(np_t)
        arg = (half + half).astype(np.float64)
        B = len(half)
        base = np.tile(PROBE_BASE, (B, 1))
        base[:, k] = half
        rho = np.zeros((B, PROBE_DIM))
        rho[:, k] = 1.0
        eta = np.stack([half.astype(np.float64), np.zeros(B)], axis=1)
        f, g, H = (t.double().cpu().numpy() for t in kb.kl_eval(model, kfit, up(base, dtype), up(rho, dtype),
                                                                  up(eta, dtype), hessian=True))
        v, d1, d2 = probe_jet(k, arg)
        v0 = probe_jet(k, half.astype(np.float64))[0]
        name = PROBE[k][0]
        for got, want, scale, what in ((-f, v, np.abs(v) + np.abs(v0), "f"), (-g[:, 0], d1, np.abs(d1), "f'"),
                                       (-H[:, 0, 0], d2, np.abs(d2), "f''")):
            want = want.astype(np_t).astype(np.float64)        # the analytic value in the arithmetic type
            err = np.abs(got - want)
            ok = err <= tol * scale + 1e-300
            assert ok.all(), (name, what, arg[~ok][:4], got[~ok][:4], want[~ok][:4])


# ------------------------------------------------------------------ restatements against the built-in targets
@pytest.mark.parametrize("name", ["es_nc", "logit", "wide", "arma"])
def test_log_density_gradient_matches_builtin_and_oracle(name):
    """fp64: user and built-in agree to 1e-12 of the terms' scale, and both match the oracle to the same bar;
    lp bitwise equal to log_density."""
    x, _ = _states(name, 256, 1, spread=3.0)
    user, bi, om = _user(name), _builtin(name), _oracle(name)
    lu, gu = (t.cpu().numpy() for t in user.log_density_gradient(up(x)))
    lb, gb = (t.cpu().numpy() for t in bi.log_density_gradient(up(x)))
    assert np.array_equal(lu, user.log_density(up(x)).cpu().numpy())
    lr, gr = om.lp_grad(x)
    sc = np.abs(lr) + 1.0
    if name == "arma":
        sc, gs = om.error_scales(x)
    else:
        gs = np.abs(gr).max(axis=1, keepdims=True) + 1.0
    for l in (lu, lb):
        assert np.all(np.abs(l - lr) <= 1e-12 * sc), np.max(np.abs(l - lr) / sc)
    for g in (gu, gb):
        assert np.all(np.abs(g - gr) <= 1e-12 * gs), np.max(np.abs(g - gr) / gs)


@pytest.mark.parametrize("name", ["es_nc", "logit", "arma"])
@pytest.mark.parametrize("family", ["gauss", "sinh"])
def test_kl_eval_matches_builtin(name, family):
    B = 64
    x, rho = _states(name, B, 4)
    eta = np.random.default_rng(5).normal(size=(B, 2 if family == "gauss" else 4)) * 0.3
    kfit, _ = fit_pair(family)
    fu, gu, Hu = (t.cpu().numpy() for t in kb.kl_eval(_user(name), kfit, up(x), up(rho), up(eta), hessian=True))
    fb, gb, Hb = (t.cpu().numpy() for t in kb.kl_eval(_builtin(name), kfit, up(x), up(rho), up(eta), hessian=True))
    sc = np.maximum(1.0, np.abs(fb))
    assert np.all(np.abs(fu - fb) <= 1e-10 * sc), np.max(np.abs(fu - fb) / sc)
    assert np.all(np.abs(gu - gb) <= 1e-10 * sc[:, None] * np.maximum(1, np.abs(gb))), np.max(np.abs(gu - gb))
    assert np.all(np.abs(Hu - Hb) <= 1e-10 * sc[:, None, None] * np.maximum(1, np.abs(Hb))), np.max(np.abs(Hu - Hb))


REPLAY = [("es_nc", "gauss", F64, "chain_serial"), ("es_nc", "sinh", F64, "chain_serial"),
          ("wide", "gauss", F64, "chain_octet"), ("arma", "gauss", F64, "octet"), ("arma", "sinh", F64, "octet"),
          ("logit", "gauss", F32, "chain_serial")]


@pytest.mark.parametrize("name,family,dtype,kernel", REPLAY, ids=[f"{r[0]}-{r[1]}-{str(r[2])[-7:]}-{r[3]}" for r in REPLAY])
def test_step_replay_matches_oracle(name, family, dtype, kernel):
    B = 512
    x, rho = _states(name, B, 6)
    rng = np.random.default_rng(7)
    z_init, z_prop, u = rng.normal(size=B), rng.normal(size=B), rng.random(B)
    init4 = rng.normal(size=(B, 4)) if family == "sinh" else None
    model = _user(name)
    kfit, ofit = fit_pair(family, dtype)
    kfit.force_octet = kernel == "octet"
    assert_kernel(model, kfit, dtype, kernel, free_running=False)
    th = up(x, dtype)
    tr = kb.step_replay(model, kfit, th, up(rho, dtype), up(z_init, dtype), up(z_prop, dtype), up(u, dtype),
                        init4=up(init4, dtype) if init4 is not None else None)
    torch.cuda.synchronize()
    gpu = dict(eta=tr.eta[0].double().cpu().numpy(), zp=tr.zp[0].double().cpu().numpy(),
               r=tr.r[0].double().cpu().numpy(), accept=tr.accept[0].cpu().numpy().astype(bool),
               evals=tr.evals[0].cpu().numpy(), theta=th.double().cpu().numpy())
    if dtype == F32:
        f32 = lambda a: None if a is None else np.asarray(a, dtype=np.float32).astype(np.float64)
        x, rho, z_init, z_prop, u, init4 = map(f32, (x, rho, z_init, z_prop, u, init4))
    ref = batched.step(_oracle(name, dtype), x, rho, z_init, z_prop, u, ofit, init4=init4, xw=(kfit.x, kfit.w))
    em, es, ez, er = rel_errors(gpu, ref, family)
    worst = np.maximum.reduce([em, es, ez])
    if dtype == F32:            # the bar of the built-in logistic regression's fp32 replay (tests/test_gpu_glm.py)
        assert np.median(worst) <= 1e-5 and (worst <= 1e-2).mean() >= 0.99
        assert (gpu["accept"] != ref["accept"]).mean() <= 0.01
        return
    if family == "gauss":
        assert worst.max() <= 1e-10 and er.max() <= 1e-10
        assert np.allclose(gpu["theta"], ref["theta"], rtol=1e-10, atol=1e-10)
    else:
        assert (worst[ref["converged"]] <= 1e-10).mean() >= 0.99
    assert np.array_equal(gpu["accept"], ref["accept"])


def test_free_running_matches_oracle_on_emitted_variates():
    """ARMA(1,1) restated, chain kernel: the free-running draws replayed through the oracle on the variates they
    emitted (fit, accept flags, evaluation counts, state)."""
    B, S, seed = 1000, 4, 11
    model = _user("arma")
    kfit, ofit = fit_pair("gauss")
    assert_kernel(model, kfit, F64, "chain_serial")
    x0, _ = _states("arma", B, 12)
    th = up(x0)
    tr = kb.Trace(S, B, model.dim(), kfit.n_eta, F64, device(), variates=True, rho=True)
    acc = torch.zeros(B, dtype=torch.int64, device=device())
    kb.run(model, kfit, th, S, seed, trace=tr, accept_count=acc)
    torch.cuda.synchronize()
    om, theta = _oracle("arma"), x0.copy()
    g = lambda t, s: t[s].double().cpu().numpy()
    for s in range(S):
        ref = batched.step(om, theta, g(tr.rho, s), g(tr.z_init, s), g(tr.z_prop, s), g(tr.u, s), ofit)
        eta = g(tr.eta, s)
        sc = np.exp(np.clip(ref["eta"][:, 1], -300, 300))
        worst = np.maximum(np.abs(eta[:, 0] - ref["eta"][:, 0]) / np.maximum(sc, np.abs(ref["eta"][:, 0])),
                           np.abs(eta[:, 1:] - ref["eta"][:, 1:]).max(1))
        assert worst.max() <= 1e-10
        assert np.array_equal(tr.accept[s].cpu().numpy().astype(bool), ref["accept"])
        assert np.array_equal(tr.evals[s].cpu().numpy(), ref["evals"])
        theta = ref["theta"]
    assert np.allclose(th.cpu().numpy(), theta, rtol=1e-10, atol=1e-10)
    assert np.array_equal(acc.cpu().numpy(), tr.accept.long().sum(0).cpu().numpy())


# ------------------------------------------------------------------ posteriors
def _z(summ, mean, var):
    zm = np.abs(summ["mean"].cpu().numpy() - mean) / summ["mcse_mean"].cpu().numpy()
    zv = np.abs(summ["var"].cpu().numpy() - var) / summ["mcse_var"].cpu().numpy()
    return zm, zv


def _check(s1, s2, n, mean, var, what):
    zm, zv = _z(chain_summary(s1, s2, n), mean, var)
    print(f"{what}: worst z mean {zm.max():.2f}, var {zv.max():.2f}")
    assert zm.max() < 4 and zv.max() < 4, (zm, zv)


@pytest.mark.parametrize("cls", ["KLHR", "KLHRSINH", "Slice", "MH"])
def test_trio_k1_posterior_within_4_mcse(cls):
    """trio, K = 1 (D = 3: the sinh family's exact gradient clip is on), 8192 chains, against digamma / trigamma."""
    model, om = _trio(1)
    mean, var = om.moments()
    if cls == "MH":
        s = kb.MH(model, 0.9, seed=41, chains=8192)
        s.run(4000)
        s1, s2 = s.run(8000, chain_stats=True)
        return _check(s1, s2, 8000, mean, var, "trio K=1 MH")
    s = kb.Slice(model, seed=42, chains=8192, warmup=500) if cls == "Slice" else \
        getattr(kb, cls)(model, seed=43, chains=8192, warmup=1000)
    s.run(1000)
    s1, s2 = s.run(2000, chain_stats=True)
    _check(s1, s2, 2000, mean, var, f"trio K=1 {cls}")


def test_trio_k18_klhr_posterior_within_4_mcse():
    model, om = _trio(18)
    mean, var = om.moments()
    s = kb.KLHR(model, seed=44, chains=8192, warmup=1000)
    s.run(1000)
    s1, s2 = s.run(2000, chain_stats=True)
    _check(s1, s2, 2000, mean, var, "trio K=18 KLHR")


@pytest.mark.parametrize("name", ["es_nc", "logit", "arma"])
def test_restated_klhr_posterior_within_4_mcse_of_exact_truth(name):
    if name == "es_nc":
        mean, var = hier_truth.posterior_moments(EIGHT_SCHOOLS_DATA["y"], EIGHT_SCHOOLS_DATA["sigma"])["noncentered"]
    elif name == "logit":
        mean, var = glm_truth.posterior_moments(_oracle(name))
    else:
        mean, var = ts_truth.posterior_moments(_oracle(name))
    s = kb.KLHR(_user(name), seed=45, chains=8192, warmup=1000)
    s.run(1000)
    s1, s2 = s.run(2000, chain_stats=True)
    _check(s1, s2, 2000, mean, var, f"{name} KLHR")


def test_readme_example_samples():
    data = {"nu": 5.0, "a": 3.0, "b": 2.0, "alpha": 2.0, "beta": 3.0}
    model = kb.CudaModel(TARGETS / "readme_example.cuh", data, dim=3, device=device())
    draws = kb.KLHR(model, chains=16_384).sample(100)
    assert tuple(draws.shape) == (100, 16_384, 3) and bool(torch.isfinite(draws).all())


# ------------------------------------------------------------------ two user targets, refusals
def test_two_user_targets_in_one_process():
    x = np.random.default_rng(9).normal(size=(64, 3)) * 0.5
    trio, _ = _trio(1)
    alone = trio.log_density_gradient(up(x))
    probe = kb.CudaModel(TARGETS / "probe.cuh", {"w": np.ones(PROBE_DIM)}, PROBE_DIM, device=device())
    assert probe._host["i0"] != trio._host["i0"]
    pl = probe.log_density(up(np.tile(PROBE_BASE, (4, 1)))).cpu().numpy()
    expect = sum(probe_jet(k, PROBE_BASE[k:k + 1])[0][0] for k in range(PROBE_DIM))
    assert np.allclose(pl, expect, rtol=1e-14)
    again = trio.log_density_gradient(up(x))
    assert all(torch.equal(a, b) for a, b in zip(alone, again))


def test_abi_refuses_bad_user_descriptors():
    lib = _lib.load()
    trio, _ = _trio(1)
    good = trio.descriptor()
    th = up(np.zeros((4, 3)))
    lp = torch.empty(4, dtype=F64, device=device())
    cases = [(dict(i0=60), -5, "registered slot"), (dict(dim=0), -3, "dim"), (dict(data1=None), -5, "data1"),
             (dict(data0=None), -5, "data0")]
    for kw, code, msg in cases:
        md = _lib.ModelDesc(**{f: getattr(good, f) for f, _ in _lib.ModelDesc._fields_})
        for k, v in kw.items():
            setattr(md, k, v)
        assert lib.klhr_model_eval(C.byref(md), _lib.KLHR_F64, th.data_ptr(), lp.data_ptr(), None, 4, None) == code
        assert msg in _lib.last_error()
    assert lib.klhr_model_eval(C.byref(good), _lib.KLHR_F64, th.data_ptr(), lp.data_ptr(), None, 4, None) == 0
    torch.cuda.synchronize()
    _, om = _trio(1)
    assert np.allclose(lp.cpu().numpy(), om.lp(np.zeros((4, 3))), rtol=1e-14)
