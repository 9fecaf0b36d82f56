"""Eight schools, non-centered and centered, on the GPU: model evaluation and the KL objective against the oracle,
step replay and free-running parity on the chain and octet kernels, and the posterior against its exact truth
(oracle/hier_truth.py: 1-D quadrature, ~1e-10) within 4 MCSE per coordinate, with no added slack."""
import numpy as np
import pytest
import torch

import klhr_b200 as kb
from gpu_util import assert_kernel, device, fit_pair, rel_errors, up
from klhr_b200.diagnostics import chain_summary
from oracle import batched
from oracle.hier_models import EIGHT_SCHOOLS_DATA, HierBSModel, make_hier_model
from oracle.hier_truth import posterior_moments
from oracle.ref_port import GaussLine, SinhLine, gauss_hermite_probabilists

pytestmark = pytest.mark.gpu

NC, C = "eight_schools_noncentered", "eight_schools_centered"
CLASSIC = EIGHT_SCHOOLS_DATA
# sigma / 10: informative data, where the centered form mixes (the classic data give it the neck at small tau)
SHARP = dict(CLASSIC, sigma=[s / 10 for s in CLASSIC["sigma"]])
_r30 = np.random.default_rng(30)
J30 = {"J": 30, "y": (_r30.normal(size=30) * 10).tolist(), "sigma": (5 + 15 * _r30.random(30)).tolist()}
F64, F32 = torch.float64, torch.float32


def _model(name, data=CLASSIC):
    return kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())


def _u_index(name, J):
    return J + 1 if name == NC else 1


def _states(name, data, B, seed, u=None, spread=1.0):
    """Points near the posterior's bulk: theta_trans ~ N(0, 1), mu ~ N(4, 9), theta ~ N(y, sigma), log tau ~ N(1, 1)."""
    J = data["J"]
    rng = np.random.default_rng(seed)
    x = np.empty((B, J + 2))
    if name == NC:
        x[:, :J] = rng.normal(size=(B, J)) * spread
        x[:, J] = 4 + 3 * spread * rng.normal(size=B)
    else:
        x[:, 0] = 4 + 3 * spread * rng.normal(size=B)
        x[:, 2:] = np.asarray(data["y"]) + np.asarray(data["sigma"]) * spread * rng.normal(size=(B, J))
    k = _u_index(name, J)
    x[:, k] = 1 + spread * rng.normal(size=B) if u is None else u
    rho = rng.normal(size=(B, J + 2))
    rho /= np.linalg.norm(rho, axis=1, keepdims=True)
    return x, rho


# ------------------------------------------------------------------ evaluation
@pytest.mark.parametrize("name", [NC, C])
def test_log_density_gradient_fp64_including_far_tails(name):
    B = 512
    x, _ = _states(name, CLASSIC, B, 1)
    k = _u_index(name, 8)
    x[:, k] = np.linspace(-300, 300, B)
    model = _model(name)
    om = make_hier_model(name, CLASSIC)
    lp, g = model.log_density_gradient(up(x))
    lp2 = model.log_density(up(x))
    lp, g, lp2 = lp.cpu().numpy(), g.cpu().numpy(), lp2.cpu().numpy()
    lr, gr = om.lp_grad(x)
    ok = np.isfinite(lr) & np.isfinite(gr).all(1)
    assert ok.all()                      # fp64: finite everywhere on |u| <= 300, both forms
    assert np.array_equal(lp, lp2)
    assert np.all(np.abs(lp - lr) <= 1e-12 * np.maximum(np.abs(lr), 1.0))
    sg = np.abs(gr).max(1, keepdims=True)
    assert np.all(np.abs(g - gr) <= 1e-12 * sg)


@pytest.mark.parametrize("name", [NC, C])
def test_log_density_gradient_fp32(name):
    B = 1024
    x, _ = _states(name, CLASSIC, B, 2)
    k = _u_index(name, 8)
    x[:, k] = np.linspace(-20, 20, B)
    x32 = x.astype(np.float32).astype(np.float64)
    model = _model(name)
    om = make_hier_model(name, CLASSIC)
    lp, g = model.log_density_gradient(up(x32, F32))
    lp, g = lp.double().cpu().numpy(), g.double().cpu().numpy()
    lr, gr = om.lp_grad(x32)
    # scale of the terms that are summed: |lp| bounds them from below only after cancellation, so use the
    # term magnitudes of the likelihood and prior (all negative except u and (1 - J) u)
    sc = np.abs(lr) + 10 * np.abs(x32[:, k]) + 1
    assert np.all(np.abs(lp - lr) <= 1e-5 * sc), np.max(np.abs(lp - lr) / sc)
    sg = np.abs(gr).max(1, keepdims=True) + 1
    assert np.all(np.abs(g - gr) <= 1e-5 * sg), np.max(np.abs(g - gr) / sg)
    # beyond |u| = 20 the fp32 exponentials leave their range somewhere: the (-inf, 0) rule, never NaN
    x[:, k] = np.concatenate([np.linspace(-300, -20, B // 2), np.linspace(20, 300, B - B // 2)])
    lp, g = model.log_density_gradient(up(x, F32))
    lp, g = lp.cpu().numpy(), g.cpu().numpy()
    assert not np.isnan(lp).any() and not np.isnan(g).any()
    bad = ~np.isfinite(lp)
    assert np.all(lp[bad] == -np.inf) and np.all(g[bad] == 0) and np.isfinite(g).all()
    assert bad.any()


# ------------------------------------------------------------------ KL objective
@pytest.mark.parametrize("family", ["gauss", "sinh"])
@pytest.mark.parametrize("name", [NC, C])
def test_kl_eval_matches_port_of_reference(name, family):
    B = 64
    model = _model(name)
    om = HierBSModel(name, CLASSIC)
    x, rho = _states(name, CLASSIC, B, 3)
    rng = np.random.default_rng(4)
    eta = rng.normal(size=(B, 2 if family == "gauss" else 4)) * 0.3
    kfit, _ = fit_pair(family)
    f, g, H = kb.kl_eval(model, kfit, up(x), up(rho), up(eta), hessian=True)
    f, g, H = f.cpu().numpy(), g.cpu().numpy(), H.cpu().numpy()
    xq, wq = gauss_hermite_probabilists(8)
    line = GaussLine(xq, wq, 1e-12, 600.0) if family == "gauss" else SinhLine(xq, wq, 1e-10, 300.0)
    for c in range(B):
        fr, gr = line.kl(eta[c], x[c], rho[c], om)
        scale = max(1.0, abs(fr))
        assert abs(f[c] - fr) <= 1e-10 * scale, (c, f[c], fr)
        assert np.allclose(g[c], gr, rtol=1e-9, atol=1e-9 * scale), (c, g[c], gr)
    # Hessian against differences of the device gradient, with the clip off
    import dataclasses
    kfit = dataclasses.replace(kfit, grad_clip=0.0)
    f, g, H = (t.cpu().numpy() for t in kb.kl_eval(model, kfit, up(x), up(rho), up(eta), hessian=True))
    h = 1e-5
    for k in range(eta.shape[1]):
        ep, em = eta.copy(), eta.copy()
        ep[:, k] += h
        em[:, k] -= h
        gp = kb.kl_eval(model, kfit, up(x), up(rho), up(ep))[1].cpu().numpy()
        gm = kb.kl_eval(model, kfit, up(x), up(rho), up(em))[1].cpu().numpy()
        assert np.allclose((gp - gm) / (2 * h), H[:, :, k], rtol=2e-5, atol=1e-5 * (1 + np.abs(f))[:, None]), k


# ------------------------------------------------------------------ replay
REPLAY = [(n, fam, data, dtype, kern) for n in (NC, C) for fam in ("gauss", "sinh") for kern in ("chain_serial", "octet")
          for data, dtype in ((CLASSIC, F64),)]
REPLAY += [(n, "gauss", CLASSIC, F32, kern) for n in (NC, C) for kern in ("chain_serial", "octet")]
REPLAY += [(n, "gauss", J30, F64, kern) for n in (NC, C) for kern in ("chain_octet", "octet")]
REPLAY += [(n, "gauss", J30, F32, "chain_octet") for n in (NC, C)]


def _replay_both(name, data, family, theta, rho, z_init, z_prop, u, init4, dtype, force_octet):
    """The CUDA replay step and the batched oracle on the same inputs (gpu_util.replay_both for these models)."""
    kfit, ofit = fit_pair(family, dtype)
    kfit.force_octet = force_octet
    th = up(theta, dtype)
    tr = kb.step_replay(_model(name, data), kfit, th, up(rho, dtype), up(z_init, dtype), up(z_prop, dtype),
                        up(u, dtype), init4=up(init4, dtype) if init4 is not None else None)
    torch.cuda.synchronize()
    gpu = dict(eta=tr.eta[0].double().cpu().numpy(), zp=tr.zp[0].double().cpu().numpy(),
               r=tr.r[0].double().cpu().numpy(), accept=tr.accept[0].cpu().numpy().astype(bool),
               evals=tr.evals[0].cpu().numpy(), theta=th.double().cpu().numpy())
    if dtype == F32:       # the oracle sees the same rounded inputs
        f32 = lambda a: None if a is None else np.asarray(a, dtype=np.float32).astype(np.float64)
        theta, rho, z_init, z_prop, u, init4 = map(f32, (theta, rho, z_init, z_prop, u, init4))
    ref = batched.step(make_hier_model(name, data), theta, rho, z_init, z_prop, u, ofit, init4=init4,
                       xw=(kfit.x, kfit.w))
    return gpu, ref


@pytest.mark.parametrize("name,family,data,dtype,kernel", REPLAY,
                         ids=[f"{r[0][14:]}-{r[1]}-J{r[2]['J']}-{str(r[3])[-7:]}-{r[4]}" for r in REPLAY])
def test_step_replay_matches_oracle(name, family, data, dtype, kernel):
    B = 2000
    x, rho = _states(name, data, B, 5)
    rng = np.random.default_rng(6)
    z_init, z_prop, u = rng.normal(size=B), rng.normal(size=B), rng.random(B)
    init4 = rng.normal(size=(B, 4)) if family == "sinh" else None
    model = _model(name, data)
    kfit, _ = fit_pair(family, dtype)
    kfit.force_octet = kernel == "octet"
    assert_kernel(model, kfit, dtype, kernel, free_running=False)
    gpu, ref = _replay_both(name, data, family, x, rho, z_init, z_prop, u, init4, dtype, kernel == "octet")
    em, es, ez, er = rel_errors(gpu, ref, family)
    worst = np.maximum.reduce([em, es, ez])
    if dtype == F32:
        assert (worst <= 1e-4).mean() >= 0.995 and worst.max() <= 1e-2
        assert (gpu["accept"] != ref["accept"]).mean() <= 0.002
        return
    if family == "gauss":
        assert worst.max() <= 1e-10 and er.max() <= 1e-10
        assert np.allclose(gpu["theta"], ref["theta"], rtol=1e-10, atol=1e-10)
    else:
        conv = ref["converged"]
        assert (worst[conv] <= 1e-10).mean() >= 0.99 and np.median(worst) <= 1e-13
    assert np.array_equal(gpu["accept"], ref["accept"])
    assert np.array_equal(gpu["evals"], ref["evals"]) or family == "sinh"


# ------------------------------------------------------------------ free running
@pytest.mark.parametrize("force_octet", [False, True])
@pytest.mark.parametrize("family", ["gauss", "sinh"])
@pytest.mark.parametrize("name", [NC, C])
def test_free_running_matches_oracle_on_emitted_variates(name, family, force_octet):
    """Draws of the free-running kernel replayed through the oracle on the variates it emitted: fit, flags, state,
    per-draw evaluation counts, and accept_count / evals_total as sums of the per-draw values."""
    B, S, seed = 1000, 4, 11
    model = _model(name)
    kfit, ofit = fit_pair(family)
    kfit.force_octet = force_octet
    assert_kernel(model, kfit, F64, "octet" if force_octet else "chain_serial")
    x0, _ = _states(name, CLASSIC, B, 12)
    th = up(x0)
    tr = kb.Trace(S, B, model.dim(), kfit.n_eta, F64, device(), variates=True, rho=True)
    acc = torch.zeros(B, dtype=torch.int64, device=device())
    ev = torch.zeros(1, dtype=torch.int64, device=device())          # evals_total: one counter for the launch
    kb.run(model, kfit, th, S, seed, trace=tr, accept_count=acc, evals_total=ev)
    torch.cuda.synchronize()
    om = make_hier_model(name, CLASSIC)
    theta = x0.copy()
    g = lambda t, s: t[s].double().cpu().numpy()
    for s in range(S):
        ref = batched.step(om, theta, g(tr.rho, s), g(tr.z_init, s), g(tr.z_prop, s), g(tr.u, s), ofit,
                           init4=g(tr.init4, s) if tr.init4 is not None else None)
        eta = g(tr.eta, s)
        sc = np.exp(np.clip(ref["eta"][:, 1], -300, 300))
        worst = np.maximum(np.abs(eta[:, 0] - ref["eta"][:, 0]) / np.maximum(sc, np.abs(ref["eta"][:, 0])),
                           np.abs(eta[:, 1:] - ref["eta"][:, 1:]).max(1))
        flags = tr.accept[s].cpu().numpy().astype(bool)
        evals = tr.evals[s].cpu().numpy()
        if family == "gauss":
            assert worst.max() <= 1e-10
            assert np.array_equal(flags, ref["accept"]) and np.array_equal(evals, ref["evals"])
            theta = ref["theta"]
        else:
            conv = ref["converged"]
            assert (worst[conv] <= 1e-10).mean() >= 0.98
            assert (evals[conv] == ref["evals"][conv]).mean() >= 0.98
            theta = np.where(flags[:, None], theta + g(tr.zp, s)[:, None] * g(tr.rho, s), theta)
    if family == "gauss":
        assert np.allclose(th.cpu().numpy(), theta, rtol=1e-10, atol=1e-10)
    assert np.array_equal(acc.cpu().numpy(), tr.accept.long().sum(0).cpu().numpy())
    assert int(ev.item()) == int(tr.evals.long().sum())


# ------------------------------------------------------------------ posterior against the exact truth
def _z(summ, mean, var):
    zm = np.abs(summ["mean"].cpu().numpy() - mean) / summ["mcse_mean"].cpu().numpy()
    zv = np.abs(summ["var"].cpu().numpy() - var) / summ["mcse_var"].cpu().numpy()
    return zm, zv


def _rows_summary(rows):
    """chain_summary of stored rows (M, B, D) via their per-chain sums."""
    r = rows.double()
    return chain_summary(r.sum(0), (r * r).sum(0), r.shape[0])


POSTERIOR = [(NC, "KLHR", CLASSIC), (NC, "KLHRSINH", CLASSIC), (C, "KLHR", SHARP), (C, "KLHRSINH", SHARP)]


@pytest.mark.parametrize("name,cls,data", POSTERIOR, ids=[f"{p[0][14:]}-{p[1]}" for p in POSTERIOR])
def test_posterior_moments_within_4_mcse_of_exact_truth(name, cls, data):
    """8192 chains, 1000 warm-up draws (the default), then 2000 draws summed in-kernel by run(chain_stats=True)
    (octet kernel) and 400 rows of sample(thin=5) (chain kernel).  Every coordinate's mean and variance must be
    within 4 MCSE of the quadrature truth."""
    B, S, M, thin = 8192, 2000, 400, 5
    model = _model(name, data)
    mean, var = posterior_moments(data["y"], data["sigma"])["noncentered" if name == NC else "centered"]
    s = getattr(kb, cls)(model, seed=21, chains=B, warmup=1000)
    s.run(1000)                                                    # the warm-up
    assert_kernel(model, s._fit, F64, "octet", accumulate=True)
    s1, s2 = s.run(S, chain_stats=True)
    zm, zv = _z(chain_summary(s1, s2, S), mean, var)
    assert zm.max() < 4 and zv.max() < 4, (zm, zv)
    assert_kernel(model, s._fit, F64, "chain_serial")
    rows = s.sample(M + 1, thin=thin)[1:]
    zm, zv = _z(_rows_summary(rows), mean, var)
    assert zm.max() < 4 and zv.max() < 4, (zm, zv)


@pytest.mark.parametrize("name", [NC, C])
def test_slice_and_mh_run_and_slice_mh_means_match_truth(name):
    """Slice and MH on both targets; on the non-centered one their posterior means are within 4 MCSE of the truth
    (8192 chains; Slice 500 warm-up + 1000 draws, MH 3000 burn-in + 6000 draws at stepsize 0.4)."""
    B = 8192
    model = _model(name)
    mean, _ = posterior_moments(CLASSIC["y"], CLASSIC["sigma"])["noncentered" if name == NC else "centered"]
    sl = kb.Slice(model, seed=31, chains=B, warmup=500)
    sl.run(500)
    s1, s2 = sl.run(1000, chain_stats=True)
    summ_s = chain_summary(s1, s2, 1000)
    mh = kb.MH(model, 0.4, seed=32, chains=B)
    mh.run(3000)
    s1, s2 = mh.run(6000, chain_stats=True)
    summ_m = chain_summary(s1, s2, 6000)
    for summ in (summ_s, summ_m):
        assert bool(torch.isfinite(summ["mean"]).all() and torch.isfinite(summ["var"]).all())
    assert 0.05 < mh.acceptance_probability < 0.95
    if name == NC:
        for summ in (summ_s, summ_m):
            zm = np.abs(summ["mean"].cpu().numpy() - mean) / summ["mcse_mean"].cpu().numpy()
            assert zm.max() < 4, zm


def test_kernels_refuse_bad_descriptors():
    """The C ABI checks the data block itself (a descriptor built by hand, not through BSModel)."""
    from klhr_b200 import _lib
    import ctypes as Cc
    lib = _lib.load()
    th = up(np.zeros((4, 10)))
    lp = torch.empty(4, dtype=F64, device=device())
    buf = up(np.ones(16))
    for kw in (dict(dim=10, i0=8, data0=None), dict(dim=11, i0=8, data0=buf.data_ptr()),
               dict(dim=2, i0=0, data0=buf.data_ptr())):
        for mid in (8, 9):
            md = _lib.ModelDesc(id=mid, i1=0, s0=0.0, s1=0.0, data1=None, **kw)
            assert lib.klhr_model_eval(Cc.byref(md), _lib.KLHR_F64, th.data_ptr(), lp.data_ptr(), None, 4, None) == -5
            assert "eight schools" in _lib.last_error()
