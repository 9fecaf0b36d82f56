"""Logistic regression on the GPU: model evaluation and the KL objective against the oracle, step replay and
free-running parity on the chain kernel (both D-phases) and the octet kernel, and the posterior against its exact
truth (oracle/glm_truth.py: tensor-product rule, < 1e-9) within 4 MCSE per coordinate, with no added slack."""
import dataclasses

import numpy as np
import pytest
import torch

import klhr_b200 as kb
from gpu_util import assert_kernel, device, fit_pair, rel_errors, up
from klhr_b200.diagnostics import chain_summary
from oracle import batched
from oracle.glm_models import EMPTY, MODERATE, SEPARATED, WIDE, GLMBSModel, make_glm_model
from oracle.glm_truth import posterior_moments
from oracle.ref_port import GaussLine, SinhLine, gauss_hermite_probabilists

pytestmark = pytest.mark.gpu

LR = "logistic_regression"
F64, F32 = torch.float64, torch.float32
EPS32 = float(np.finfo(np.float32).eps)


def _model(data):
    return kb.BSModel(stan_file=f"stan/{LR}.stan", data=data, device=device())


def _oracle(data, dtype=F64):
    """The oracle on the data the device holds: X rounded to fp32 for fp32 launches."""
    if dtype == F32:
        data = dict(data, x=np.asarray(data["x"], dtype=np.float32).astype(np.float64).reshape(data["N"], data["K"]))
    return make_glm_model(LR, data)


def _states(data, B, seed, spread=1.0):
    """Points near the posterior bulk (theta ~ N(0, spread^2 / 4 I)) and unit directions."""
    rng = np.random.default_rng(seed)
    D = data["K"] + 1
    x = rng.normal(size=(B, D)) * 0.5 * spread
    rho = rng.normal(size=(B, D))
    rho /= np.linalg.norm(rho, axis=1, keepdims=True)
    return x, rho


# ------------------------------------------------------------------ evaluation
def test_log_density_gradient_fp64_including_far_tails():
    """fp64 against the oracle to 1e-12 of the summed magnitudes, up to |eta| ~ 700; lp bitwise equal to log_density."""
    B = 512
    om = _oracle(MODERATE)
    x, _ = _states(MODERATE, B, 1)
    eta_max = np.abs(x @ om.X.T).max(1)
    x *= np.geomspace(1e-2, 700.0, B)[:, None] / eta_max[:, None]      # largest |eta| of row c: 0.01 .. 700
    model = _model(MODERATE)
    lp, g = (t.cpu().numpy() for t in model.log_density_gradient(up(x)))
    lp2 = model.log_density(up(x)).cpu().numpy()
    lr, gr = om.lp_grad(x)
    assert np.isfinite(lp).all() and np.array_equal(lp, lp2)
    sc = om.terms_scale(x)
    assert np.all(np.abs(lp - lr) <= 1e-12 * sc), np.max(np.abs(lp - lr) / sc)
    gs = (np.abs(om.X).sum(0) + np.abs(x) / 6.25).max() * np.maximum(1.0, np.abs(gr).max(1, keepdims=True))
    assert np.all(np.abs(g - gr) <= 1e-12 * gs)


def test_log_density_gradient_fp32_and_range():
    """fp32 within the recursive-summation bound 4 N eps32 sum |terms| (N = 200); past the fp32 range of eta the
    (-inf, 0) rule, never NaN."""
    B = 1024
    om = _oracle(MODERATE, F32)
    x, _ = _states(MODERATE, B, 2, spread=4.0)
    x32 = x.astype(np.float32).astype(np.float64)
    model = _model(MODERATE)
    lp, g = (t.double().cpu().numpy() for t in model.log_density_gradient(up(x32, F32)))
    lp2 = model.log_density(up(x32, F32)).double().cpu().numpy()
    assert np.array_equal(lp, lp2)
    lr, gr = om.lp_grad(x32)
    N = MODERATE["N"]
    bound = 4 * N * EPS32 * om.terms_scale(x32)
    assert np.all(np.abs(lp - lr) <= bound), np.max(np.abs(lp - lr) / bound)
    # gradient: sum_i x_ik (y_i - sigma_i), sigma off by at most |d eta| / 4 with |d eta| <= D eps |x_i| |theta|
    ax = np.abs(om.X)
    deta = (om.dim() + 2) * EPS32 * (np.abs(x32) @ ax.T)                 # (B, N)
    gbound = 4 * N * EPS32 * (ax.sum(0) + np.abs(x32) / 6.25) + 0.25 * deta @ ax
    assert np.all(np.abs(g - gr) <= gbound + 4 * N * EPS32 * np.abs(gr)), np.max(np.abs(g - gr) / gbound)
    big = x32 * 1e37                                                      # |eta| overflows fp32 somewhere
    lp, g = (t.cpu().numpy() for t in model.log_density_gradient(up(big, F32)))
    assert not np.isnan(lp).any() and not np.isnan(g).any()
    bad = ~np.isfinite(lp)
    assert bad.any() and np.all(lp[bad] == -np.inf) and np.all(g[bad] == 0) and np.isfinite(g).all()


# ------------------------------------------------------------------ KL objective
@pytest.mark.parametrize("family", ["gauss", "sinh"])
@pytest.mark.parametrize("data", [MODERATE, SEPARATED], ids=["moderate", "separated"])
def test_kl_eval_matches_port_of_reference(data, family):
    B = 48
    model = _model(data)
    om = GLMBSModel(LR, data)
    x, rho = _states(data, B, 3)
    rng = np.random.default_rng(4)
    eta = rng.normal(size=(B, 2 if family == "gauss" else 4)) * 0.3
    kfit, _ = fit_pair(family)
    f, g, H = (t.cpu().numpy() for t in kb.kl_eval(model, kfit, up(x), up(rho), up(eta), hessian=True))
    xq, wq = gauss_hermite_probabilists(8)
    line = GaussLine(xq, wq, 1e-12, 600.0) if family == "gauss" else SinhLine(xq, wq, 1e-10, 300.0)
    for c in range(B):
        fr, gr = line.kl(eta[c], x[c], rho[c], om)
        scale = max(1.0, abs(fr))
        assert abs(f[c] - fr) <= 1e-10 * scale, (c, f[c], fr)
        assert np.allclose(g[c], gr, rtol=1e-10, atol=1e-10 * scale), (c, g[c], gr)
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
REPLAY = [(fam, "moderate", F64, kern) for fam in ("gauss", "sinh") for kern in ("chain_serial", "octet")]
REPLAY += [("gauss", "moderate", F32, kern) for kern in ("chain_serial", "octet")]
REPLAY += [("gauss", "wide", F64, kern) for kern in ("chain_octet", "octet")]
REPLAY += [("gauss", "wide", F32, "chain_octet")]
DATA = {"moderate": MODERATE, "separated": SEPARATED, "wide": WIDE}


@pytest.mark.parametrize("family,dname,dtype,kernel", REPLAY,
                         ids=[f"{r[0]}-{r[1]}-{str(r[2])[-7:]}-{r[3]}" for r in REPLAY])
def test_step_replay_matches_oracle(family, dname, dtype, kernel):
    data = DATA[dname]
    B = 2000 if dname == "moderate" else 256
    x, rho = _states(data, B, 5)
    rng = np.random.default_rng(6)
    z_init, z_prop, u = rng.normal(size=B), rng.normal(size=B), rng.random(B)
    init4 = rng.normal(size=(B, 4)) if family == "sinh" else None
    model = _model(data)
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
    if dtype == F32:       # the oracle sees the same rounded inputs
        f32 = lambda a: None if a is None else np.asarray(a, dtype=np.float32).astype(np.float64)
        x, rho, z_init, z_prop, u, init4 = map(f32, (x, rho, z_init, z_prop, u, init4))
    ref = batched.step(_oracle(data, dtype), x, rho, z_init, z_prop, u, ofit, init4=init4, xw=(kfit.x, kfit.w))
    em, es, ez, er = rel_errors(gpu, ref, family)
    worst = np.maximum.reduce([em, es, ez])
    if dtype == F32:
        # l(t) - l(0) is a difference of two fp32 sums over N terms (error ~ N eps32 sum |terms|): most fits agree to
        # ~1e-7, a tail of sharp lines (many observations, points away from the bulk) only to ~1e-3 of the scale
        assert np.median(worst) <= 1e-5 and (worst <= 1e-2).mean() >= 0.99
        assert (worst <= 1e-4).mean() >= (0.95 if dname == "moderate" else 0.5)
        assert (gpu["accept"] != ref["accept"]).mean() <= 0.01
        return
    if family == "gauss":
        assert worst.max() <= 1e-10 and er.max() <= 1e-10
        assert np.allclose(gpu["theta"], ref["theta"], rtol=1e-10, atol=1e-10)
        assert np.array_equal(gpu["evals"], ref["evals"])
    else:
        conv = ref["converged"]
        assert (worst[conv] <= 1e-10).mean() >= 0.99
    assert np.array_equal(gpu["accept"], ref["accept"])


# ------------------------------------------------------------------ free running
@pytest.mark.parametrize("force_octet", [False, True])
@pytest.mark.parametrize("family", ["gauss", "sinh"])
def test_free_running_matches_oracle_on_emitted_variates(family, force_octet):
    """Draws of the free-running kernel replayed through the oracle on the variates it emitted: fit, flags, state,
    per-draw evaluation counts, and accept_count / evals_total as sums of the per-draw values."""
    B, S, seed = 1000, 4, 11
    model = _model(MODERATE)
    kfit, ofit = fit_pair(family)
    kfit.force_octet = force_octet
    assert_kernel(model, kfit, F64, "octet" if force_octet else "chain_serial")
    x0, _ = _states(MODERATE, B, 12)
    th = up(x0)
    tr = kb.Trace(S, B, model.dim(), kfit.n_eta, F64, device(), variates=True, rho=True)
    acc = torch.zeros(B, dtype=torch.int64, device=device())
    ev = torch.zeros(1, dtype=torch.int64, device=device())
    kb.run(model, kfit, th, S, seed, trace=tr, accept_count=acc, evals_total=ev)
    torch.cuda.synchronize()
    om = _oracle(MODERATE)
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


POSTERIOR = [("KLHR", "moderate", F64), ("KLHRSINH", "moderate", F64), ("KLHR", "separated", F64),
             ("KLHRSINH", "separated", F64), ("KLHR", "moderate", F32)]


@pytest.mark.parametrize("cls,dname,dtype", POSTERIOR, ids=[f"{p[0]}-{p[1]}-{str(p[2])[-7:]}" for p in POSTERIOR])
def test_posterior_moments_within_4_mcse_of_exact_truth(cls, dname, dtype):
    """8192 chains, 1000 warm-up draws (the default), then 2000 draws summed in-kernel (octet kernel) and 400 rows of
    sample(thin=5) (chain kernel): every coordinate's mean and variance within 4 MCSE of the quadrature truth."""
    data = DATA[dname]
    B, S, M, thin = 8192, 2000, 400, 5
    model = _model(data)
    mean, var = posterior_moments(_oracle(data, dtype))
    s = getattr(kb, cls)(model, seed=21, chains=B, warmup=1000, dtype=dtype)
    s.run(1000)
    assert_kernel(model, s._fit, dtype, "octet", accumulate=True)
    s1, s2 = s.run(S, chain_stats=True)
    zm, zv = _z(chain_summary(s1, s2, S), mean, var)
    assert zm.max() < 4 and zv.max() < 4, (zm, zv)
    assert_kernel(model, s._fit, dtype, "chain_serial")
    r = s.sample(M + 1, thin=thin)[1:].double()
    zm, zv = _z(chain_summary(r.sum(0), (r * r).sum(0), M), mean, var)
    assert zm.max() < 4 and zv.max() < 4, (zm, zv)


def test_slice_and_mh_posterior_means_and_variances_match_truth():
    """Slice (500 warm-up + 1000 draws) and MH (3000 burn-in + 6000 draws at stepsize 0.15), 8192 chains, on MODERATE."""
    B = 8192
    model = _model(MODERATE)
    mean, var = posterior_moments(_oracle(MODERATE))
    sl = kb.Slice(model, seed=31, chains=B, warmup=500)
    sl.run(500)
    s1, s2 = sl.run(1000, chain_stats=True)
    mh = kb.MH(model, 0.15, seed=32, chains=B)
    mh.run(3000)
    m1, m2 = mh.run(6000, chain_stats=True)
    assert 0.1 < mh.acceptance_probability < 0.9
    for summ in (chain_summary(s1, s2, 1000), chain_summary(m1, m2, 6000)):
        zm, zv = _z(summ, mean, var)
        assert zm.max() < 4 and zv.max() < 4, (zm, zv)


@pytest.mark.parametrize("cls", ["KLHR", "KLHRSINH", "SUBKLHRSINH", "Slice", "MH"])
def test_no_observations_samples_the_prior(cls):
    """N = 0: every sampler against N(0, 6.25 I)."""
    B = 8192
    model = _model(EMPTY)
    if cls == "MH":
        s = kb.MH(model, 2.5, seed=41, chains=B)
        s.run(2000)
        s1, s2 = s.run(4000, chain_stats=True)
        n = 4000
    else:
        s = getattr(kb, cls)(model, seed=41, chains=B, warmup=500 if cls == "Slice" else 1000)
        s.run(500 if cls == "Slice" else 1000)
        n = 1000 if cls == "Slice" else 2000
        s1, s2 = s.run(n, chain_stats=True)
    zm, zv = _z(chain_summary(s1, s2, n), np.zeros(3), np.full(3, 6.25))
    assert zm.max() < 4 and zv.max() < 4, (zm, zv)


# ------------------------------------------------------------------ refusals
def test_kernels_refuse_bad_descriptors():
    """The C ABI checks the descriptor itself (built by hand, not through BSModel)."""
    from klhr_b200 import _lib
    import ctypes as Cc
    lib = _lib.load()
    th = up(np.zeros((4, 3)))
    lp = torch.empty(4, dtype=F64, device=device())
    buf = up(np.ones(64))
    cases = [(dict(dim=3, i0=5, i1=2, data0=None), "data0"),
             (dict(dim=3, i0=-1, i1=2, data0=buf.data_ptr()), "N must be >= 0"),
             (dict(dim=3, i0=5, i1=0, data0=buf.data_ptr()), "K must be >= 1"),
             (dict(dim=3, i0=5, i1=3, data0=buf.data_ptr()), "dim must equal")]
    for kw, msg in cases:
        md = _lib.ModelDesc(id=_lib.MODEL_IDS[LR], s0=0.0, s1=0.0, data1=None, **kw)
        assert lib.klhr_model_eval(Cc.byref(md), _lib.KLHR_F64, th.data_ptr(), lp.data_ptr(), None, 4, None) == -5
        assert "logistic regression" in _lib.last_error() and msg in _lib.last_error()
    md = _lib.ModelDesc(id=_lib.MODEL_IDS[LR], dim=3, i0=0, i1=2, s0=0.0, s1=0.0, data0=None, data1=None)
    assert lib.klhr_model_eval(Cc.byref(md), _lib.KLHR_F64, th.data_ptr(), lp.data_ptr(), None, 4, None) == 0
    torch.cuda.synchronize()
    assert np.array_equal(lp.cpu().numpy(), np.zeros(4))
