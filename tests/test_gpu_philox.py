"""The in-kernel Philox4x32-10 streams: known-answer vectors (Random123) through the C ABI, and every variate the
kernels emit -- direction, z_init, z_prop, u, the sinh start values, the over-relaxation pair (r, v), the Slice
scalars and shrinkage uniforms, the MH accept uniform and proposal normals -- re-derived on the CPU from
(seed, chain, draw) by oracle/philox.py, with 64-bit chain ids and draw indices past 2^32.  The replay tests take
these variates as given; here they are held to their definition.

Tolerances: uniforms bitwise; fp64 z_prop and the Slice exponential 1e-13; values of the fp32 approximate units
(z_init, fp32 z_prop, the sinh start values) 5e-6 absolute; direction and MH normals the same plus a term for
radii near 0 (_normal_tol), unit directions 2e-6 plus the normals' error through x."""
import numpy as np
import pytest
import scipy.special as sp
import torch

import klhr_b200 as kb
from gpu_util import assert_kernel, device, fit_pair, up
from oracle import philox as P, stan_models

pytestmark = pytest.mark.gpu
F64, F32 = torch.float64, torch.float32
NP = {F64: np.float64, F32: np.float32}
SEED = 0x1234_5678_9ABC_DEF0
CHAIN_OFFSET, DRAW_OFFSET = (1 << 33) + 5, (1 << 32) + 7


def _device_blocks(rows):
    lib = kb._lib.load()
    inp = torch.as_tensor(np.asarray(rows, dtype=np.int64), device=device()).to(torch.int32).contiguous()
    out = torch.zeros(len(rows), 4, dtype=torch.int32, device=device())
    rc = lib.klhr_philox_eval(inp.data_ptr(), out.data_ptr(), len(rows), None)
    assert rc == 0
    torch.cuda.synchronize()
    return out.cpu().numpy().view(np.uint32)


def test_known_answer_vectors_on_device():
    rows = [list(c) + list(k) for c, k, _ in P.KAT]
    rows = [[(v - (1 << 32)) if v >= (1 << 31) else v for v in r] for r in rows]       # as int32 bit patterns
    got = _device_blocks(rows)
    for g, (_, _, out) in zip(got, P.KAT):
        assert tuple(int(x) for x in g) == out
    rng = np.random.default_rng(0)
    rnd = rng.integers(0, 1 << 32, size=(5000, 6), dtype=np.uint64)
    dev = _device_blocks(rnd.astype(np.int64).astype(np.uint32).view(np.int32).astype(np.int64))
    ref = np.stack(P.philox4x32_10(*(rnd[:, k] for k in range(6))), axis=1)
    assert np.array_equal(dev.astype(np.uint64), ref)


def _direction_law(D, dtype):
    """Two stored mean columns, one zero column, non-unit sd; returns (Direction, cols, sd, cdf)."""
    sd = np.linspace(0.5, 2.0, D)
    cols = np.zeros((2, D))
    cols[0, 1], cols[1, D // 2] = 3.0, -2.0
    cdf = np.array([0.3, 0.8, 1.0])
    return kb.Direction(mean_cols=up(cols, dtype), sd=up(sd, dtype), cdf=up(cdf, dtype), n_zero_cols=1), cols, sd, cdf


def _normal_tol(z):
    """Error bound of a normal of the fp32 Box-Muller (approximate units) against exact arithmetic: ~1e-6 relative
    to the radius from the angle's rounding and __cosf / __sinf, plus lg2.approx's ~2^-22 absolute error on log2 u,
    which the square root turns into ~1.4 2^-22 / (2 radius) <= 2e-7 / |z| -- large only for a radius near 0."""
    with np.errstate(divide="ignore"):
        return 1e-6 * np.maximum(1.0, np.abs(z)) + 2e-7 / np.abs(z)


def _expected_rho(seed, chains, draw, D, cols, sd, cdf, u_col, tol):
    """rho = x / ||x + tol||, x = mean_j + sd z formed in fp32, j = searchsorted(cdf, u_col, 'right'); and the bound
    per chain: 2e-6, plus the normals' error (_normal_tol) through x, relative to ||x||."""
    z = P.direction_normals(seed, chains, draw, D)
    j = np.searchsorted(cdf.astype(np.float32), u_col.astype(np.float32), side="right")
    mean = np.where((j < 2)[:, None], cols[np.minimum(j, 1)], 0.0)
    x = mean.astype(np.float32) + sd.astype(np.float32) * z
    nx = np.linalg.norm(x + tol, axis=1, keepdims=True)
    return x / nx, z, 2e-6 + 2 * np.linalg.norm(sd * _normal_tol(z), axis=1, keepdims=True) / nx


# (id, model, data, family, force, dtype, kernel, draws rows).  corr-normal D = 128 / 256 runs on the warp-specialised
# dense kernel, and with draws rows on the plain dense kernel (klhr_densek.cu; launch_info has no draws argument, so
# the plain kernel's plan is proven through its replay launch, the plan the rows run on too).
STREAMS = [
    ("lane", "normal", {"D": 100}, "gauss", None, F64, "lane", False),
    ("tile", "normal", {"D": 100}, "gauss", "tile", F64, "tile", False),
    ("octet", "normal", {"D": 100}, "gauss", "octet", F64, "octet", False),
    ("tile-f32", "normal", {"D": 100}, "gauss", None, F32, "tile", False),
    ("octet-f32", "normal", {"D": 100}, "gauss", "octet", F32, "octet", False),
    ("chain-serial", "funnel", {"D": 10}, "gauss", None, F64, "chain_serial", False),
    ("chain-octet", "funnel", {"D": 30}, "gauss", None, F64, "chain_octet", False),
    ("chain-serial-f32", "funnel", {"D": 10}, "gauss", None, F32, "chain_serial", False),
    ("chain-serial-sinh", "funnel", {"D": 1}, "sinh", None, F64, "chain_serial", False),
    ("octet-sinh", "funnel", {"D": 1}, "sinh", "octet", F64, "octet", False),
    ("dense-ws-128", "corr-normal", {"N": 128, "rho": 0.5}, "gauss", None, F64, "dense_ws", False),
    ("dense-ws-256", "corr-normal", {"N": 256, "rho": 0.9}, "gauss", None, F64, "dense_ws", False),
    ("dense-128", "corr-normal", {"N": 128, "rho": 0.5}, "gauss", None, F64, "dense", True),
]


@pytest.mark.parametrize("case", STREAMS, ids=[c[0] for c in STREAMS])
def test_emitted_variates_are_the_documented_function_of_seed_chain_draw(case):
    """u bitwise, z_prop to 1e-13 (fp64) / 5e-6 (fp32), z_init, the sinh start values and the direction to the
    accuracy of the fp32 approximate units -- including the |z| > 4 tail of the direction normals where there are
    enough of them -- for chains with 64-bit ids and a draw index beyond 2^32."""
    cid, name, data, family, force, dtype, kernel, rows = case
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
    D, B, S = model.dim(), 3000, 2
    kfit, _ = fit_pair(family, dtype)
    kfit.force_octet, kfit.force_tile = force == "octet", force == "tile"
    assert_kernel(model, kfit, dtype, kernel, free_running=kernel != "dense")
    direction, cols, sd, cdf = _direction_law(D, dtype)
    th = up(np.zeros((B, D)), dtype)
    tr = kb.Trace(S, B, D, kfit.n_eta, dtype, device(), variates=True, rho=True)
    draws = torch.empty(S, B, D, dtype=dtype, device=device()) if rows else None
    kb.run(model, kfit, th, S, SEED, direction, chain_offset=CHAIN_OFFSET, draw_offset=DRAW_OFFSET, trace=tr,
           draws=draws, thin=1)
    torch.cuda.synchronize()
    chains = CHAIN_OFFSET + np.arange(B)
    g = lambda t, s: t[s].double().cpu().numpy()
    n_tail = 0
    for s in range(S):
        u_col, z_init, z_prop, u = P.chain_scalars(SEED, chains, DRAW_OFFSET + s, NP[dtype])
        assert np.array_equal(g(tr.u, s), u), cid
        zp_tol = 1e-13 if dtype == F64 else 5e-6
        assert np.allclose(g(tr.z_prop, s), z_prop, rtol=zp_tol, atol=zp_tol), cid
        assert np.allclose(g(tr.z_init, s), z_init, rtol=0, atol=5e-6), cid
        if family == "sinh":
            i4 = g(tr.init4, s)
            init2, init3 = P.init4(SEED, chains, DRAW_OFFSET + s)
            assert (i4[:, :2] == 0).all()
            assert np.allclose(i4[:, 2], init2, rtol=0, atol=5e-6) and np.allclose(i4[:, 3], init3, rtol=0, atol=5e-6)
        rho, z, tol = _expected_rho(SEED, chains, DRAW_OFFSET + s, D, cols, sd, cdf, u_col, kfit.tol)
        err = np.abs(g(tr.rho, s) - rho)
        assert (err <= tol).all(), (cid, float(err.max()), float((err / tol).max()))
        n_tail += int((np.abs(z) > 4).sum())
    if B * S * D >= 500_000:
        assert n_tail >= 10          # ~38 expected beyond 4 sigma in 6e5 normals, all reproduced above


@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
def test_slice_and_mh_variates_are_the_documented_function_of_seed_chain_draw(dtype):
    """Slice: the direction, e = -log u53 (1e-13 relative; fp32: the rounding of the fp64 value), u0 and the traced
    shrinkage uniforms (bitwise; NaN past the shrink count).  MH: the accept uniform (bitwise) and the proposal
    normals (the direction map, 5e-6 absolute)."""
    D, B, S, cap = 100, 2000, 2, 16
    model = kb.BSModel(stan_file="stan/ill-normal.stan", data={"D": D}, device=device())
    chains = CHAIN_OFFSET + np.arange(B)
    direction, cols, sd, cdf = _direction_law(D, dtype)
    cfg = kb.SliceConfig(w=0.5, cap=cap)
    th = up(np.random.default_rng(0).normal(size=(B, D)), dtype)
    tr = kb.Trace(S, B, D, 0, dtype, device(), variates=True, rho=True, slice_cap=cap)
    kb.slice_run(model, cfg, th, S, SEED, direction, chain_offset=CHAIN_OFFSET, draw_offset=DRAW_OFFSET, trace=tr)
    m = kb.MH(model, 0.3, seed=SEED, chains=B, dtype=dtype, chain_offset=CHAIN_OFFSET)
    m._draw = DRAW_OFFSET
    tm = kb.Trace(S, B, D, 2, dtype, device(), variates=True, rho=True)
    m._advance(S, trace=tm)
    torch.cuda.synchronize()
    g = lambda t, s: t[s].double().cpu().numpy()
    n_shrunk = 0
    for s in range(S):
        draw = DRAW_OFFSET + s
        u_col, e, u0 = P.slice_scalars(SEED, chains, draw, NP[dtype])
        assert np.allclose(g(tr.z_init, s), e, rtol=1e-13 if dtype == F64 else 2.0 ** -23, atol=0)
        assert np.array_equal(g(tr.u, s), u0)
        rho, _, tol = _expected_rho(SEED, chains, draw, D, cols, sd, cdf, u_col, cfg.tol)
        assert (np.abs(g(tr.rho, s) - rho) <= tol).all()
        su, n = g(tr.slice_u, s), tr.slice_n[s].cpu().numpy()
        assert (n >= 1).all()
        ref = P.slice_shrink_u(SEED, chains, draw, cap, NP[dtype])
        used = np.arange(cap)[None, :] < n[:, None]          # every traced column up to the shrink count
        assert np.array_equal(su[used], ref[used]) and np.isnan(su[~used]).all()
        n_shrunk += int((n > 1).sum())
        assert np.array_equal(g(tm.u, s), P.mh_accept_u(SEED, chains, draw, NP[dtype]))
        z = P.direction_normals(SEED, chains, draw, D)
        err = np.abs(g(tm.rho, s) - z)
        assert (err <= 5e-6 + _normal_tol(z)).all(), float(err.max())
    assert n_shrunk >= 100           # the traced shrinkage uniforms reach past the first block's words


# ---------------------------------------------------------------------------------------------------- over-relaxation
def _u0(eta, family, fp, dtype):
    """CDF of the fitted proposal at the current point, from the traced eta: ndtr(-m / s) for the Gaussian family,
    klhr_sinh.py's _CDF(0) (the clamp of klhr_fit.cuh:fit_and_propose) for sinh."""
    c = fp.scale_clip
    if family == "gauss":
        return sp.ndtr(-eta[:, 0] / np.exp(np.clip(eta[:, 1], -c, c)))
    s = np.exp(np.clip(eta[:, 1], -c, c)) + fp.tol
    d = np.exp(np.clip(eta[:, 2], -c, c)) + fp.tol
    return sp.ndtr(np.sinh(np.clip(d * np.arcsinh(-eta[:, 0] / s) - eta[:, 3], -c, c)))


def _v_bound(K):
    """Relative error of the kernel's v against exact logs: each exponential within 1 ulp (logf / log1pf of an exact
    argument), at most K + 1 of them summed in fp32, one quotient -- (2K + 6) 2^-24 in all, with a factor of 2."""
    return 2 * (2 * K + 6) * 2.0 ** -24


def _check_overrelax(seed, chains, draw, K, family, fp, dtype, r_dev, v_dev, eta):
    """or_r equal to the restatement except on chains with a uniform within the dtype's rounding of u0 (counted,
    returned); or_v to _v_bound(K) of the exact-log restatement on every chain (given the device's r)."""
    u0 = _u0(eta, family, fp, dtype)
    r_ref, _ = P.overrelax(seed, chains, draw, K, u0)
    words = np.stack([w for q in range(-(-K // 4)) for w in P.block(seed, chains, draw, P.SLOT_OVERRELAX + q)],
                     axis=1)[:, :K]
    near = (np.abs(P.u01_32(words) - u0[:, None]) <= (1e-12 if dtype == F64 else 1e-6)).any(axis=1)
    bad = (r_dev != r_ref) & ~near
    assert not bad.any(), (int(bad.sum()), np.flatnonzero(bad)[:5], r_dev[bad][:5], r_ref[bad][:5])
    _, v_ref = P.overrelax(seed, chains, draw, K, None, r=r_dev)
    rel = np.abs(v_dev - v_ref) / v_ref
    assert (v_dev > 0).all() and (v_dev <= 1).all()
    i = int(np.argmax(rel))
    assert rel[i] <= _v_bound(K), (float(rel[i]), i, v_dev[i], v_ref[i], r_dev[i])
    return int(near.sum())


# (id, model, data, family, force, dtype, kernel)
OVERRELAX = [
    ("tile", "ill-normal", {"D": 20}, "gauss", "tile", F64, "tile"),
    ("tile-f32", "ill-normal", {"D": 20}, "gauss", "tile", F32, "tile"),
    ("octet", "ill-normal", {"D": 20}, "gauss", "octet", F64, "octet"),
    ("octet-f32", "ill-normal", {"D": 20}, "gauss", "octet", F32, "octet"),
    ("chain-funnel2", "funnel", {"D": 2}, "gauss", None, F64, "chain_serial"),
    ("chain-funnel1-sinh", "funnel", {"D": 1}, "sinh", None, F64, "chain_serial"),
]


@pytest.mark.parametrize("case", OVERRELAX, ids=[c[0] for c in OVERRELAX])
def test_overrelaxation_pair_equals_the_restatement(case):
    """K = 10 over-relaxation on 4000 chains, two draws: or_r exactly the restated binomial count from the traced
    fit's u0 (chains where a uniform falls within rounding of u0 exempt and counted), or_v within _v_bound(K) of the
    beta variate with exact logs."""
    cid, name, data, family, force, dtype, kernel = case
    K, B, S = 10, 4000, 2
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
    kfit, _ = fit_pair(family, dtype)
    kfit.force_octet, kfit.force_tile = force == "octet", force == "tile"
    kfit.overrelax_K = K
    assert_kernel(model, kfit, dtype, kernel)
    D = model.dim()
    th = up(np.random.default_rng(1).normal(size=(B, D)) * 0.7, dtype)
    tr = kb.Trace(S, B, D, kfit.n_eta, dtype, device(), variates=True, rho=True)
    kb.run(model, kfit, th, S, SEED, chain_offset=CHAIN_OFFSET, draw_offset=DRAW_OFFSET, trace=tr)
    torch.cuda.synchronize()
    chains = CHAIN_OFFSET + np.arange(B)
    r, v, eta = tr.or_r.cpu().numpy().astype(np.int64), tr.or_v.double().cpu().numpy(), tr.eta.double().cpu().numpy()
    n_near = sum(_check_overrelax(SEED, chains, DRAW_OFFSET + s, K, family, kfit, dtype, r[s], v[s], eta[s])
                 for s in range(S))
    assert n_near <= 0.01 * B * S, n_near
    assert len(np.unique(r)) >= 5, cid                    # the fits' u0 spread: many (na, nb) classes are reached


def test_overrelaxation_beta_near_u_equal_1_on_4m_chains():
    """2^22 chains of normal D = 1 at theta = +-8, K = 10: u0 = Phi(+-8) is saturated, so r is 0 or K and v ~ Beta(1,
    10) for every chain, its one Ga term from word 10.  About 64 chains have that word >= 0xFFFF0000, u within 2^-16
    of 1, where an exponential formed as -log u loses its relative accuracy: or_v against exact logs on every chain."""
    K, B = 10, 1 << 22
    model = kb.BSModel(stan_file="stan/normal.stan", data={"D": 1}, device=device())
    kfit, _ = fit_pair("gauss")
    kfit.overrelax_K = K
    assert_kernel(model, kfit, F64, "tile")
    theta = np.where(np.arange(B) % 2 == 0, 8.0, -8.0)[:, None]
    th = up(theta)
    tr = kb.Trace(1, B, 1, 2, F64, device(), variates=True, rho=True)
    kb.run(model, kfit, th, 1, SEED, chain_offset=CHAIN_OFFSET, draw_offset=DRAW_OFFSET, trace=tr)
    torch.cuda.synchronize()
    r, v, eta = tr.or_r[0].cpu().numpy().astype(np.int64), tr.or_v[0].cpu().numpy(), tr.eta[0].cpu().numpy()
    assert np.isin(r, (0, K)).mean() > 0.999
    zp = tr.zp[0].cpu().numpy()
    assert np.isfinite(zp).all()
    w10 = P.block(SEED, CHAIN_OFFSET + np.arange(B), DRAW_OFFSET, P.SLOT_OVERRELAX + 2)[2]
    assert int((w10 >= 0xFFFF0000).sum()) >= 30
    for lo in range(0, B, 1 << 20):                      # in slices: the restatement's word arrays stay ~200 MB
        sl = slice(lo, lo + (1 << 20))
        n_near = _check_overrelax(SEED, CHAIN_OFFSET + np.arange(lo, lo + (1 << 20)), DRAW_OFFSET, K, "gauss", kfit,
                                  F64, r[sl], v[sl], eta[sl])
        assert n_near <= 20, n_near


# ---------------------------------------------------------------------------------------------------- edge words
def _edge(name):
    seed, draw, chain, slot, word, value = P.EDGE_WORDS[name]
    assert draw == 0
    return seed, chain


@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
def test_edge_word_overrelaxation_beta_is_inside_0_1(dtype):
    """Chains whose first beta exponential comes from a word with u01_32 = 1.0 (P.EDGE_WORDS), at normal D = 1,
    theta = +-8, K = 10: u0 = Phi(+-8) is saturated, so na = 1 and v = Ga / (Ga + Gb) with Ga from that word.  v must
    lie strictly inside (0, 1) and agree with exact logs, and the proposal must be finite (an exponential of 0 made
    v = 0, an infinite proposal and r = NaN).  fp32 runs the side where u' = u0 v (r = K): there 1 - (1 - u0) v, the
    other side, rounds to 1 for v this small."""
    K = 10
    model = kb.BSModel(stan_file="stan/normal.stan", data={"D": 1}, device=device())
    kfit, _ = fit_pair("gauss", dtype)
    kfit.overrelax_K = K
    assert_kernel(model, kfit, dtype, "tile")
    for name in ("overrelax_a", "overrelax_b"):
        seed, chain = _edge(name)
        side = np.sign(P.direction_normals(seed, [chain], 0, 1)[0, 0])      # rho; u0 = Phi(theta rho)
        for theta in ((8.0 * side, -8.0 * side) if dtype == F64 else (8.0 * side,)):
            th = up(np.array([[theta]]), dtype)
            tr = kb.Trace(1, 1, 1, 2, dtype, device(), variates=True, rho=True)
            kb.run(model, kfit, th, 1, seed, chain_offset=chain, draw_offset=0, trace=tr)
            torch.cuda.synchronize()
            r, v = int(tr.or_r[0, 0]), float(tr.or_v[0, 0])
            zp, lr = float(tr.zp[0, 0]), float(tr.r[0, 0])
            assert r == (K if theta * side > 0 else 0), (name, theta, r)
            _, v_ref = P.overrelax(seed, [chain], 0, K, None, r=[r])
            assert 0 < v < 1 and abs(v - v_ref[0]) <= _v_bound(K) * v_ref[0], (name, theta, v, v_ref[0])
            assert np.isfinite(zp) and np.isfinite(lr), (name, theta, zp, lr)


def test_edge_word_direction_radius_zero_gives_a_unit_direction():
    """Direction element 0 from a Box-Muller radius word with u01_32 = 1.0: that normal is exactly 0; the
    direction stays finite and of unit norm on the lane, tile and octet kernels."""
    seed, chain = _edge("direction")
    D = 4
    model = kb.BSModel(stan_file="stan/normal.stan", data={"D": D}, device=device())
    kfit, _ = fit_pair("gauss")
    z = P.direction_normals(seed, [chain], 0, D)[0]
    assert z[0] == 0 and (z[1:] != 0).all()
    for force, kernel in ((None, "lane"), ("tile", "tile"), ("octet", "octet")):
        kfit.force_octet, kfit.force_tile = force == "octet", force == "tile"
        assert_kernel(model, kfit, F64, kernel)
        th = up(np.zeros((1, D)))
        tr = kb.Trace(1, 1, D, 2, F64, device(), variates=True, rho=True)
        kb.run(model, kfit, th, 1, seed, chain_offset=chain, draw_offset=0, trace=tr)
        torch.cuda.synchronize()
        rho = tr.rho[0, 0].cpu().numpy()
        assert np.isfinite(rho).all() and rho[0] == 0 and abs(np.linalg.norm(rho) - 1) <= 1e-6, (kernel, rho)
        assert np.allclose(rho, z / np.linalg.norm(z), rtol=0, atol=2e-6), kernel
        assert np.isfinite(th.cpu().numpy()).all()


def test_edge_word_fp32_accept_uniform_of_1_rejects():
    """The fp32 accept uniform u01_32 = 1.0 (P.EDGE_WORDS): log u = 0 is never below min(0, r), so the draw is
    rejected -- without a NaN -- on the tile kernel (a Gaussian target that otherwise accepts every draw) and on MH."""
    seed, chain = _edge("accept_f32")
    D = 2
    model = kb.BSModel(stan_file="stan/normal.stan", data={"D": D}, device=device())
    kfit, _ = fit_pair("gauss", F32)
    assert_kernel(model, kfit, F32, "tile")
    th = up(np.array([[0.3, -0.2]]), F32)
    tr = kb.Trace(1, 1, D, 2, F32, device(), variates=True, rho=True)
    kb.run(model, kfit, th, 1, seed, chain_offset=chain, draw_offset=0, trace=tr)
    m = kb.MH(model, 0.5, seed=seed, chains=1, dtype=F32, theta=np.array([[0.3, -0.2]]), chain_offset=chain)
    tm = kb.Trace(1, 1, D, 2, F32, device(), variates=True, rho=True)
    m._advance(1, trace=tm)
    torch.cuda.synchronize()
    for t, what in ((tr, "klhr"), (tm, "mh")):
        assert float(t.u[0, 0]) == 1.0, what
        assert int(t.accept[0, 0]) == 0 and np.isfinite(float(t.r[0, 0])), (what, float(t.r[0, 0]))
    start = np.array([0.3, -0.2], dtype=np.float32)
    assert np.array_equal(th[0].cpu().numpy(), start) and np.array_equal(m.theta, start)


def test_edge_word_fp32_slice_shrinkage_uniform_of_1():
    """The first fp32 shrinkage uniform u01_32 = 1.0 (P.EDGE_WORDS): the candidate is the right end of the bracket.
    The draw still ends inside the slice, at a finite x1 with l(x1) >= l(0) - e."""
    seed, chain = _edge("slice_shrink_f32")
    D = 2
    model = kb.BSModel(stan_file="stan/normal.stan", data={"D": D}, device=device())
    om = stan_models.make_model("normal", {"D": D})
    theta0 = np.array([[0.4, -0.1]], dtype=np.float32).astype(np.float64)
    th = up(theta0, F32)
    tr = kb.Trace(1, 1, D, 0, F32, device(), variates=True, rho=True, slice_cap=8)
    kb.slice_run(model, kb.SliceConfig(w=1.0, cap=8), th, 1, seed, chain_offset=chain, draw_offset=0, trace=tr)
    torch.cuda.synchronize()
    assert float(tr.slice_u[0, 0, 0]) == 1.0 and int(tr.slice_n[0, 0]) >= 1
    x1, e = float(tr.zp[0, 0]), float(tr.z_init[0, 0])
    rho = tr.rho[0].double().cpu().numpy()
    assert np.isfinite(x1) and np.isfinite(th.cpu().numpy()).all()
    assert om.lp(theta0 + x1 * rho)[0] >= om.lp(theta0)[0] - e - 1e-5
