"""What a launch reports besides the chain state: per-draw evaluation counts, ``evals_total`` / ``grad_evals``,
``accept_count``, per-chain and pooled moment sums (with ``shift`` and ``skip_accum_last``), thinned ``draws`` rows
across launch cuts, and free-running fp32 parity.  Every reference value is computed on the host in fp64 from what
the kernel emitted -- its trace, its ``draws`` rows, or the oracle replaying its variates -- so a dropped or doubled
draw, an ignored shift or a miscounted evaluation fails here even where the chain state is right.

The kernel each case runs on is proven with ``launch_info`` (threads and dynamic shared memory of the launch plan)."""
import ctypes as C

import numpy as np
import pytest
import torch

import klhr_b200 as kb
from gpu_util import GAUSS_TAPES, SINH_TAPES, assert_kernel, device, fit_pair, rel_errors, replay_both, up
from oracle import batched, stan_models
from oracle.ref_port import gauss_hermite_probabilists

gpu = pytest.mark.gpu
F64, F32 = torch.float64, torch.float32
U32 = 2.0 ** -24                                    # unit roundoff of fp32

_rng = np.random.default_rng(0)
ARK = {"K": 5, "T": 300, "y": stan_models.simulate_ark_series(T=300, seed=5).tolist()}
EARNINGS = {"N": 50, "earn": (3 + _rng.normal(size=50)).tolist(), "height": (66 + 4 * _rng.normal(size=50)).tolist()}


# ---------------------------------------------------------------------------------------------------- CPU section
@pytest.mark.parametrize("N", [3, 8, 16])
def test_concave_quadratic_line_costs_the_closed_form_evaluation_count(N):
    """On a concave quadratic line the specification's fit costs 1 + 8 + N + 2 evaluations: the stage-1 start, one
    Newton step scored at 8 candidates (it lands on the mode), one KL evaluation of N nodes that already meets gtol2,
    then the proposal and the current point.  The lane and dense kernels report this constant without counting
    (csrc/klhr_lane.cuh), so it is pinned here to the oracle."""
    rng = np.random.default_rng(N)
    cfg = batched.FitConfig(N=N)
    xw = gauss_hermite_probabilists(N)
    B = 400
    for name, data in (("ill-normal", {"D": 20}), ("normal", {"D": 7}), ("corr-normal", {"N": 12, "rho": 0.9})):
        om = stan_models.make_model(name, data)
        D = om.dim()
        theta = rng.normal(size=(B, D)) * rng.uniform(0.05, 3.0, size=(B, 1))
        rho = rng.normal(size=(B, D))
        rho /= np.linalg.norm(rho, axis=1, keepdims=True)
        ref = batched.step(om, theta, rho, rng.normal(size=B), rng.normal(size=B), rng.random(B), cfg, xw=xw)
        assert ref["converged"].all(), name
        assert (ref["evals"] == 1 + 8 + N + 2).all(), (name, np.unique(ref["evals"]))


def test_mh_run_refuses_pooled_moments_and_a_lone_chain_s2():
    """klhr_mh_run has per-chain sums only: pooled sums and chain_s2 without chain_s1 are refused with a message
    (as klhr_slice_run does) instead of being silently ignored."""
    from klhr_b200 import _lib
    lib = _lib.load()
    model = _lib.ModelDesc(id=0, dim=4)
    pooled = _lib.AccumDesc(thin=1, pooled_s1=1, pooled_s2=2)
    assert lib.klhr_mh_run(C.byref(model), 0, None, 0.5, 8, 0, 0, 3, 1, C.byref(pooled), None, None) < 0
    assert "pooled" in _lib.last_error()
    lone = _lib.AccumDesc(thin=1, chain_s2=1)
    assert lib.klhr_mh_run(C.byref(model), 0, None, 0.5, 8, 0, 0, 3, 1, C.byref(lone), None, None) < 0
    assert "chain_s1" in _lib.last_error()
    assert lib.klhr_mh_run(C.byref(model), 0, None, 0.5, 0, 0, 0, 3, 1, C.byref(_lib.AccumDesc(thin=1)), None, None) == 0


# ---------------------------------------------------------------------------------------------------- helpers
def _direction(D, dtype=F64):
    """An adapted-looking direction law: two stored mean columns, one zero column, non-unit sd."""
    cols = np.zeros((2, D))
    cols[0, 0], cols[1, D - 1] = 1.5, -0.7
    return kb.Direction(mean_cols=up(cols, dtype), sd=up(np.linspace(0.5, 2.0, D), dtype),
                        cdf=up(np.array([0.3, 0.8, 1.0]), dtype), n_zero_cols=1)


def _kfit(family, dtype, force=None, or_K=0):
    kfit, ofit = fit_pair(family, dtype)
    kfit.force_octet, kfit.force_tile = force == "octet", force == "tile"
    kfit.overrelax_K = or_K
    return kfit, ofit


def _f32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


TRACE_FIELDS = ("eta", "zp", "r", "accept", "evals", "rho", "z_init", "z_prop", "u", "init4", "or_r", "or_v")


def _traced_run(model, kfit, theta0, dtype, cuts, seed, direction, rows=False):
    """Free-running draws split into launches of ``cuts`` draws, every launch traced (variates too) and adding into
    the same accept_count / evals_total.  ``rows``: also write every draw's state as a thin = 1 ``draws`` row (the
    kernels' kDraws instantiations).  Returns (theta, accept_count, evals_total, trace arrays over all draws, rows)."""
    B, D = theta0.shape
    th = up(theta0, dtype)
    acc = torch.zeros(B, dtype=torch.int64, device=device())
    ev = torch.zeros(1, dtype=torch.int64, device=device())
    draws = torch.full((sum(cuts), B, D), float("nan"), dtype=dtype, device=device()) if rows else None
    trs, off = [], 0
    for n in cuts:
        tr = kb.Trace(n, B, D, kfit.n_eta, dtype, device(), variates=True, rho=True)
        kb.run(model, kfit, th, n, seed, direction, draw_offset=off, accept_count=acc, evals_total=ev, trace=tr,
               draws=draws, thin=1, thin_offset=off)
        trs.append(tr)
        off += n
    torch.cuda.synchronize()
    out = {}
    for f in TRACE_FIELDS:
        if getattr(trs[0], f) is None:
            out[f] = None
            continue
        x = torch.cat([getattr(t, f) for t in trs])
        out[f] = (x if x.dtype in (torch.int32, torch.int64) else x.double()).cpu().numpy()
    if rows:
        assert torch.equal(draws[-1], th)
    return th, acc.cpu().numpy(), int(ev.item()), out, None if draws is None else draws.double().cpu().numpy()


def _replay(om, t, s, theta, ofit, kfit):
    g = lambda f: None if t[f] is None else t[f][s]
    return batched.step(om, theta, g("rho"), g("z_init"), g("z_prop"), g("u"), ofit, init4=g("init4"),
                        xw=(kfit.x, kfit.w), or_K=kfit.overrelax_K, or_r=g("or_r"), or_v=g("or_v"))


# ---------------------------------------------------------------------------------------------------- 1. evaluations
from conftest import load_tape                        # noqa: E402


def _replay_tape(name, force_octet):
    t, meta, data = load_tape(name)
    return replay_both(meta["model"], data, meta["family"], t["theta0"], t["rho"], t["z_init"], t["z_prop"], t["u"],
                       init4=t.get("init4"), xw=(t["x_nodes"], t["w_nodes"]), force_octet=force_octet)


@gpu
@pytest.mark.parametrize("name,force_octet", [(n, f) for n in GAUSS_TAPES for f in (False, True)])
def test_replay_evaluation_counts_gauss_tapes(name, force_octet):
    gpu_, ref = _replay_tape(name, force_octet)
    assert np.array_equal(gpu_["evals"], ref["evals"]), np.flatnonzero(gpu_["evals"] != ref["evals"])[:10]


@gpu
@pytest.mark.parametrize("name,force_octet", [(n, f) for n in SINH_TAPES for f in (False, True)])
def test_replay_evaluation_counts_sinh_tapes(name, force_octet):
    gpu_, ref = _replay_tape(name, force_octet)
    conv = ref["converged"]
    bad = conv & (gpu_["evals"] != ref["evals"])
    assert not bad.any(), (f"{bad.sum()} converged fits differ; not converged: {1 - conv.mean():.4f}",
                           np.flatnonzero(bad)[:10])


@gpu
@pytest.mark.parametrize("N,rho,B", [(128, 0.5, 333), (256, 0.9, 500)])
def test_dense_kernel_replay_evaluation_and_accept_counts(N, rho, B):
    """The plain dense kernel in replay (none of the tapes is at D = 128 / 256): per-draw evals and accept flags equal
    the oracle's on every chain, ragged last CTA included."""
    data = {"N": N, "rho": rho}
    model = kb.BSModel(stan_file="stan/corr-normal.stan", data=data, device=device())
    assert_kernel(model, _kfit("gauss", F64)[0], F64, "dense", free_running=False)
    rng = np.random.default_rng(N + B)
    theta = rng.normal(size=(B, N)) * 0.7
    r = rng.normal(size=(B, N))
    r /= np.linalg.norm(r, axis=1, keepdims=True)
    gpu_, ref = replay_both("corr-normal", data, "gauss", theta, r, rng.normal(size=B), rng.normal(size=B), rng.random(B))
    assert np.array_equal(gpu_["evals"], ref["evals"]) and np.array_equal(gpu_["accept"], ref["accept"])


# (id, model, data, family, force, dtype, B, kernel, kernel with draws rows, overrelax_K).  The draws rows run on the
# kDraws instantiation of the same kernel, except on corr-normal D = 128 / 256: there launches without rows take the
# warp-specialised kernel and launches with rows the plain dense kernel (klhr_densek.cu).
FREE = [
    ("lane-d100", "ill-normal", {"D": 100}, "gauss", None, F64, 777, "lane", "lane", 0),
    ("lane-d33", "ill-normal", {"D": 33}, "gauss", None, F64, 777, "lane", "lane", 0),
    ("lane-d40-b19", "ill-normal", {"D": 40}, "gauss", None, F64, 19, "lane", "lane", 0),
    ("tile-d100", "ill-normal", {"D": 100}, "gauss", "tile", F64, 777, "tile", "tile", 0),
    ("tile-d33", "ill-normal", {"D": 33}, "gauss", "tile", F64, 777, "tile", "tile", 0),
    ("tile-f32-d100", "ill-normal", {"D": 100}, "gauss", None, F32, 777, "tile", "tile", 0),
    ("tile-f32-normal5-b19", "normal", {"D": 5}, "gauss", None, F32, 19, "tile", "tile", 0),
    ("chain-funnel1-sinh", "funnel", {"D": 1}, "sinh", None, F64, 777, "chain_serial", "chain_serial", 0),
    ("chain-funnel10", "funnel", {"D": 10}, "gauss", None, F64, 777, "chain_serial", "chain_serial", 0),
    ("chain-rosenbrock2-b19", "rosenbrock", {"D": 2}, "gauss", None, F64, 19, "chain_serial", "chain_serial", 0),
    ("chain-ark5", "arK", ARK, "gauss", None, F64, 333, "chain_serial", "chain_serial", 0),
    ("chain-earnings", "earnings", EARNINGS, "gauss", None, F64, 333, "chain_serial", "chain_serial", 0),
    ("chain-funnel2-overrelaxed", "funnel", {"D": 2}, "gauss", None, F64, 777, "chain_serial", "chain_serial", 10),
    ("chain-funnel30", "funnel", {"D": 30}, "gauss", None, F64, 777, "chain_octet", "chain_octet", 0),
    ("octet-d100", "ill-normal", {"D": 100}, "gauss", "octet", F64, 777, "octet", "octet", 0),
    ("octet-funnel1-sinh", "funnel", {"D": 1}, "sinh", "octet", F64, 777, "octet", "octet", 0),
    ("octet-funnel10-b19", "funnel", {"D": 10}, "gauss", "octet", F64, 19, "octet", "octet", 0),
    ("octet-rosenbrock2", "rosenbrock", {"D": 2}, "gauss", "octet", F64, 777, "octet", "octet", 0),
    ("octet-ark5", "arK", ARK, "gauss", "octet", F64, 333, "octet", "octet", 0),
    ("octet-earnings", "earnings", EARNINGS, "gauss", "octet", F64, 333, "octet", "octet", 0),
    ("octet-funnel2-overrelaxed", "funnel", {"D": 2}, "gauss", "octet", F64, 777, "octet", "octet", 10),
    ("octet-funnel30", "funnel", {"D": 30}, "gauss", "octet", F64, 777, "octet", "octet", 0),
    ("octet-corr44-dense-cta", "corr-normal", {"N": 44, "rho": 0.5}, "gauss", "octet", F64, 77, "octet", "octet", 0),
    ("dense-128", "corr-normal", {"N": 128, "rho": 0.5}, "gauss", None, F64, 500, "dense_ws", "dense", 0),
    ("dense-256", "corr-normal", {"N": 256, "rho": 0.9}, "gauss", None, F64, 500, "dense_ws", "dense", 0),
    ("dense-128-b333", "corr-normal", {"N": 128, "rho": 0.5}, "gauss", None, F64, 333, "dense_ws", "dense", 0),
]


@gpu
@pytest.mark.parametrize("case", FREE, ids=[c[0] for c in FREE])
def test_free_running_evaluation_and_accept_counts(case):
    """Five draws in two launches cut at draw 2, run twice: without and with thin = 1 draws rows.  Every draw is
    replayed through the oracle on the emitted variates from the device's own state (the rows): per-draw evals equal
    the oracle's (Gaussian family: every chain; sinh: converged fits) in both runs, evals_total is the sum of the
    per-draw counts and accept_count the sum of the accept flags, exactly."""
    cid, name, data, family, force, dtype, B, kernel, kernel_rows, or_K = case
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
    om = stan_models.make_model(name, data)
    kfit, ofit = _kfit(family, dtype, force, or_K)
    assert_kernel(model, kfit, dtype, kernel)
    assert_kernel(model, kfit, dtype, kernel_rows, free_running=kernel_rows != "dense")
    D, S = model.dim(), 5
    rng = np.random.default_rng(B + D)
    theta0 = rng.normal(size=(B, D)) * 0.3
    if dtype == F32:
        theta0 = _f32(theta0)
    runs = [_traced_run(model, kfit, theta0, dtype, (2, 3), 13, _direction(D, dtype), rows=r) for r in (False, True)]
    rows = runs[1][4]
    companion = None
    if name == "earnings":                      # the other of the chain / octet kernels on the same draws
        kc, _ = _kfit(family, dtype, None if force == "octet" else "octet", or_K)
        companion = _traced_run(model, kc, theta0, dtype, (2, 3), 13, _direction(D, dtype), rows=True)[3]
    for th, acc, ev, t, _ in runs:
        assert ev == int(t["evals"].astype(np.int64).sum())
        assert np.array_equal(acc, t["accept"].astype(np.int64).sum(0))
        if "funnel" in name:                    # these cases do reject, so the count is not B * S by construction
            assert (t["accept"] == 0).any()
        states = np.concatenate([theta0[None], rows])
        scale = np.maximum(1.0, np.abs(rows[-1]))
        assert (np.abs(th.double().cpu().numpy() - rows[-1]) <= 1e-12 * scale).all()
        n_bad = 0
        for s in range(S):
            ref = _replay(om, t, s, states[s], ofit, kfit)
            mask = np.ones(B, dtype=bool) if family == "gauss" else ref["converged"]
            bad = mask & (t["evals"][s] != ref["evals"])
            if name == "earnings":
                # lp up to ~1e11: a stopping test of the Newton loop can fall within rounding of its threshold, and the
                # same fit then ends one or two KL evaluations off the oracle (measured: 1 of 1665 chain-draws).  The
                # chain and octet kernels must still agree with each other on those chains.
                assert np.array_equal(t["evals"][s][bad], companion["evals"][s][bad]), (cid, s)
                n_bad += int(bad.sum())
            else:
                assert not bad.any(), (cid, s, int(bad.sum()), t["evals"][s][bad][:5], ref["evals"][bad][:5],
                                       f"not converged: {1 - ref['converged'].mean():.4f}")
        assert n_bad <= 0.002 * B * S, (cid, n_bad)


@gpu
@pytest.mark.parametrize("cls,name,data", [("KLHR", "ill-normal", {"D": 100}), ("KLHR", "funnel", {"D": 10}),
                                           ("Slice", "funnel", {"D": 1})])
def test_sampler_grad_evals_is_the_sum_of_the_per_draw_counts(cls, name, data):
    """grad_evals of KLHR(..., warmup=0).run(3); run(4) against a traced kb.run / slice_run of the same chains, seed,
    direction law and draw offsets."""
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
    s = getattr(kb, cls)(model, seed=6, chains=333, warmup=0)
    th, direction = s._theta.clone(), s._direction
    s.run(3)
    s.run(4)
    B, D, per_draw = 333, model.dim(), 0
    for off, n in ((0, 3), (3, 4)):
        if cls == "KLHR":
            tr = kb.Trace(n, B, D, 2, F64, device())
            kb.run(model, s._fit, th, n, s.seed, direction, draw_offset=off, trace=tr)
        else:
            tr = kb.Trace(n, B, D, 0, F64, device(), slice_cap=s._slice.cap)
            kb.slice_run(model, s._slice, th, n, s.seed, direction, draw_offset=off, trace=tr)
        per_draw += int(tr.evals.long().sum())
    torch.cuda.synchronize()
    assert s.grad_evals == per_draw and torch.equal(th, s.theta)


# ---------------------------------------------------------------------------------------------------- 3. moment sums
def _check_sum(dev, ref, mag, dtype, S, what):
    """fp64: 1e-12 of the sum of |terms|; fp32: the recursive-summation bound S u sum|terms| (one missing or doubled
    draw of S = 60 is ~100x more)."""
    dev = dev.double().cpu().numpy() if torch.is_tensor(dev) else dev
    tol = (1e-12 if dtype == F64 else S * U32) * mag
    err = np.abs(dev - ref)
    assert (err <= tol).all(), (what, float((err / np.maximum(tol, 1e-300)).max()))


def _check_moments(rows, keep, shift, s1, s2, dtype, S, pooled=None):
    x = rows[keep]
    d = x - (shift if shift is not None else 0.0)
    _check_sum(s1, d.sum(0), np.abs(d).sum(0), dtype, S, "chain_s1")
    _check_sum(s2, (d * d).sum(0), (d * d).sum(0), dtype, S, "chain_s2")
    if pooled is not None:
        _check_sum(pooled[0], d.sum((0, 1)), np.abs(d).sum((0, 1)), dtype, S, "pooled_s1")
        _check_sum(pooled[1], (d * d).sum((0, 1)), (d * d).sum((0, 1)), dtype, S, "pooled_s2")


def _moved(rows, theta0):
    """Accepted draws per chain read off the rows: a draw is accepted iff the state moved."""
    prev = np.concatenate([theta0[None], rows[:-1]])
    return (rows != prev).any(axis=2).sum(0)


ACCUM = [("ill-normal", {"D": 100}, F64, 777), ("ill-normal", {"D": 100}, F32, 777), ("funnel", {"D": 10}, F64, 19),
         ("funnel", {"D": 10}, F32, 333), ("corr-normal", {"N": 44, "rho": 0.5}, F64, 77)]


@gpu
@pytest.mark.parametrize("name,data,dtype,B", ACCUM, ids=[f"{a}-{str(c)[6:]}-b{d}" for a, _, c, d in ACCUM])
def test_step_kernel_moment_sums_shift_and_skip_accum_last(name, data, dtype, B):
    """The octet step kernel's per-chain and pooled sums (ragged last CTA) over the kernel's own thin = 1 rows: two
    launches of 25 + 35 draws add; a per-coordinate shift is subtracted; skip_accum_last leaves out the last draw of
    each launch; shift=None gives raw sums."""
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
    kfit, _ = _kfit("gauss", dtype)
    assert_kernel(model, kfit, dtype, "octet", accumulate=True)
    D, S, cut = model.dim(), 60, 25
    rng = np.random.default_rng(D)
    theta0 = _f32(rng.normal(size=(B, D)) * 0.3)
    shift_h = _f32(rng.normal(size=D) * 0.7 + 0.3)
    direction = _direction(D, dtype)
    for shift, skip in ((up(shift_h, dtype), False), (None, True)):
        th = up(theta0, dtype)
        z = lambda *sh: torch.zeros(*sh, dtype=F64, device=device())
        cs1, cs2, ps1, ps2 = z(B, D), z(B, D), z(D), z(D)
        acc = torch.zeros(B, dtype=torch.int64, device=device())
        draws = torch.empty(S, B, D, dtype=dtype, device=device())
        for off, n in ((0, cut), (cut, S - cut)):
            kb.run(model, kfit, th, n, 21, direction, draw_offset=off, shift=shift, pooled_s1=ps1, pooled_s2=ps2,
                   chain_s1=cs1, chain_s2=cs2, accept_count=acc, draws=draws, thin=1, thin_offset=off,
                   skip_accum_last=skip)
        torch.cuda.synchronize()
        rows = draws.double().cpu().numpy()
        assert torch.equal(draws[-1], th)
        keep = np.ones(S, dtype=bool)
        if skip:
            keep[[cut - 1, S - 1]] = False
        _check_moments(rows, keep, shift_h if shift is not None else None, cs1, cs2, dtype, S, pooled=(ps1, ps2))
        assert np.array_equal(acc.cpu().numpy(), _moved(rows, theta0))
        if name == "funnel":
            assert int(acc.sum()) < B * S


@gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("name,data,step", [("normal", {"D": 10}, 0.5), ("funnel", {"D": 2}, 1.0)])
def test_mh_moment_sums_shift_and_accept_count(name, data, step, dtype):
    """MH adds (theta - shift) to fp64 per-chain sums every draw; two launches add; accept_count counts the moves."""
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
    D, B, S, cut = model.dim(), 1000, 60, 25
    rng = np.random.default_rng(3)
    shift_h = _f32(rng.normal(size=D) * 0.7 + 0.3)
    for shift in (up(shift_h, dtype), None):
        m = kb.MH(model, step, seed=4, chains=B, dtype=dtype, theta=_f32(rng.normal(size=(B, D)) * 0.5))
        theta0 = m.theta.double().cpu().numpy()
        z = lambda *sh: torch.zeros(*sh, dtype=F64, device=device())
        cs1, cs2 = z(B, D), z(B, D)
        draws = torch.empty(S, B, D, dtype=dtype, device=device())
        for off, n in ((0, cut), (cut, S - cut)):
            m._advance(n, draws=draws, thin=1, thin_offset=off, chain_s1=cs1, chain_s2=cs2, shift=shift)
        torch.cuda.synchronize()
        rows = draws.double().cpu().numpy()
        _check_moments(rows, np.ones(S, dtype=bool), shift_h if shift is not None else None, cs1, cs2, dtype, S)
        acc = m._accept_count.cpu().numpy()
        assert np.array_equal(acc, _moved(rows, theta0))
        assert 0.2 < acc.sum() / (B * S) < 0.8                   # it does reject
        assert m.acceptance_probability == acc.sum() / B / S


@gpu
@pytest.mark.parametrize("dtype", [F64, F32], ids=["f64", "f32"])
@pytest.mark.parametrize("name,data", [("ill-normal", {"D": 100}), ("funnel", {"D": 1})])
def test_slice_moment_sums_shift_and_accept_count(name, data, dtype):
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
    D, B, S, cut = model.dim(), 777, 60, 25
    rng = np.random.default_rng(4)
    theta0 = _f32(rng.normal(size=(B, D)) * 0.5)
    shift_h = _f32(rng.normal(size=D) * 0.7 + 0.3)
    cfg = kb.SliceConfig(w=1.0)
    for shift in (up(shift_h, dtype), None):
        th = up(theta0, dtype)
        z = lambda *sh: torch.zeros(*sh, dtype=F64, device=device())
        cs1, cs2 = z(B, D), z(B, D)
        acc = torch.zeros(B, dtype=torch.int64, device=device())
        draws = torch.empty(S, B, D, dtype=dtype, device=device())
        for off, n in ((0, cut), (cut, S - cut)):
            kb.slice_run(model, cfg, th, n, 8, _direction(D, dtype), draw_offset=off, shift=shift, chain_s1=cs1,
                         chain_s2=cs2, accept_count=acc, draws=draws, thin=1, thin_offset=off)
        torch.cuda.synchronize()
        rows = draws.double().cpu().numpy()
        _check_moments(rows, np.ones(S, dtype=bool), shift_h if shift is not None else None, cs1, cs2, dtype, S)
        assert (acc == S).all()


# ---------------------------------------------------------------------------------------------------- 4. thinned rows
# (id, model, data, family, force, dtype, kernel, bitwise).  Bitwise where the kernel is cut-invariant (lane, octet:
# theta is re-read from the state every draw); the tile and chain kernels carry pending moves across the draws of a
# launch, the dense kernel w = L' theta, and they are held to 1e-12 relative.  launch_info has no draws argument: the
# dense case proves the plain dense kernel's plan through its replay launch, the plan sample() rows run on too.
DRAWS = [
    ("lane", "ill-normal", {"D": 100}, "gauss", None, F64, "lane", True),
    ("tile", "ill-normal", {"D": 33}, "gauss", "tile", F64, "tile", False),
    ("tile-f32", "normal", {"D": 5}, "gauss", None, F32, "tile", False),
    ("chain", "funnel", {"D": 10}, "gauss", None, F64, "chain_serial", False),
    ("chain-sinh", "funnel", {"D": 1}, "sinh", None, F64, "chain_serial", False),
    ("octet", "funnel", {"D": 10}, "gauss", "octet", F64, "octet", True),
    ("dense", "corr-normal", {"N": 128, "rho": 0.5}, "gauss", None, F64, "dense", False),
]


def _same_rows(a, b, bitwise, what):
    if bitwise:
        assert torch.equal(a, b), what
    else:
        err = ((a - b).abs() / b.abs().clamp(min=1.0)).max()
        assert float(err) <= 1e-12, (what, float(err))


@gpu
@pytest.mark.parametrize("case", DRAWS, ids=[c[0] for c in DRAWS])
def test_thinned_rows_across_a_launch_cut(case):
    """Rows of thin in {1, 3, 4} written over two launches cut at a draw that is not a multiple of thin (thin_offset):
    row r is the state after global draw (r + 1) thin, taken from a separate single launch of that many draws."""
    cid, name, data, family, force, dtype, kernel, bitwise = case
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
    kfit, _ = _kfit(family, dtype, force)
    assert_kernel(model, kfit, dtype, kernel, free_running=kernel != "dense")
    D, B, M = model.dim(), 333, 4
    rng = np.random.default_rng(7)
    theta0 = rng.normal(size=(B, D)) * 0.3
    direction = _direction(D, dtype)
    for thin in (1, 3, 4):
        T, cut = M * thin, 5 if thin > 1 else 2
        th = up(theta0, dtype)
        rows = torch.full((M, B, D), float("nan"), dtype=dtype, device=device())
        for off, n in ((0, cut), (cut, T - cut)):
            kb.run(model, kfit, th, n, 31, direction, draw_offset=off, draws=rows, thin=thin, thin_offset=off)
        for r in range(M):
            ref = up(theta0, dtype)
            # corr-normal D = 128: rows keep the reference launch on the plain dense kernel (without them it would run
            # on the warp-specialised one)
            keep = torch.empty((r + 1) * thin, B, D, dtype=dtype, device=device()) if kernel == "dense" else None
            kb.run(model, kfit, ref, (r + 1) * thin, 31, direction, draws=keep)
            torch.cuda.synchronize()
            _same_rows(rows[r], ref, bitwise, (cid, thin, r))
        assert torch.equal(rows[-1], th)


@gpu
@pytest.mark.parametrize("thin", [1, 3, 4])
def test_mh_and_slice_thinned_rows_across_a_launch_cut(thin):
    """Same for the MH and Slice kernels (cut-invariant: bitwise)."""
    B, M = 333, 4
    T, cut = M * thin, 5 if thin > 1 else 2
    rng = np.random.default_rng(thin)
    mm = kb.BSModel(stan_file="stan/funnel.stan", data={"D": 2}, device=device())
    theta0 = rng.normal(size=(B, 3)) * 0.5
    m = kb.MH(mm, 0.8, seed=2, chains=B, theta=theta0)
    rows = torch.full((M, B, 3), float("nan"), dtype=F64, device=device())
    m._advance(cut, draws=rows, thin=thin, thin_offset=0)
    m._advance(T - cut, draws=rows, thin=thin, thin_offset=cut)
    for r in range(M):
        ref = kb.MH(mm, 0.8, seed=2, chains=B, theta=theta0)
        ref.run((r + 1) * thin)
        assert torch.equal(rows[r], ref.theta), ("mh", r)
    sm = kb.BSModel(stan_file="stan/ill-normal.stan", data={"D": 100}, device=device())
    theta0 = rng.normal(size=(B, 100)) * 0.5
    cfg, direction = kb.SliceConfig(w=1.0), _direction(100)
    th = up(theta0)
    rows = torch.full((M, B, 100), float("nan"), dtype=F64, device=device())
    for off, n in ((0, cut), (cut, T - cut)):
        kb.slice_run(sm, cfg, th, n, 5, direction, draw_offset=off, draws=rows, thin=thin, thin_offset=off)
    for r in range(M):
        ref = up(theta0)
        kb.slice_run(sm, cfg, ref, (r + 1) * thin, 5, direction)
        torch.cuda.synchronize()
        assert torch.equal(rows[r], ref), ("slice", r)


@gpu
def test_sample_rows_are_the_start_and_the_thinned_states():
    """sample(M, thin) of KLHR, MH and Slice: row 0 is the starting state, row r the state after r thin draws."""
    model = kb.BSModel(stan_file="stan/ill-normal.stan", data={"D": 100}, device=device())
    B, M, thin = 333, 4, 3
    theta0 = np.random.default_rng(1).normal(size=(B, 100)) * 0.3
    makers = {"KLHR": lambda: kb.KLHR(model, seed=3, chains=B, warmup=0, theta=theta0),
              "Slice": lambda: kb.Slice(model, seed=3, chains=B, warmup=0, theta=theta0),
              "MH": lambda: kb.MH(model, 0.2, seed=3, chains=B, theta=theta0)}
    for cls, mk in makers.items():
        out = mk().sample(M, thin=thin)
        assert torch.equal(out[0], up(theta0)), cls
        for r in range(1, M):
            s = mk()
            s.run(r * thin)
            assert torch.equal(out[r], s.theta), (cls, r)


# ---------------------------------------------------------------------------------------------------- 5. fp32
F32_CASES = [("ill-normal", {"D": 100}), ("normal", {"D": 5}), ("funnel", {"D": 4}), ("rosenbrock", {"D": 2}),
             ("ar1", {"N": 20}), ("arK", ARK)]


@gpu
@pytest.mark.parametrize("force_octet", [False, True], ids=["default", "octet"])
@pytest.mark.parametrize("name,data", F32_CASES, ids=[c[0] for c in F32_CASES])
def test_fp32_free_running_step_equals_oracle_on_emitted_variates(name, data, force_octet):
    """fp32 klhr_run (tile / chain / octet kernel) replayed through the oracle on the emitted fp32 variates, from the
    device's state, at the fp32 replay bar of test_gpu_replay."""
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
    om = stan_models.make_model(name, data)
    kfit, ofit = _kfit("gauss", F32, "octet" if force_octet else None)
    D, B, S = model.dim(), 500, 3
    assert_kernel(model, kfit, F32, "octet" if force_octet else
                  "tile" if name in ("normal", "ill-normal") else "chain_serial" if D <= 16 else "chain_octet")
    theta0 = _f32(np.random.default_rng(D).normal(size=(B, D)) * 0.3)
    th, acc, ev, t, _ = _traced_run(model, kfit, theta0, F32, (1, 2), 17, _direction(D, F32))
    assert ev == int(t["evals"].astype(np.int64).sum()) and np.array_equal(acc, t["accept"].astype(np.int64).sum(0))
    # the device's state after every draw: the same launches again with thin = 1 rows
    rows = _traced_run(model, kfit, theta0, F32, (1, 2), 17, _direction(D, F32), rows=True)[4]
    states = np.concatenate([theta0[None], rows])
    worst, flips = [], []
    for s in range(S):
        ref = _replay(om, t, s, states[s], ofit, kfit)
        em, es, ez, _ = rel_errors(dict(eta=t["eta"][s], zp=t["zp"][s], r=t["r"][s]), ref, "gauss")
        worst.append(np.maximum.reduce([em, es, ez]))
        flips.append(t["accept"][s].astype(bool) != ref["accept"])
    worst, flips = np.concatenate(worst), np.concatenate(flips)
    assert (worst <= 1e-4).mean() >= 0.995 and worst.max() <= 1e-2, (float((worst <= 1e-4).mean()), float(worst.max()))
    if name in ("normal", "ill-normal", "ar1"):
        assert worst.max() <= 1e-4, float(worst.max())
    assert flips.mean() <= 0.002


@gpu
@pytest.mark.parametrize("name,data,step", [("normal", {"D": 10}, 0.5), ("funnel", {"D": 2}, 1.0)])
def test_fp32_mh_equals_numpy_replay(name, data, step):
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
    om = stan_models.make_model(name, data)
    B, S, D = 2000, 5, model.dim()
    theta0 = _f32(np.random.default_rng(2).normal(size=(B, D)) * 0.5)
    m = kb.MH(model, step, seed=3, chains=B, dtype=F32, theta=theta0)
    tr = kb.Trace(S, B, D, 2, F32, device(), variates=True, rho=True)
    m._advance(S, trace=tr)
    torch.cuda.synchronize()
    theta, flips = theta0, []
    step32 = np.float32(step)
    for k in range(S):
        xi = tr.rho[k].cpu().numpy()
        u = tr.u[k].double().cpu().numpy()
        cand = (theta.astype(np.float32) + xi * step32).astype(np.float64)
        l0, l1 = om.lp(theta), om.lp(cand)
        r = l1 - l0
        ok = np.isfinite(r)
        r_dev = tr.r[k].double().cpu().numpy()
        assert (np.abs(r_dev - r)[ok] <= 1e-5 * (1 + np.abs(l0) + np.abs(l1))[ok]).all()
        acc_dev = tr.accept[k].cpu().numpy().astype(bool)
        flips.append(acc_dev != (np.log(u) < np.minimum(0.0, r)))
        theta = np.where(acc_dev[:, None], cand, theta)
    assert np.concatenate(flips).mean() <= 0.002
    assert np.allclose(m.theta.double().cpu().numpy(), theta, rtol=1e-6, atol=1e-6)


@gpu
@pytest.mark.parametrize("name,data", [("ill-normal", {"D": 100}), ("funnel", {"D": 1})])
def test_fp32_slice_equals_oracle_on_emitted_variates(name, data):
    model = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
    om = stan_models.make_model(name, data)
    B, S, D, cap, w = 1500, 4, model.dim(), 40, 1.0
    theta0 = _f32(np.random.default_rng(1).normal(size=(B, D)) * 0.5)
    th = up(theta0, F32)
    tr = kb.Trace(S, B, D, 0, F32, device(), variates=True, rho=True, slice_cap=cap)
    kb.slice_run(model, kb.SliceConfig(w=w, cap=cap), th, S, 11, _direction(D, F32), trace=tr)
    torch.cuda.synchronize()
    g = lambda f, k: getattr(tr, f)[k].double().cpu().numpy()
    theta, same_all = theta0, []
    for k in range(S):
        rho = g("rho", k)
        ref = batched.slice_step(om, theta, rho, g("z_init", k), g("u", k), g("slice_u", k), w=w)
        same = (tr.slice_n[k].cpu().numpy() == ref["n_shrink"]) & (tr.evals[k].cpu().numpy() == ref["evals"])
        same_all.append(same)
        x1 = g("zp", k)
        assert (np.abs(x1 - ref["x1"])[same] <= 1e-4 * (w + np.abs(ref["x1"]))[same]).all()
        theta = (theta.astype(np.float32) + x1.astype(np.float32)[:, None] * rho.astype(np.float32)).astype(np.float64)
    assert np.concatenate(same_all).mean() >= 0.99


@gpu
def test_fp32_model_eval_outer_accumulate_and_sinh_refusal():
    """klhr_model_eval and the pooled outer-product snapshot (outer_kernel<float>) on fp32 input against fp64 on the
    same rounded input; KLHRSINH refuses fp32 by design."""
    rng = np.random.default_rng(0)
    cases = [("normal", {"D": 5}), ("ill-normal", {"D": 33}), ("funnel", {"D": 6}),
             ("corr-normal", {"N": 20, "rho": 0.9}), ("ar1", {"N": 17}), ("arK", ARK), ("rosenbrock", {"D": 3}),
             ("earnings", EARNINGS)]
    for name, data in cases:
        m = kb.BSModel(stan_file=f"stan/{name}.stan", data=data, device=device())
        om = stan_models.make_model(name, data)
        th = _f32(rng.normal(size=(257, m.dim())) * 0.5)
        lp, g = m.log_density_gradient(up(th, F32))
        assert lp.dtype == F32 and g.dtype == F32
        rl, rg = om.lp_grad(th)
        lp, g = lp.double().cpu().numpy(), g.double().cpu().numpy()
        assert (np.abs(lp - rl) <= 1e-5 * (1 + np.abs(rl))).all(), (name, float(np.abs(lp - rl).max()))
        assert (np.abs(g - rg).max(1) <= 1e-5 * (1 + np.abs(rg).max(1))).all(), (name, float(np.abs(g - rg).max()))
    for B, D in ((1000, 7), (33, 40), (5000, 100)):
        x, sh = _f32(rng.normal(size=(B, D)) + 0.5), _f32(rng.normal(size=D) * 0.3)
        d = x - sh
        for scratch in (False, True):
            outer = torch.zeros(D, D, dtype=F64, device=device())
            s1 = torch.zeros(D, dtype=F64, device=device())
            xt = up(x, F32)
            scr = kb.outer_scratch(xt) if scratch else None
            kb.outer_accumulate(xt, up(sh, F32), outer, s1, scratch=scr)
            if scratch:
                kb.outer_reduce(scr, outer, s1, B, D)
            torch.cuda.synchronize()
            # outer_kernel promotes theta and shift to fp64 before subtracting, so the fp64 bound applies: one chain
            # dropped or doubled is 1 / B of the sum, far above it even at B = 5000
            _check_sum(outer, d.T @ d, np.abs(d).T @ np.abs(d), F64, B, "outer")
            _check_sum(s1, d.sum(0), np.abs(d).sum(0), F64, B, "s1")
    model = kb.BSModel(stan_file="stan/funnel.stan", data={"D": 1}, device=device())
    with pytest.raises(TypeError, match="float64"):
        kb.KLHRSINH(model, dtype=F32)


@gpu
def test_fp32_klhr_posterior_ill_normal_within_4_mcse():
    """The fp32 sampler end to end: the adaptation and chain_stats launches carry accumulators and run on the fp32
    octet step kernel (kAccum), plain stretches on the tile kernel, with outer_kernel<float> snapshots of the adaptation:
    posterior means and variances of ill-normal D = 100 within 4.5 MCSE of the truth."""
    from klhr_b200.diagnostics import chain_summary
    D, B = 100, 4096
    model = kb.BSModel(stan_file="stan/ill-normal.stan", data={"D": D}, device=device())
    s = kb.KLHR(model, seed=3, chains=B, dtype=F32)
    s.run(1000)
    assert s._windowedadaptation.closures == [50, 150, 350, 1000]
    s.run(2000)
    S = 3000
    s1, s2 = s.run(S, chain_stats=True)
    summ = chain_summary(s1, s2, S)
    truth = torch.arange(1, D + 1, dtype=F64, device=device()) ** 2 / D
    zm = summ["mean"].abs() / summ["mcse_mean"]
    zv = (summ["var"] - truth).abs() / summ["mcse_var"]
    assert float(zm.max()) < 4.5 and float((zm > 4).float().mean()) <= 0.02, float(zm.max())
    assert float(zv.max()) < 4.5 and float((zv > 4).float().mean()) <= 0.02, float(zv.max())
