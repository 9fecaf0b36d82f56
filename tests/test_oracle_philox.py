"""oracle/philox.py against the Random123 known-answer vectors, and the laws of the variates it derives (CPU).

The law tests are seeded and deterministic; their thresholds are p-values of 1e-6."""
import numpy as np
import pytest
from scipy import stats

from oracle import philox as P

P_MIN = 1e-6


def test_philox4x32_10_known_answers():
    for ctr, key, out in P.KAT:
        got = tuple(int(x) for x in P.philox4x32_10(*ctr, *key))
        assert got == out, [hex(g) for g in got]


def test_direction_normals_have_gaussian_moments_and_tails():
    """Box-Muller on 24-bit uniforms: radius capped at sqrt(2 * 25 * ln 2) = 5.9 sigma; the tail frequencies up to
    there must be those of N(0, 1) (|z| > 3: 2.70e-3, |z| > 4: 6.33e-5)."""
    z = P.direction_normals(seed=20261018, chain=np.arange(20000), draw=3, D=128).ravel()      # 2.56e6 normals
    n = z.size
    assert abs(z.mean()) < 4 / np.sqrt(n) and abs(z.var() - 1) < 4 * np.sqrt(2 / n)
    assert abs(np.mean(z ** 4) - 3) < 4 * np.sqrt(96 / n)
    for cut, p in ((3.0, 2.6998e-3), (4.0, 6.3342e-5)):
        k = int((np.abs(z) > cut).sum())
        assert abs(k - n * p) < 4.5 * np.sqrt(n * p), (cut, k, n * p)
    assert np.abs(z).max() < 5.9
    u_col, z_init, z_prop, u = P.chain_scalars(7, np.arange(100000), 11)
    assert 0 < u.min() and u.max() < 1 and abs(u.mean() - 0.5) < 4 / np.sqrt(12 * u.size)
    assert abs(z_prop.mean()) < 4 / np.sqrt(z_prop.size) and abs(z_prop.var() - 1) < 4 * np.sqrt(2 / z_prop.size)


# ---------------------------------------------------------------------------------------------------- edge words
def test_edge_words_still_hit_the_top_of_the_uniform_range():
    """Each hard-coded (seed, draw, chain, slot, word) of P.EDGE_WORDS still yields its word, and u01_32 of it is
    exactly 1.0 -- the fp32 rounding the GPU edge-word tests drive through the kernels.  u01_32 reaches 1.0 exactly
    from 0xFFFFFF00 up and nowhere else."""
    for name, (seed, draw, chain, slot, word, value) in P.EDGE_WORDS.items():
        got = int(P.block(seed, [chain], draw, slot)[word][0])
        assert got == value, (name, hex(got))
        assert P.u01_32(value) == 1.0, name
    assert P.u01_32(0xFFFFFF00) == 1.0 and P.u01_32(0xFFFFFEFF) < 1.0 and P.u01_32(0) == 2.0 ** -25
    e = P.exp1_words(np.array([0xFFFFFF00, 0xFFFFFFFF, 0x7FFFFFFF, 0x80000000, 0], dtype=np.uint64), exact_log=False)
    assert (e > 0).all() and e[0] == e[1] == np.float32(2.0 ** -25) and e[-1] == np.float32(25 * np.log(2))


# ---------------------------------------------------------------------------------------------------- over-relaxation
def _lattice():
    """All 2^24 values u01_32 takes, sorted (it is non-decreasing in the word)."""
    return P.u01_32(np.arange(1 << 24, dtype=np.uint64) << np.uint64(8))


U0_GRID = [1e-9, 2.0 ** -25, 0.01, 0.3, 0.5 - 2.0 ** -24, 0.5, 0.5 + 2.0 ** -24, 0.7, 0.99, 1 - 1e-9]


def test_binomial_trial_probability_is_u0_within_2_to_the_minus_24():
    """p(u0) = P(u01_32(w) < u0) counted exactly over the lattice, for u0 in fp64 (the fp64 kernels compare in fp64)
    and rounded to fp32 (the fp32 kernels): |p - u0| <= 2^-24 -- the rounding of the top lattice value to 1.0 costs
    no more than that."""
    lat = _lattice()
    for u0 in U0_GRID:
        for x in (np.float64(u0), np.float32(u0)):
            p = np.searchsorted(lat, x, side="left") / 2.0 ** 24
            assert abs(p - float(x)) <= 2.0 ** -24, (u0, x.dtype, p)


@pytest.mark.parametrize("K", [1, 2, 10, 50])
def test_overrelax_r_is_binomial_on_the_lattice_probability(K):
    """The restated r over 20000 chains per u0 against Binomial(K, p(u0)), p(u0) the exact lattice probability
    (chi-square, bins pooled to an expected count of >= 5)."""
    lat = _lattice()
    n = 20000
    for i, u0 in enumerate(U0_GRID):
        p = np.searchsorted(lat, u0, side="left") / 2.0 ** 24
        r, _ = P.overrelax(5, np.arange(n) + (1 << 40), 100 + i, K, np.full(n, u0))
        if p == 0:
            assert (r == 0).all(), u0
            continue
        obs = np.bincount(r, minlength=K + 1)
        exp = n * stats.binom.pmf(np.arange(K + 1), K, p)
        keep = exp >= 5
        if keep.sum() < 2:                           # (almost) all mass in one bin: count the rest directly
            j = int(np.argmax(exp))
            assert n - obs[j] <= stats.poisson.isf(P_MIN, n - exp[j]), (u0, obs)
            continue
        o = np.append(obs[keep], obs[~keep].sum())
        e = np.append(exp[keep], exp[~keep].sum())
        if e[-1] < 5:
            o, e = np.append(o[:-2], o[-2] + o[-1]), np.append(e[:-2], e[-2] + e[-1])
        pv = stats.chisquare(o, e * o.sum() / e.sum()).pvalue
        assert pv > P_MIN, (K, u0, pv, o, e)


BETA_CLASSES = [(1, 10), (2, 8), (3, 6), (4, 4), (5, 2)]      # (na, nb) that K = 10 reaches: r = 0..4 (and 10..6)


def test_overrelax_v_is_beta_for_every_class_k10_reaches():
    """v as the kernel rounds it, for 2^20 chains in each (na, nb) class of K = 10 (r forced to na - 1 < K - r): KS
    against Beta(na, nb).  Left tail of na = 1, down to 1e-7: the counts below 1e-7 .. 1e-3 against their Poisson laws; v is
    never 0 (the exponentials never vanish)."""
    K, n = 10, 1 << 20
    chains = np.arange(n, dtype=np.uint64) + (1 << 33)
    for na, nb in BETA_CLASSES:
        r, v = P.overrelax(21, chains, 7, K, None, exact_log=False, r=np.full(n, na - 1))
        assert na == r[0] + 1 and nb == K - 2 * r[0]
        assert (v > 0).all() and (v < 1).all(), (na, nb)
        pv = stats.kstest(v, stats.beta(na, nb).cdf).pvalue
        assert pv > P_MIN, (na, nb, pv)
        if na == 1:
            for x in (1e-7, 1e-6, 1e-5, 1e-4, 1e-3):
                k, lam = int((v < x).sum()), n * stats.beta(1, nb).cdf(x)
                assert stats.poisson.sf(k - 1, lam) > P_MIN and stats.poisson.cdf(k, lam) > P_MIN, (x, k, lam)


@pytest.mark.parametrize("K", [1, 10, 50])
def test_overrelaxed_uniform_is_uniform_neal_invariance(K):
    """Neal (1998): with u0 ~ U(0, 1), r ~ Binomial(K, u0) and v ~ Beta(na, nb), the over-relaxed
    u' = u0 v (r > K - r), 1 - (1 - u0) v (r < K - r), u0 (r = K - r) is again U(0, 1) -- KS over 2^16 chains."""
    n = 1 << 16
    u0 = np.random.default_rng(K).random(n)
    r, v = P.overrelax(9, np.arange(n) + (1 << 35), (1 << 32) + 3, K, u0, exact_log=False)
    up = np.where(r > K - r, u0 * v, np.where(r < K - r, 1 - (1 - u0) * v, u0))
    pv = stats.kstest(up, "uniform").pvalue
    assert pv > P_MIN, (K, pv)


# ---------------------------------------------------------------------------------------------------- slice
def test_slice_e_is_exponential():
    """e = -log u53 of the Slice kernel: KS against Exp(1) over 2^18 chains; shrinkage uniforms in (0, 1)."""
    n = 1 << 18
    _, e, u0 = P.slice_scalars(3, np.arange(n) + (1 << 36), 12)
    assert stats.kstest(e, "expon").pvalue > P_MIN
    assert stats.kstest(u0, "uniform").pvalue > P_MIN
    for dt in (np.float64, np.float32):
        su = P.slice_shrink_u(3, np.arange(4096), 12, 7, dt)
        assert su.shape == (4096, 7) and (su > 0).all() and (su <= 1).all()
        assert stats.kstest(su.ravel(), "uniform").pvalue > P_MIN
