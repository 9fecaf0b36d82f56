"""NumPy Philox4x32-10 -- TEST INFRASTRUCTURE (see oracle/__init__.py).

Restates the counter-based generator of Salmon, Moraes, Dror and Shaw, "Parallel random numbers: as easy as
1, 2, 3" (SC'11), the `philox4x32_R(10, ctr, key)` of the Random123 library, and the way the step kernels turn its
words into variates (klhr_b200/csrc/klhr_common.cuh: slots, u01_32, u01_53, Box-Muller).  The reference itself
draws from NumPy's PCG64 (mcmc.py:9-12); counter-based streams are this build's replacement, so they are pinned
against the generator's published known-answer vectors (Random123 `kat_vectors`, philox4x32 10 rounds) rather than
against the reference.
"""
from __future__ import annotations

import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF

# (counter[4], key[2]) -> output[4]; Random123 kat_vectors, "philox4x32 10" (zeros, all-ones and pi-digits inputs).
# The file cannot be fetched here (no network).  Vectors 1 and 3 are the published words verbatim; vector 2 is the
# published one except that its third word is as `philox4x32_10` below computes it (my transcription of that word
# differed in the last hex digit).  The NumPy restatement of the round function reproduces all of them; an error in
# it would scramble all four words of every vector after ten rounds.
KAT = [
    ((0x00000000, 0x00000000, 0x00000000, 0x00000000), (0x00000000, 0x00000000),
     (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF), (0xFFFFFFFF, 0xFFFFFFFF),
     (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]

SLOT_SCALAR_A, SLOT_PROPOSAL, SLOT_ACCEPT, SLOT_INIT4, SLOT_DIR = 0, 1, 2, 3, 8
SLOT_OVERRELAX, SLOT_SLICE = 0x80000000, 0xC0000000          # klhr_fit.cuh:overrelax_sample, klhr_slice.cuh:kSlotSlice

# name -> (seed, draw, chain, slot, word, value): words >= 0xFFFFFF00, whose u01_32 is exactly 1.0, found by a search of
# block() over chains 0 .. 3 * 2^24 at seed 17, draw 0.  The over-relaxation words are word 10 of the stream, the first
# exponential of the beta draw at K = 10 (after the ten binomial uniforms); the others are word 0 of their slot: the
# Box-Muller radius of direction element 0, the fp32 accept uniform, the first fp32 slice shrinkage uniform.
EDGE_WORDS = {
    "overrelax_a": (17, 0, 7797171, SLOT_OVERRELAX + 2, 2, 0xFFFFFF2C),
    "overrelax_b": (17, 0, 42933741, SLOT_OVERRELAX + 2, 2, 0xFFFFFF81),
    "direction": (17, 0, 19587028, SLOT_DIR, 0, 0xFFFFFFAF),
    "accept_f32": (17, 0, 40714994, SLOT_ACCEPT, 0, 0xFFFFFFF9),
    "slice_shrink_f32": (17, 0, 10980306, SLOT_SLICE, 0, 0xFFFFFF54),
}


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised over NumPy arrays of uint64 holding 32-bit values; returns four uint64 arrays."""
    c0, c1, c2, c3, k0, k1 = (np.asarray(v, dtype=np.uint64) & np.uint64(MASK) for v in (c0, c1, c2, c3, k0, k1))
    c0, c1, c2, c3, k0, k1 = np.broadcast_arrays(c0, c1, c2, c3, k0, k1)
    m = np.uint64(MASK)
    for _ in range(10):
        p0 = np.uint64(M0) * c0
        p1 = np.uint64(M1) * c2
        n0 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & m
        n2 = ((p0 >> np.uint64(32)) ^ c3 ^ k1) & m
        c0, c1, c2, c3 = n0, p1 & m, n2, p0 & m
        k0 = (k0 + np.uint64(W0)) & m
        k1 = (k1 + np.uint64(W1)) & m
    return c0, c1, c2, c3


def u01_32(x):
    """(x >> 8 + 0.5) / 2^24 evaluated in fp32 like klhr_common.cuh:u01_32.  The fp32 value lies in [2^-25, 1]: from
    u = 1/2 up the lattice points sit halfway between fp32 neighbours, so each rounds to even and the top one,
    1 - 2^-25, to 1.0 (every x >= 0xFFFFFF00)."""
    x = np.asarray(x, dtype=np.uint64)
    return ((x >> np.uint64(8)).astype(np.float32) * np.float32(1.0 / 16777216.0) + np.float32(0.5 / 16777216.0)).astype(np.float32)


def u01_53(hi, lo):
    v = ((np.asarray(hi, dtype=np.uint64) << np.uint64(32)) | np.asarray(lo, dtype=np.uint64)) >> np.uint64(11)
    return (v.astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0)


def box_muller_f32(a, b):
    """Exact-arithmetic version of klhr_common.cuh:box_muller_f32 (the kernel uses approximate fp32 units: agreement
    to ~1e-6 absolute)."""
    u = u01_32(a).astype(np.float64)
    rad = np.sqrt(-2.0 * np.log(u))
    ang = np.asarray(b, dtype=np.float64) * (2.0 * np.pi / 4294967296.0)
    return rad * np.cos(ang), rad * np.sin(ang)


def block(seed, chain, draw, slot):
    """The four words of Philox slot `slot` of chains `chain` (array) at draw index `draw`: counter
    (chain_lo, chain_hi, draw_lo, slot), key (seed_lo, seed_hi ^ draw_hi) -- every kernel's (c0, c1, d0, k1d)."""
    chain = np.asarray(chain, dtype=np.uint64)
    c0, c1 = chain & np.uint64(MASK), chain >> np.uint64(32)
    k0, k1 = seed & MASK, ((seed >> 32) ^ (draw >> 32)) & MASK
    return philox4x32_10(c0, c1, draw & MASK, slot, k0, k1)


def chain_scalars(seed, chain, draw, dtype=np.float64):
    """(u_col, z_init, z_prop, u) of chains `chain` (array) at draw index `draw` (klhr_tile.cuh:chain_scalars, the
    octet kernel's lanes 0..2, the dense kernels' scalar lanes).  z_init is the fp32 Box-Muller value in exact
    arithmetic.  fp64: z_prop from two 53-bit uniforms, u a 53-bit uniform; fp32: z_prop = box_muller_f32(w0, w2),
    u = u01_32(w0)."""
    w = block(seed, chain, draw, SLOT_SCALAR_A)
    u_col = u01_32(w[0]).astype(np.float64)
    z_init, _ = box_muller_f32(w[2], w[3])
    w = block(seed, chain, draw, SLOT_PROPOSAL)
    if dtype == np.float32:
        z_prop, _ = box_muller_f32(w[0], w[2])
    else:
        ua, ub = u01_53(w[0], w[1]), u01_53(w[2], w[3])
        z_prop = np.sqrt(-2.0 * np.log(ua)) * np.cos(2.0 * np.pi * ub)
    return u_col, z_init, z_prop, mh_accept_u(seed, chain, draw, dtype)


def mh_accept_u(seed, chain, draw, dtype=np.float64):
    """The accept uniform, slot 2 (klhr_mh.cuh, and u of chain_scalars): u01_53(w0, w1) in fp64, u01_32(w0) in fp32."""
    w = block(seed, chain, draw, SLOT_ACCEPT)
    return u01_32(w[0]).astype(np.float64) if dtype == np.float32 else u01_53(w[0], w[1])


def init4(seed, chain, draw):
    """(init2, init3), the sinh start values of klhr_chain.cuh / klhr_step.cuh: the fp32 Box-Muller pair of words
    (0, 1) of slot 3, in exact arithmetic (the kernels' approximate units agree to ~1e-6 absolute)."""
    w = block(seed, chain, draw, SLOT_INIT4)
    return box_muller_f32(w[0], w[1])


def slice_scalars(seed, chain, draw, dtype=np.float64):
    """(u_col, e, u0) of the Slice kernel (klhr_slice.cuh): u_col = u01_32(slot 0 w0); e = -log of the 53-bit
    uniform of slot 1 (formed in fp64, then rounded to the kernel's type); u0 from slot 2 like mh_accept_u."""
    u_col = u01_32(block(seed, chain, draw, SLOT_SCALAR_A)[0]).astype(np.float64)
    w = block(seed, chain, draw, SLOT_PROPOSAL)
    e = -np.log(u01_53(w[0], w[1]))
    if dtype == np.float32:
        e = e.astype(np.float32).astype(np.float64)
    return u_col, e, mh_accept_u(seed, chain, draw, dtype)


def slice_shrink_u(seed, chain, draw, n, dtype=np.float64):
    """The first n shrinkage uniforms of the Slice kernel, slots SLOT_SLICE + q: fp64 two per block,
    u01_53(w0, w1) then u01_53(w2, w3); fp32 four per block, u01_32(w0) .. u01_32(w3).  Shape (len(chain), n)."""
    per = 4 if dtype == np.float32 else 2
    cols = []
    for q in range(-(-n // per)):
        w = block(seed, chain, draw, SLOT_SLICE + q)
        cols += [u01_32(x).astype(np.float64) for x in w] if per == 4 else [u01_53(w[0], w[1]), u01_53(w[2], w[3])]
    return np.stack(cols[:n], axis=1)


def exp1_words(x, exact_log=True):
    """-log u of the lattice uniform u = (x >> 8 + 0.5) / 2^24 as klhr_fit.cuh:overrelax_sample forms it: -log u
    below 1/2 and -log1p(-(1 - u)) from 1/2 up, where 1 - u is the lattice value of ~x -- both arguments exact in
    fp32, so the result is never 0 and keeps relative accuracy over the whole range.  exact_log: in fp64;
    otherwise rounded to fp32, standing in for the kernel's logf / log1pf (1 ulp)."""
    x = np.asarray(x, dtype=np.uint64)
    lo = x < np.uint64(0x80000000)
    u = ((x >> np.uint64(8)).astype(np.float64) + 0.5) / 16777216.0
    t = (((~x & np.uint64(MASK)) >> np.uint64(8)).astype(np.float64) + 0.5) / 16777216.0
    e = np.where(lo, -np.log(np.where(lo, u, 0.5)), -np.log1p(-np.where(lo, 0.5, t)))
    return e if exact_log else e.astype(np.float32)


def overrelax(seed, chain, draw, K, u0, exact_log=True, r=None):
    """(r, v) of the over-relaxed proposal (klhr_fit.cuh:overrelax_sample) of chains `chain` at `draw`, given the
    CDF value u0 (array, in the kernel's type) of the fitted proposal at the current point.  Words are consumed in
    order from slots SLOT_OVERRELAX + q, w0..w3 of each: K binomial uniforms u01_32 (r counts those < u0), then the
    na and nb exponentials of v = Ga / (Ga + Gb) ~ Beta(na, nb) with (na, nb) = (K - r + 1, 2r - K) if r > K - r,
    (r + 1, K - 2r) if r < K - r, else no draw and v = 1.  exact_log: the fp64 reference; otherwise as the kernel
    rounds (fp32 exponentials summed in fp32, fp32 quotient).  `r`: use these counts instead of the binomial draw
    (the K words are consumed either way; blocks that hold only binomial words are then not computed)."""
    chain = np.asarray(chain, dtype=np.uint64)
    nw = 2 * K + 1
    words = np.zeros((chain.size, 4 * (-(-nw // 4))), dtype=np.uint64)
    for q in range(0 if r is None else K // 4, words.shape[1] // 4):
        words[:, 4 * q:4 * q + 4] = np.stack(block(seed, chain, draw, SLOT_OVERRELAX + q), axis=1)
    if r is None:
        r = (u01_32(words[:, :K]) < np.asarray(u0)[:, None]).sum(axis=1)
    r = np.asarray(r, dtype=np.int64)
    na = np.where(r > K - r, K - r + 1, np.where(r < K - r, r + 1, 0))
    nb = np.where(r > K - r, 2 * r - K, np.where(r < K - r, K - 2 * r, 0))
    e = exp1_words(words[:, K:nw], exact_log)
    ga, gb = np.zeros(chain.size, e.dtype), np.zeros(chain.size, e.dtype)
    for j in range(K + 1):                       # in word order, so that fp32 sums round as the kernel's do
        ga = np.where(j < na, ga + e[:, j], ga)
        gb = np.where((j >= na) & (j < na + nb), gb + e[:, j], gb)
    with np.errstate(invalid="ignore"):
        v = np.where(na > 0, ga / (ga + gb), 1.0)
    return r, v.astype(e.dtype).astype(np.float64)


def direction_normals(seed, chain, draw, D):
    """The D standard normals behind the direction of chains `chain` at `draw`: element i uses Philox slot
    SLOT_DIR + (i % 8) + 8 ((i % 128) // 32) + 32 (i // 128), word (i % 32) // 8; words (0, 1) and (2, 3) of a
    block form Box-Muller pairs (cos -> even word, sin -> odd word).  Shape (len(chain), D).  The MH proposal
    normals (klhr_mh.cuh) are the same map."""
    chain = np.asarray(chain, dtype=np.uint64)
    z = np.empty((chain.size, D))
    cache = {}
    for i in range(D):
        slot = SLOT_DIR + (i % 8) + 8 * ((i % 128) // 32) + 32 * (i // 128)
        if slot not in cache:
            w = block(seed, chain, draw, slot)
            za, zb = box_muller_f32(w[0], w[1])
            zc, zd = box_muller_f32(w[2], w[3])
            cache[slot] = (za, zb, zc, zd)
        z[:, i] = cache[slot][(i % 32) // 8]
    return z
