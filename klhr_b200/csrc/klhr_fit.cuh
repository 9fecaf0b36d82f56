// klhr_b200 -- the line fit (reference KLHR.fit klhr.py:126-141, KLHRSINH.fit
// klhr_sinh.py:182-201) with scipy.optimize.minimize replaced by a fixed-budget damped
// Newton iteration, and the Metropolis-Hastings pieces (klhr.py:155-158,175-190,
// klhr_sinh.py:112-114,233-260).  Mirrors oracle/batched.py operation for operation.
//
// Every function is templated on the group size G that cooperates on ONE chain:
//   G = 8  the 8 lanes of an octet call together; lane n owns quadrature node n (n, n+8, ..)
//          and back-tracking candidate n; sums are 3-level xor-shuffles; results are uniform
//          across the octet (klhr_step.cuh);
//   G = 1  a single thread owns the chain and loops over nodes / candidates itself, no
//          shuffles (klhr_tile.cuh, thread-per-chain fit).
// Both produce the same iterates up to the summation order of the quadrature sums.
#pragma once
#include "klhr_common.cuh"

namespace klhr {
struct ModelParams;

struct FitParams {
    int family;            // KLHR_FAMILY_GAUSS | KLHR_FAMILY_SINH
    int N;                 // quadrature nodes (<= kMaxNodes)
    int n1, n2, nb;        // stage-1 iterations, stage-2 Newton steps, halvings per step
    int kmax;              // cap on stage-2 KL evaluations
    int or_K;              // > 0: over-relaxed proposal with K trials (klhr.py:160-173)
    int fix_d;             // sinh family with d = 1 frozen (sub_klhr_sinh.py)
    double initscale, tol, scale_clip;
    double gtol1, gtol2, step_cap, c1, basin;
    double grad_clip;      // > 0: elementwise clip of the model gradient inside the sinh-family KL (klhr_sinh.py:158-161)
    double x[kMaxNodes], w[kMaxNodes], cx[kMaxNodes];   // nodes, weights, asinh(nodes)
};

constexpr double kNewtonCapD = 64.0;

// ------------------------------------------------------------------ stage 1: 1-D mode search
// A Newton step may be at most kNewtonCap trust radii long (oracle/batched.py:NEWTON_CAP): the candidates
// step * 2^-k are scored by l, so a long step is only taken when it is the best point, and the exact Newton
// step of a quadratic target gets through in ONE iteration at the posterior scales of the benchmark targets.
template <int G, typename R, typename Model>
__device__ void stage1_mode(const typename Model::Coef& cf, R z_init, const FitParams& fp, int lane,
                            unsigned m, R& xi_out, R& tau0_out, int& nev) {
    R xi = z_init * (R)fp.initscale;
    R trust = 1;
    bool done = false;
    Jet<R> J = Model::eval(cf, xi);
    nev = 1;
    const R gt1sq = (R)fp.gtol1 * (R)fp.gtol1;
    const unsigned wm = __activemask();
    for (int it = 0; it < fp.n1; ++it) {
        const bool concave = J.l2 < R(0);
        // |l'| / sqrt(-l'') <= gtol1, written without the square root and the division
        const bool conv = concave && (J.l1 * J.l1 <= gt1sq * (-J.l2));
        done = done || conv || !r_finite(J.l);
        if (!__any_sync(wm, !done)) break;      // lock-step: finished chains idle, nobody serialises
        if (done) continue;
        const R newton = concave ? -J.l1 / J.l2 : R(0);
        const R step = concave ? r_clamp(newton, -(R)kNewtonCapD * trust, (R)kNewtonCapD * trust) : r_clamp(J.l1, -trust, trust);
        nev += kOct;
        // the 8 candidates xi + 2^-k step: keep the arg-max of l, first maximum on ties
        R bv, bx, b1, b2;
        int bi;
        if constexpr (G == kOct) {
            const R cand = xi + step * ((R)1 / (R)(1 << lane));
            const Jet<R> C = Model::eval(cf, cand);
            bv = C.l;
            bi = lane;
#pragma unroll
            for (int off = 1; off < kOct; off <<= 1) {
                const R ov = __shfl_xor_sync(m, bv, off);
                const int oi = __shfl_xor_sync(m, bi, off);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            bx = oct_bcast(cand, bi, m);
            b1 = oct_bcast(C.l1, bi, m);
            b2 = oct_bcast(C.l2, bi, m);
        } else {
            bv = -Num<R>::inf(); bi = 0; bx = xi; b1 = 0; b2 = 0;
            R ks = 1;
#pragma unroll
            for (int k = 0; k < kOct; ++k) {
                const R cand = xi + step * ks;
                const Jet<R> C = Model::eval(cf, cand);
                if (C.l > bv) { bv = C.l; bi = k; bx = cand; b1 = C.l1; b2 = C.l2; }
                ks *= R(0.5);
            }
        }
        const bool improve = bv > J.l;
        const bool full = improve && bi == 0;
        if (improve) {
            xi = bx;
            J.l = bv;
            J.l1 = b1;
            J.l2 = b2;
        }
        trust = full ? trust * R(2) : (improve ? trust : trust * R(1.0 / 256.0));
        done = done || (!improve && (r_abs(step) * R(1.0 / 128.0) <= Num<R>::eps * (R(1) + r_abs(xi))));
    }
    xi_out = xi;
    tau0_out = (J.l2 < R(0)) ? -R(0.5) * r_log(-J.l2) : R(0);
}

// ------------------------------------------------------------------ small dense algebra
template <typename R, int n>
struct KLState {
    R f;
    R g[n];
    R H[n][n];          // full symmetric storage (n = 2 or 4)
    R s;                // the family's scale at the evaluated eta (saves recomputing exp(eta_1) for the proposal)
};

// Solve (H) p = -g by Cholesky, entry by entry like oracle/batched.py:_chol_solve.
template <typename R, int n>
__device__ __forceinline__ bool chol_solve(const R (&H)[n][n], R shift, const R (&g)[n], R (&p)[n]) {
    // one reciprocal square root per pivot, multiplications everywhere else: the diagonal of L is never needed, only
    // its reciprocal (sqrt followed by a division was a quarter of the dependent-latency chain of a Newton step)
    R L[n][n], iL[n];
    bool ok = true;
#pragma unroll
    for (int j = 0; j < n; ++j) {
        R acc = H[j][j] + shift;
#pragma unroll
        for (int k = 0; k < j; ++k) acc = acc - L[j][k] * L[j][k];
        ok = ok && (acc > R(0));
        iL[j] = r_rsqrt(acc > R(0) ? acc : R(1));
#pragma unroll
        for (int i = j + 1; i < n; ++i) {
            R a2 = H[i][j];
#pragma unroll
            for (int k = 0; k < j; ++k) a2 = a2 - L[i][k] * L[j][k];
            L[i][j] = a2 * iL[j];
        }
    }
    R y[n];
#pragma unroll
    for (int i = 0; i < n; ++i) {
        R acc = -g[i];
#pragma unroll
        for (int k = 0; k < i; ++k) acc = acc - L[i][k] * y[k];
        y[i] = acc * iL[i];
    }
#pragma unroll
    for (int i = n - 1; i >= 0; --i) {
        R acc = y[i];
#pragma unroll
        for (int k = i + 1; k < n; ++k) acc = acc - L[k][i] * p[k];
        p[i] = acc * iL[i];
    }
#pragma unroll
    for (int i = 0; i < n; ++i) ok = ok && r_finite(p[i]);
    return ok;
}

template <typename R, int n>
__device__ __forceinline__ void newton_direction(const KLState<R, n>& S, const FitParams& fp, R (&p)[n]) {
    R mu = 0;
#pragma unroll
    for (int i = 0; i < n; ++i) mu = r_max(mu, r_abs(S.H[i][i]));   // NaN-safe: comparisons drop NaN
    bool mu_ok = true;
#pragma unroll
    for (int i = 0; i < n; ++i) mu_ok = mu_ok && r_finite(S.H[i][i]);
    if (!(mu_ok && mu > R(0))) mu = R(1);
    // Levenberg shifts (x mu): 0, 1e-3, 1e-2, 1e-1, 1, 10, 100, 1e3, 1e4, 1e6 -- same list as
    // oracle/batched.py:LM_SHIFTS; generated arithmetically to keep the table out of local memory
    bool have = false;
    R shift = R(0);
    for (int k = 0; k < 10 && !have; ++k) {
        R pk[n];
        if (chol_solve<R, n>(S.H, shift * mu, S.g, pk)) {
            have = true;
#pragma unroll
            for (int i = 0; i < n; ++i) p[i] = pk[i];
        }
        shift = k == 0 ? R(1e-3) : (k == 8 ? R(1e6) : shift * R(10));
    }
    if (!have) {
#pragma unroll
        for (int i = 0; i < n; ++i) p[i] = -S.g[i];
    }
    R big = 0;
#pragma unroll
    for (int i = 0; i < n; ++i) {
        if (!r_finite(p[i])) p[i] = R(0);
        big = r_max(big, r_abs(p[i]));
    }
    const R cap = (R)fp.step_cap;
    if (big > cap) {                               // rare: keeps the division off the common path
        const R scale = cap / big;
#pragma unroll
        for (int i = 0; i < n; ++i) p[i] = p[i] * scale;
    }
}

// ------------------------------------------------------------------ KL objective, Gaussian family
// reference klhr.py:106-120 in scaled coordinates (m/s, tau); Hessian from l''.
template <int G, typename R, typename Model>
__device__ void kl_gauss(const typename Model::Coef& cf, const R (&eta)[2], const FitParams& fp, int lane,
                         unsigned m, KLState<R, 2>& S) {
    const R clip = (R)fp.scale_clip;
    const R s = r_exp(r_clamp(eta[1], -clip, clip));
    R S0 = 0, S1 = 0, S1x = 0, S2 = 0, S2x = 0, S2xx = 0;
    for (int n = lane; n < fp.N; n += G) {
        const R x = (R)fp.x[n], w = (R)fp.w[n];
        const R y = s * x + eta[0];
        const Jet<R> J = Model::eval(cf, y);
        S0 += w * J.l;
        const R w1 = w * J.l1;
        S1 += w1;
        S1x += w1 * x;
        const R w2 = w * J.l2;
        S2 += w2;
        S2x += w2 * x;
        S2xx += w2 * x * x;
    }
    S0 = grp_sum<G>(S0, m); S1 = grp_sum<G>(S1, m); S1x = grp_sum<G>(S1x, m);
    S2 = grp_sum<G>(S2, m); S2x = grp_sum<G>(S2x, m); S2xx = grp_sum<G>(S2xx, m);
    const R s2 = s * s;
    S.s = s;
    S.f = -(S0 + eta[1]);
    S.g[0] = -S1 * s;
    S.g[1] = -(S1x * s + R(1));
    S.H[0][0] = -S2 * s2;
    S.H[0][1] = S.H[1][0] = -S2x * s2;
    S.H[1][1] = -(S2xx * s2 + S1x * s);
}

// ------------------------------------------------------------------ elementwise gradient clip (sinh family)
// The reference's KLHRSINH.KL projects np.clip(grad lp, -c, c) on rho (klhr_sinh.py:158-161,171-173) -- a clip of
// every COMPONENT of the model gradient, which the O(1) line restriction cannot see.  Where Model::eval_mc says a
// component may exceed c at theta + y rho, the full gradient is formed there by one thread (Model::lp_grad<1>,
// D <= kClipMaxD) and l'(y) is replaced by sum_i clip(g_i) rho_i; evaluations on which nothing is clipped keep the
// closed-form l'.  l'' (the Newton matrix) stays that of the unclipped density: same fixed points, and the
// iteration is restated in oracle/batched.py with the same rule.
// grad_clip applies to the sinh family only (klhr.py:106-120 does not clip) and to targets of at most kClipMaxD dims
template <typename R>
__device__ __forceinline__ ClipCtx<R> clip_ctx(const FitParams& fp, const ModelParams& mp, int D, const R* th, const R* rh) {
    ClipCtx<R> cc = clip_off<R>();
    if (fp.family == 1 && fp.grad_clip > 0.0 && fp.grad_clip < 1e300 && D <= kClipMaxD) {
        cc.c = (R)fp.grad_clip; cc.th = th; cc.rh = rh; cc.mp = &mp; cc.D = D;
    }
    return cc;
}

// (jet, clipped l') of the line restriction at y
template <typename R, typename Model>
__device__ __forceinline__ Jet<R> eval_clipped(const typename Model::Coef& cf, R y, const ClipCtx<R>& cc, R& l1c) {
    if (!cc.on()) {
        const Jet<R> J = Model::eval(cf, y);
        l1c = J.l1;
        return J;
    }
    return Model::eval_clip(cf, y, cc, l1c);
}

// ------------------------------------------------------------------ sinh-arcsinh family
template <typename R>
struct SinhPar { R m, s, d, e; };

template <typename R>
__device__ __forceinline__ SinhPar<R> sinh_unpack(const R (&eta)[4], const FitParams& fp) {   // klhr_sinh.py:78-84
    const R c = (R)fp.scale_clip, tol = (R)fp.tol;
    SinhPar<R> q;
    q.m = eta[0];
    q.s = r_exp(r_clamp(eta[1], -c, c)) + tol;
    q.d = fp.fix_d ? R(1) : r_exp(r_clamp(eta[2], -c, c)) + tol;      // sub_klhr_sinh.py:92-97: no d
    q.e = eta[3];
    return q;
}

// reference klhr_sinh.py:163-176; gradients are _grad_T (:116-124) and _grad_log_abs_jac
// (:146-156); second derivatives are those expressions differentiated once more.
template <int G, typename R, typename Model>
__device__ void kl_sinh(const typename Model::Coef& cf, const R (&eta)[4], const FitParams& fp, int lane,
                        unsigned m, KLState<R, 4>& S, const ClipCtx<R>& cc) {
    const SinhPar<R> q = sinh_unpack<R>(eta, fp);
    const R c = (R)fp.scale_clip;
    const R invd = R(1) / q.d;
    R f = 0, g1 = 0, g2 = 0, g3 = 0, g0 = 0;
    R h00 = 0, h01 = 0, h02 = 0, h03 = 0, h11 = 0, h12 = 0, h13 = 0, h22 = 0, h23 = 0, h33 = 0;
    // not unrolled on purpose: two nodes in flight cost more in registers (spills at the 128-register budget of the chain
    // kernel, fewer resident warps above it) than their overlap returns (measured, DESIGN.md section 7)
#pragma unroll 1
    for (int n = lane; n < fp.N; n += G) {
        const R w = (R)fp.w[n];
        const R a = ((R)fp.cx[n] + q.e) * invd;
        const R ac = r_clamp(a, -c, c);
        // sinh, cosh, tanh and log cosh from ONE exponential (|ac| <= scale_clip = 300 keeps e^ac
        // finite in fp64); absolute accuracy ~1 ulp of cosh, which is what T and the KL sums need
        // e^-ac and tanh through Newton reciprocals of e^ac and cosh (e^-300 <= e^ac <= e^300, 1 <= cosh <= e^300 / 2: no
        // special cases to guard) instead of IEEE divisions (~25 dependent instructions each); a second exponential for
        // e^-ac overlaps with the first but costs 35 more instructions per node: measured 6 % slower
        const R E = r_exp(ac), Ei = r_rcp_normal(E);
        const R sh = R(0.5) * (E - Ei), ch = R(0.5) * (E + Ei);
        const R th = sh * r_rcp_normal(ch);
        const R sech2 = R(1) - th * th;
        const R T = q.m + q.s * sh;
        R l1c;                                                                    // l' with the elementwise clip
        const Jet<R> J = eval_clipped<R, Model>(cf, T, cc, l1c);
        const R logJ = (eta[2] - eta[1]) - r_log(ch);
        f += w * (logJ - J.l);
        const R t1 = q.s * sh, t2 = -q.s * ch * a, t3 = q.s * ch * invd;          // grad T (t0 = 1)
        const R L2 = R(1) + th * a, L3 = -th * invd;                              // grad log|J| (L0 = 0, L1 = -1)
        g0 += w * (-l1c);
        g1 += w * (-R(1) - l1c * t1);
        g2 += w * (L2 - l1c * t2);
        g3 += w * (L3 - l1c * t3);
        const R T11 = q.s * sh, T12 = -q.s * a * ch, T13 = q.s * ch * invd;
        const R T22 = q.s * a * ch + q.s * a * a * sh;
        const R T23 = -(q.s * invd) * (ch + a * sh);
        const R T33 = q.s * sh * invd * invd;
        const R L22 = -a * th - a * a * sech2;
        const R L23 = (th + a * sech2) * invd;
        const R L33 = -sech2 * invd * invd;
        h00 += w * (-J.l2);
        h01 += w * (-J.l2 * t1);
        h02 += w * (-J.l2 * t2);
        h03 += w * (-J.l2 * t3);
        h11 += w * (-J.l2 * t1 * t1 - l1c * T11);
        h12 += w * (-J.l2 * t1 * t2 - l1c * T12);
        h13 += w * (-J.l2 * t1 * t3 - l1c * T13);
        h22 += w * (L22 - J.l2 * t2 * t2 - l1c * T22);
        h23 += w * (L23 - J.l2 * t2 * t3 - l1c * T23);
        h33 += w * (L33 - J.l2 * t3 * t3 - l1c * T33);
    }
    S.f = grp_sum<G>(f, m);
    g0 = grp_sum<G>(g0, m); g1 = grp_sum<G>(g1, m); g2 = grp_sum<G>(g2, m); g3 = grp_sum<G>(g3, m);
    h00 = grp_sum<G>(h00, m); h01 = grp_sum<G>(h01, m); h02 = grp_sum<G>(h02, m); h03 = grp_sum<G>(h03, m);
    h11 = grp_sum<G>(h11, m); h12 = grp_sum<G>(h12, m); h13 = grp_sum<G>(h13, m);
    h22 = grp_sum<G>(h22, m); h23 = grp_sum<G>(h23, m); h33 = grp_sum<G>(h33, m);
    if (fp.fix_d) {                    // d frozen: its row and column drop out of the Newton system
        g2 = 0; h02 = 0; h12 = 0; h23 = 0; h22 = 1;
    }
    const R s = q.s;
    S.s = s;
    S.g[0] = g0 * s; S.g[1] = g1; S.g[2] = g2; S.g[3] = g3;
    S.H[0][0] = h00 * s * s;
    S.H[0][1] = S.H[1][0] = h01 * s;
    S.H[0][2] = S.H[2][0] = h02 * s;
    S.H[0][3] = S.H[3][0] = h03 * s;
    S.H[1][1] = h11; S.H[1][2] = S.H[2][1] = h12; S.H[1][3] = S.H[3][1] = h13;
    S.H[2][2] = h22; S.H[2][3] = S.H[3][2] = h23; S.H[3][3] = h33;
}

template <int G, typename R, typename Model, int n>
__device__ __forceinline__ void kl_eval(const typename Model::Coef& cf, const R (&eta)[n], const FitParams& fp,
                                        int lane, unsigned m, KLState<R, n>& S, const ClipCtx<R>& cc) {
    if constexpr (n == 2) kl_gauss<G, R, Model>(cf, eta, fp, lane, m, S);
    else kl_sinh<G, R, Model>(cf, eta, fp, lane, m, S, cc);
}

template <typename R, int n>
__device__ __forceinline__ R scale_of(const R (&eta)[n], const FitParams& fp) {
    const R c = (R)fp.scale_clip;
    const R s = r_exp(r_clamp(eta[1], -c, c));
    return n == 4 ? s + (R)fp.tol : s;
}

// ------------------------------------------------------------------ stage 2: damped Newton on KL
// Written as a lock-step state machine: every trip of the ONE loop performs exactly one KL
// evaluation (the expensive, uniform part) for every chain of the warp, followed by a short
// per-chain decision (accept / halve / new Newton direction).  The per-chain sequence of
// evaluations is exactly the nested loop of oracle/batched.py:stage2_newton, but chains that
// sit in different phases (back-tracking vs. new direction) no longer serialise each other:
// with 4 octets (or 32 single-thread chains) per warp the nested form ran one group at a time.
template <int G, typename R, typename Model, int n>
__device__ void stage2_newton(const typename Model::Coef& cf, R (&eta)[n], const FitParams& fp, int lane,
                              unsigned m, int& nev, bool& converged, R& s_out, const ClipCtx<R>& cc) {
    const unsigned wm = __activemask();        // the lanes that entered together stay in lock-step
    R S_f = 0, S_s = 1;        // objective and family scale at the last accepted point (its gradient and Hessian are used up
                               // in the trip that accepts it: nothing else of the 22-double KLState has to be carried)
    R p[n], trial[n];
#pragma unroll
    for (int i = 0; i < n; ++i) { trial[i] = eta[i]; p[i] = 0; }
    R gp = 0, t = 1, s_cur = 1;
    bool have_S = false, done = false, conv = false, in_basin = false;
    int it = 0, bt = 0, slow = 0;
    R g_prev = Num<R>::inf();
    nev = 0;
    const int max_evals = fp.kmax;
    for (int k = 0; k < max_evals; ++k) {
        if (!__any_sync(wm, !done)) break;
        KLState<R, n> St;
        kl_eval<G, R, Model, n>(cf, trial, fp, lane, m, St, cc);
        if (!done) {
            nev += 1;
            bool accepted;
            if (!have_S) {
                accepted = true;
                have_S = true;
            } else {
                const R slack = R(8) * Num<R>::eps * (R(1) + r_abs(S_f));
                accepted = r_finite(St.f) &&
                           ((St.f <= S_f + (R)fp.c1 * t * gp + slack) || !r_finite(S_f) || in_basin);
            }
            if (accepted) {
#pragma unroll
                for (int i = 0; i < n; ++i) eta[i] = trial[i];
                S_f = St.f;
                S_s = St.s;
                R gmax = 0;
                bool gnan = false;
#pragma unroll
                for (int i = 0; i < n; ++i) {
                    gmax = r_max(gmax, r_abs(St.g[i]));
                    gnan = gnan || (St.g[i] != St.g[i]);
                }
                // flat valley: inside the basin a Newton step must at least halve the gradient; two in
                // a row that do not -> stop (see oracle/batched.py:stage2_newton)
                const bool lag = in_basin && !(gmax <= R(0.5) * g_prev);
                slow = lag ? slow + 1 : 0;
                if (!gnan && gmax <= (R)fp.gtol2) {
                    conv = true;
                    done = true;
                } else if (it >= fp.n2 || slow >= 2) {
                    done = true;                   // Newton-step budget exhausted, or flat valley
                } else {
                    g_prev = gmax;
                    newton_direction<R, n>(St, fp, p);
                    gp = 0;
#pragma unroll
                    for (int i = 0; i < n; ++i) gp += St.g[i] * p[i];
                    if (!r_finite(gp)) gp = 0;
                    s_cur = St.s;                  // = scale_of(eta): the evaluation formed it with the same operations
                    in_basin = !gnan && gmax <= (R)fp.basin;
                    t = 1;
                    bt = 0;
                    it += 1;
                }
            } else {
                t *= R(0.5);
                bt += 1;
                if (bt >= fp.nb) done = true;      // stalled: keep the current iterate
            }
            if (!done) {
                trial[0] = eta[0] + t * p[0] * s_cur;
#pragma unroll
                for (int i = 1; i < n; ++i) trial[i] = eta[i] + t * p[i];
            }
        }
    }
    converged = conv;
    s_out = S_s;               // scale at the returned eta (the last accepted evaluation)
}

// ------------------------------------------------------------------ family densities / transport
template <typename R>
__device__ __forceinline__ R logq_gauss(R x, const R (&eta)[2], const FitParams& fp) {          // klhr.py:155-158
    const R c = (R)fp.scale_clip;
    const R s = r_exp(r_clamp(eta[1], -c, c));
    const R z = (x - eta[0]) / s;
    return -r_log(s) - R(0.5) * z * z;
}

template <typename R>
__device__ __forceinline__ R transport_sinh(R z, const R (&eta)[4], const FitParams& fp) {       // klhr_sinh.py:112-114
    const SinhPar<R> q = sinh_unpack<R>(eta, fp);
    const R c = (R)fp.scale_clip;
    return q.m + q.s * r_sinh(r_clamp((r_asinh(z) + q.e) / q.d, -c, c));
}

template <typename R>
__device__ __forceinline__ R logq_sinh(R x, const R (&eta)[4], const FitParams& fp) {            // klhr_sinh.py:233-240
    const SinhPar<R> q = sinh_unpack<R>(eta, fp);
    const R c = (R)fp.scale_clip;
    const R z = (x - q.m) / q.s;
    const R b = r_clamp(q.d * r_asinh(z) - q.e, -c, c);
    const R ti = r_sinh(b);
    return -R(0.5) * ti * ti + r_log(r_cosh(b)) + eta[2] - eta[1] - R(0.5) * r_log1p(z * z);
}

// ------------------------------------------------------------------ fit + proposal + MH ratio
template <typename R>
struct StepOut {
    R eta[4];
    R zp, r;
    bool accept, converged;
    int evals;
};

__device__ __forceinline__ double r_normcdf(double x) { return normcdf(x); }
__device__ __forceinline__ float r_normcdf(float x) { return normcdff(x); }
__device__ __forceinline__ double r_normcdfinv(double x) { return normcdfinv(x); }
__device__ __forceinline__ float r_normcdfinv(float x) { return normcdfinvf(x); }

// Over-relaxed proposal (Neal 1998 as used by reference klhr.py:160-173 / klhr_sinh.py:215-228):
// u = CDF_q(0); r ~ Binomial(K, u); if r > K - r: v ~ Beta(K-r+1, 2r-K), u' = u v;
// if r < K - r: v ~ Beta(r+1, K-2r), u' = 1 - (1-u) v; else u' = u; z' = CDF_q^{-1}(u').
// The reference draws r and v from SciPy's global RNG; here they come from the chain's Philox
// stream (slots 0x80000000+), or are injected in replay mode.
template <typename R>
struct OrCtx {
    int K;                       // 0: standard proposal
    bool inject;                 // replay: r and v are inputs
    int r;
    R v;
    uint32_t c0, c1, d0, k0, k1d;
};

template <typename R>
__device__ inline void overrelax_sample(OrCtx<R>& oc, R u0) {
    const int K = oc.K;
    uint32_t w[4];
    int have = 0, q = 0;
    auto next_word = [&]() -> uint32_t {
        if (have == 0) {
            Philox::block(oc.c0, oc.c1, oc.d0, 0x80000000u + (uint32_t)q, oc.k0, oc.k1d, w);
            ++q;
            have = 4;
        }
        return w[4 - have--];
    };
    int r = 0;
    for (int k = 0; k < K; ++k) r += ((R)u01_32(next_word()) < u0) ? 1 : 0;
    int na = 0, nb = 0;
    if (r > K - r) { na = K - r + 1; nb = 2 * r - K; }
    else if (r < K - r) { na = r + 1; nb = K - 2 * r; }
    R v = 1;
    if (na > 0) {                // Beta(a, b), integer a, b: Ga / (Ga + Gb) with Gamma(n) = -sum log U
        float ga = 0, gb = 0;
        for (int i = 0; i < na; ++i) ga += exp1_32(next_word());
        for (int i = 0; i < nb; ++i) gb += exp1_32(next_word());
        v = (R)(ga / (ga + gb));
    }
    oc.r = r;
    oc.v = v;
}

// z_init, init2/init3 (sinh start for log d, e), z_prop, u are the step's variates
// (reference draw order: klhr.py:129,180,188 ; klhr_sinh.py:184,191,246,255).
template <int G, typename R, typename Model, int n>
__device__ void fit_and_propose(const typename Model::Coef& cf, const FitParams& fp, int lane, unsigned m,
                                R z_init, R init2, R init3, R z_prop, R u, StepOut<R>& o, OrCtx<R>& oc,
                                const ClipCtx<R>& cc = clip_off<R>()) {
    R xi, tau0;
    int nev1, nev2;
    stage1_mode<G, R, Model>(cf, z_init, fp, lane, m, xi, tau0, nev1);
    R eta[n];
    eta[0] = xi;
    eta[1] = tau0;
    if constexpr (n == 4) {
        eta[2] = init2 * (R)fp.initscale;          // klhr_sinh.py:191-193
        eta[3] = init3 * (R)fp.initscale;
        if (fp.fix_d) {                             // sub_klhr_sinh.py:184-186: start (xi, log s, e)
            eta[3] = eta[2];
            eta[2] = 0;
        }
    }
    bool conv;
    R s_fit;
    stage2_newton<G, R, Model, n>(cf, eta, fp, lane, m, nev2, conv, s_fit, cc);
    R zp, lq0, lq1;
    if constexpr (n == 2) {
        const R s = s_fit;                          // = exp(clamp(eta[1])), klhr.py:81-85
        if (oc.K > 0) {                             // klhr.py:160-173
            const R u0 = r_normcdf((R(0) - eta[0]) / s);
            if (!oc.inject) overrelax_sample<R>(oc, u0);
            R up = u0;
            if (oc.r > oc.K - oc.r) up = u0 * oc.v;
            else if (oc.r < oc.K - oc.r) up = R(1) - (R(1) - u0) * oc.v;
            z_prop = r_normcdfinv(up);
        }
        zp = eta[0] + s * z_prop;                   // klhr.py:180
        // _logq(0) - _logq(zp) (klhr.py:155-158,185-186): the two -log(s) terms cancel, so only
        // the quadratic parts are formed (saves two logs and two exps per draw)
        const R is = R(1) / s;                      // one division for both standardised points
        const R z0 = (R(0) - eta[0]) * is, z1 = (zp - eta[0]) * is;
        lq0 = -R(0.5) * z0 * z0;
        lq1 = -R(0.5) * z1 * z1;
    } else {
        if (oc.K > 0) {                             // klhr_sinh.py:215-228
            const SinhPar<R> q = sinh_unpack<R>(eta, fp);
            const R c = (R)fp.scale_clip;
            const R z0 = (R(0) - q.m) / q.s;
            const R u0 = r_normcdf(r_sinh(r_clamp(q.d * r_asinh(z0) - q.e, -c, c)));    // _CDF(0), :131-133
            if (!oc.inject) overrelax_sample<R>(oc, u0);
            R up = u0;
            if (oc.r > oc.K - oc.r) up = u0 * oc.v;
            else if (oc.r < oc.K - oc.r) up = R(1) - (R(1) - u0) * oc.v;
            z_prop = r_normcdfinv(up);              // _CDF_inv, :135-137
        }
        zp = transport_sinh<R>(z_prop, eta, fp);    // klhr_sinh.py:246
        lq0 = logq_sinh<R>(R(0), eta, fp);
        lq1 = logq_sinh<R>(zp, eta, fp);
    }
    const Jet<R> Jz = Model::eval(cf, zp);
    const R r = Jz.l + lq0 - lq1;                   // klhr.py:183-186 with lp(theta) = l(0)
    const R rm = r < R(0) ? r : R(0);               // np.minimum(0, r); NaN falls through to reject
    o.accept = (r == r) && (r_log(u) < rm);
#pragma unroll
    for (int i = 0; i < n; ++i) o.eta[i] = eta[i];
    o.zp = zp;
    o.r = r;
    o.converged = conv;
    o.evals = nev1 + nev2 * fp.N + 2;
}

}  // namespace klhr
