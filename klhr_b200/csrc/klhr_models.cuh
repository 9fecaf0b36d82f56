// klhr_b200 -- target densities as hand-written device functions (replaces BridgeStan).
//
// Each model provides
//   setup<GS>(th, rh, lane, mask, mp) -> Coef   reductions over the D-vector by the GS lanes of a chain: GS = 8
//                                           octet-cooperative (th = theta row, rh = rho row, both in shared
//                                           memory), result uniform across the 8 lanes; GS = 1 one thread
//                                           (lane = 0), no shuffles -- the chain kernel's D-phase for small D;
//   eval(coef, y) -> Jet                    O(1): l(y) - l(0), l'(y), l''(y) of the line
//                                           restriction l(y) = lp(theta + y rho) (logistic regression: O(N D),
//                                           a sum over the observations);
//   lp_grad(th, g, lane, mask, mp) -> lp    full-D log density and gradient (the
//                                           log_density[_gradient] API, bsmodel.py:15-30).
// The reference evaluates lp at every quadrature node through the full D-vector
// (klhr.py:110-113); every named Stan program has a closed-form restriction to a line, so
// the kernels pay O(D) once per draw and O(1) per evaluation.
// Conventions: BridgeStan propto=True, jacobian=True (bsmodel.py:18,27 forward no kwargs).
#pragma once
#include "klhr_common.cuh"
#include "../../include/klhr_sm100.h"

namespace klhr {

#define KLHR_DEFAULT_EVAL_CLIP                                                                                       \
    __device__ static __forceinline__ Jet<R> eval_clip(const Coef& c, R y, const ClipCtx<R>& cc, R& l1c) {             \
        return eval_clip_generic<R, Self>(c, y, cc, l1c);                                                             \
    }

// A model whose Coef keeps the theta / rho row pointers handed to setup (its eval walks the rows: LogisticRegression)
// declares kCoefKeepsRows = true.  Those rows must stay valid through the fit, so a kernel whose staged theta row is
// reused before the fit ends hands such a model the chain's own row instead (klhr_chain.cuh, octet D-phase).
template <typename M, typename = void> struct CoefKeepsRows { static constexpr bool value = false; };
template <typename M>
struct CoefKeepsRows<M, decltype((void)M::kCoefKeepsRows)> { static constexpr bool value = M::kCoefKeepsRows; };

struct ModelParams {
    int id;            // KLHR_MODEL_*
    int D;             // model.dim()
    int i0, i1;        // funnel: Da ; arK: K, n = T-K ; rosenbrock: Dh
    double s0, s1;     // ar1: alpha, 1/beta^2
    const void* p0;    // ill-normal: inv_s2[D] ; corr-normal: P[D*D] ; arK: pack[G|c|yy]
    const void* p1;
};

// ------------------------------------------------------------------ quadratic line
template <typename R>
struct QuadCoef { R A, Bq; };          // l(y) - l(0) = Bq y - A y^2 / 2

// For a quadratic a finite l implies finite y, A and Bq (0 * inf and inf - inf are NaN), hence finite l' and
// l'': one finiteness test gives the same (-inf, 0, 0) rule as the three of jet_guard.
template <typename R>
__device__ __forceinline__ Jet<R> quad_eval(const QuadCoef<R>& c, R y) {
    const R l = y * (c.Bq - R(0.5) * c.A * y);
    const bool ok = r_finite(l);
    Jet<R> j;
    j.l = ok ? l : -Num<R>::inf();
    j.l1 = ok ? c.Bq - c.A * y : R(0);
    j.l2 = ok ? -c.A : R(0);
    return j;
}

// ---- stan/normal.stan:1-9 and stan/ill-normal.stan:1-12  (diagonal Gaussian)
template <typename R, bool kScaled>
struct DiagNormal {
    using Self = DiagNormal<R, kScaled>;
    static constexpr bool kDenseCta = false;
    using Coef = QuadCoef<R>;
    __device__ static __forceinline__ R wgt(int i, const ModelParams& mp) {
        return kScaled ? __ldg(reinterpret_cast<const R*>(mp.p0) + i) : R(1);
    }
    template <int GS = kOct>
    __device__ static Coef setup(const R* th, const R* rh, int lane, unsigned m, const ModelParams& mp) {
        R a = 0, b = 0;
        for (int i = lane; i < mp.D; i += GS) {
            const R r = rh[i], t = th[i], w = wgt(i, mp);
            a += r * r * w;
            b -= r * t * w;
        }
        Coef c;
        c.A = grp_sum<GS>(a, m);
        c.Bq = grp_sum<GS>(b, m);
        return c;
    }
    __device__ static __forceinline__ Jet<R> eval(const Coef& c, R y) { return quad_eval(c, y); }
    KLHR_DEFAULT_EVAL_CLIP
    template <int G = kOct>
    __device__ static R lp_grad(const R* th, R* g, int lane, unsigned m, const ModelParams& mp) {
        R acc = 0;
        for (int i = lane; i < mp.D; i += G) {
            const R gi = -th[i] * wgt(i, mp);
            if (g) g[i] = gi;
            acc += th[i] * gi;
        }
        return R(0.5) * grp_sum<G>(acc, m);
    }
};

// ---- stan/corr-normal.stan:1-20  (dense precision P = Sigma^-1, symmetric)
template <typename R>
struct CorrNormal {
    using Self = CorrNormal<R>;
    static constexpr bool kDenseCta = true;     // fp64: CTA-cooperative DMMA path, klhr_dense.cuh
    using Coef = QuadCoef<R>;
    template <int GS = kOct>
    __device__ static Coef setup(const R* th, const R* rh, int lane, unsigned m, const ModelParams& mp) {
        const R* P = reinterpret_cast<const R*>(mp.p0);
        const int D = mp.D;
        R a = 0, b = 0;
        for (int i = lane; i < D; i += GS) {
            R v = 0;                                      // v_i = (P rho)_i ; P symmetric -> column walk is coalesced
            for (int k = 0; k < D; ++k) v += __ldg(P + (size_t)k * D + i) * rh[k];
            a += rh[i] * v;
            b -= th[i] * v;
        }
        Coef c;
        c.A = grp_sum<GS>(a, m);
        c.Bq = grp_sum<GS>(b, m);
        return c;
    }
    __device__ static __forceinline__ Jet<R> eval(const Coef& c, R y) { return quad_eval(c, y); }
    KLHR_DEFAULT_EVAL_CLIP
    template <int G = kOct>
    __device__ static R lp_grad(const R* th, R* g, int lane, unsigned m, const ModelParams& mp) {
        const R* P = reinterpret_cast<const R*>(mp.p0);
        const int D = mp.D;
        R acc = 0;
        for (int i = lane; i < D; i += G) {
            R v = 0;
            for (int k = 0; k < D; ++k) v += __ldg(P + (size_t)k * D + i) * th[k];
            if (g) g[i] = -v;
            acc -= th[i] * v;
        }
        return R(0.5) * grp_sum<G>(acc, m);
    }
};

// ---- stan/ar1.stan:1-14   e_t(v) = v_t - alpha v_{t-1}
template <typename R>
struct AR1 {
    using Self = AR1<R>;
    static constexpr bool kDenseCta = false;
    using Coef = QuadCoef<R>;
    template <int GS = kOct>
    __device__ static Coef setup(const R* th, const R* rh, int lane, unsigned m, const ModelParams& mp) {
        const R al = (R)mp.s0, ib2 = (R)mp.s1;
        R a = 0, b = 0;
        for (int i = lane; i < mp.D; i += GS) {
            if (i == 0) {
                a += rh[0] * rh[0];
                b -= rh[0] * th[0];
            } else {
                const R er = rh[i] - al * rh[i - 1];
                const R et = th[i] - al * th[i - 1];
                a += ib2 * er * er;
                b -= ib2 * er * et;
            }
        }
        Coef c;
        c.A = grp_sum<GS>(a, m);
        c.Bq = grp_sum<GS>(b, m);
        return c;
    }
    __device__ static __forceinline__ Jet<R> eval(const Coef& c, R y) { return quad_eval(c, y); }
    KLHR_DEFAULT_EVAL_CLIP
    template <int G = kOct>
    __device__ static R lp_grad(const R* th, R* g, int lane, unsigned m, const ModelParams& mp) {
        const R al = (R)mp.s0, ib2 = (R)mp.s1;
        const int D = mp.D;
        R acc = 0;
        for (int i = lane; i < D; i += G) {
            R gi;
            if (i == 0) {
                acc -= R(0.5) * th[0] * th[0];
                gi = -th[0];
            } else {
                const R e = th[i] - al * th[i - 1];
                acc -= R(0.5) * ib2 * e * e;
                gi = -ib2 * e;
            }
            if (i + 1 < D) gi += ib2 * al * (th[i + 1] - al * th[i]);
            if (g) g[i] = gi;
        }
        return grp_sum<G>(acc, m);
    }
};

// ---- stan/funnel.stan:1-11   params [x, alpha_1..alpha_Da]
template <typename R>
struct Funnel {
    using Self = Funnel<R>;
    static constexpr bool kDenseCta = false;
    struct Coef { R x0, r0, a0, a1, a2, hd, l0, t1, r1; };     // t1, r1: first alpha and its direction (dims = 2 clip path)
    template <int GS = kOct>
    __device__ static Coef setup(const R* th, const R* rh, int lane, unsigned m, const ModelParams& mp) {
        R a0 = 0, a1 = 0, a2 = 0;
        for (int i = 1 + lane; i < mp.D; i += GS) {
            const R t = th[i], r = rh[i];
            a0 += t * t;
            a1 += t * r;
            a2 += r * r;
        }
        Coef c;
        c.a0 = grp_sum<GS>(a0, m);
        c.a1 = grp_sum<GS>(a1, m);
        c.a2 = grp_sum<GS>(a2, m);
        c.x0 = th[0];
        c.r0 = rh[0];
        c.hd = R(0.5) * (R)mp.i0;
        c.t1 = mp.D > 1 ? th[1] : R(0);
        c.r1 = mp.D > 1 ? rh[1] : R(0);
        c.l0 = -c.x0 * c.x0 * R(1.0 / 18.0) - c.hd * c.x0 - R(0.5) * r_exp(-c.x0) * c.a0;
        return c;
    }
    __device__ static __forceinline__ Jet<R> eval(const Coef& c, R y) {
        const R x = c.x0 + y * c.r0;
        const R ex = r_exp(-x);
        const R S = c.a0 + y * (R(2) * c.a1 + y * c.a2);
        const R S1 = R(2) * (c.a1 + y * c.a2);
        const R S2 = R(2) * c.a2;
        // x^2 / 18 and friends as multiplications by the rounded reciprocal: an fp64 division costs ~20
        // instructions and this runs once per quadrature node (1 ulp away from the oracle's division)
        const R l = -x * x * R(1.0 / 18.0) - c.hd * x - R(0.5) * ex * S - c.l0;
        const R l1 = -c.r0 * x * R(1.0 / 9.0) - c.hd * c.r0 - R(0.5) * ex * (S1 - c.r0 * S);
        const R l2 = -c.r0 * c.r0 * R(1.0 / 9.0) - R(0.5) * ex * (c.r0 * c.r0 * S - R(2) * c.r0 * S1 + S2);
        return jet_guard<R>(l, l1, l2);
    }
    // eval + l' of the elementwise clipped gradient (klhr_sinh.py:158-161).  d/dx is formed exactly; the alpha
    // components are -alpha_i e^-x, bounded together by e^-x sqrt(sum alpha^2): only when one of the two can
    // exceed the clip are the components walked (theta / rho rows of the chain), sharing the exponential.
    __device__ static __forceinline__ Jet<R> eval_clip(const Coef& c, R y, const ClipCtx<R>& cc, R& l1c) {
        const R x = c.x0 + y * c.r0;
        const R ex = r_exp(-x);
        const R S = c.a0 + y * (R(2) * c.a1 + y * c.a2);
        const R S1 = R(2) * (c.a1 + y * c.a2);
        const R S2 = R(2) * c.a2;
        const R l = -x * x * R(1.0 / 18.0) - c.hd * x - R(0.5) * ex * S - c.l0;
        const R l1 = -c.r0 * x * R(1.0 / 9.0) - c.hd * c.r0 - R(0.5) * ex * (S1 - c.r0 * S);
        const R l2 = -c.r0 * c.r0 * R(1.0 / 9.0) - R(0.5) * ex * (c.r0 * c.r0 * S - R(2) * c.r0 * S1 + S2);
        const Jet<R> J = jet_guard<R>(l, l1, l2);
        l1c = J.l1;
        const R clip = cc.c;
        const R gxa = -x * R(1.0 / 9.0) - c.hd + R(0.5) * ex * S;           // d/dx (reciprocal multiply)
        if (cc.D == 2) {
            // stan/funnel.json (one alpha): both components in closed form, no branch in the node loop
            const R ga = -(c.t1 + y * c.r1) * ex;
            const R cx = r_clamp(gxa, -clip, clip), ca = r_clamp(ga, -clip, clip);
            const bool any = (cx != gxa) || (ca != ga);
            const R acc = cx * c.r0 + ca * c.r1;
            l1c = (any && r_finite(J.l)) ? acc : J.l1;
            return J;
        }
        // more alphas: cheap guard with a 1 % margin; the components are walked only when it trips
        const bool may = !(r_abs(gxa) < R(0.99) * clip) || !(ex * ex * S < R(0.98) * clip * clip);
        if (may && r_finite(J.l)) {
            const R gx = -x / R(9) - c.hd + R(0.5) * ex * S;                  // as lp_grad forms it
            const R cx = r_clamp(gx, -clip, clip);
            bool any = cx != gx;
            R acc = cx * c.r0;
            for (int i = 1; i < cc.D; ++i) {
                const R gi = -(cc.th[i] + y * cc.rh[i]) * ex;
                const R ci = r_clamp(gi, -clip, clip);
                any = any || (ci != gi);
                acc += ci * cc.rh[i];
            }
            if (any) l1c = acc;
        }
        return J;
    }
    template <int G = kOct>
    __device__ static R lp_grad(const R* th, R* g, int lane, unsigned m, const ModelParams& mp) {
        const R x = th[0];
        const R ex = r_exp(-x);
        R ss = 0;
        for (int i = 1 + lane; i < mp.D; i += G) {
            ss += th[i] * th[i];
            if (g) g[i] = -th[i] * ex;
        }
        ss = grp_sum<G>(ss, m);
        const R hd = R(0.5) * (R)mp.i0;
        if (g && lane == 0) g[0] = -x / R(9) - hd + R(0.5) * ex * ss;
        return -x * x / R(18) - hd * x - R(0.5) * ex * ss;
    }
};

// ---- stan/rosenbrock.stan:1-12   params [v_1..v_Dh, t_1..t_Dh]
template <typename R>
struct Rosenbrock {
    using Self = Rosenbrock<R>;
    static constexpr bool kDenseCta = false;
    struct Coef { R b1, b2, b3, b4; };      // l(y) - l(0) = b1 y + b2 y^2 + b3 y^3 + b4 y^4
    template <int GS = kOct>
    __device__ static Coef setup(const R* th, const R* rh, int lane, unsigned m, const ModelParams& mp) {
        const int Dh = mp.i0;
        R p1 = 0, p2 = 0, q1 = 0, q2 = 0, q3 = 0, q4 = 0;
        for (int i = lane; i < Dh; i += GS) {
            const R v = th[i], t = th[Dh + i], rv = rh[i], rt = rh[Dh + i];
            const R c0 = t - v * v, c1 = rt - R(2) * v * rv, c2 = -rv * rv;
            p1 += (v - R(1)) * rv;
            p2 += rv * rv;
            q1 += c0 * c1;
            q2 += c1 * c1 + R(2) * c0 * c2;
            q3 += c1 * c2;
            q4 += c2 * c2;
        }
        p1 = grp_sum<GS>(p1, m); p2 = grp_sum<GS>(p2, m);
        q1 = grp_sum<GS>(q1, m); q2 = grp_sum<GS>(q2, m); q3 = grp_sum<GS>(q3, m); q4 = grp_sum<GS>(q4, m);
        Coef c;
        c.b1 = -p1 - R(100) * q1;
        c.b2 = -R(0.5) * p2 - R(50) * q2;
        c.b3 = -R(100) * q3;
        c.b4 = -R(50) * q4;
        return c;
    }
    __device__ static __forceinline__ Jet<R> eval(const Coef& c, R y) {
        const R l = y * (c.b1 + y * (c.b2 + y * (c.b3 + y * c.b4)));
        const R l1 = c.b1 + y * (R(2) * c.b2 + y * (R(3) * c.b3 + y * R(4) * c.b4));
        const R l2 = R(2) * c.b2 + y * (R(6) * c.b3 + y * R(12) * c.b4);
        return jet_guard<R>(l, l1, l2);
    }
    KLHR_DEFAULT_EVAL_CLIP
    template <int G = kOct>
    __device__ static R lp_grad(const R* th, R* g, int lane, unsigned m, const ModelParams& mp) {
        const int Dh = mp.i0;
        R acc = 0;
        for (int i = lane; i < Dh; i += G) {
            const R v = th[i], t = th[Dh + i];
            const R c = t - v * v;
            acc -= R(0.5) * (v - R(1)) * (v - R(1)) + R(50) * c * c;
            if (g) {
                g[i] = -(v - R(1)) + R(200) * v * c;
                g[Dh + i] = -R(100) * c;
            }
        }
        return grp_sum<G>(acc, m);
    }
};

// ---- stan/arK.stan:1-20   unconstrained [alpha, beta_1..beta_K, u = log sigma]
// Sufficient statistics (host, fp64): X_t = (1, y_{t-K..t-1}), G = X^T X, c = X^T y, yy = y^T y
// over t = K+1..T, packed [G (K+1)^2 | c (K+1) | yy].  sum r^2 = yy - 2 phi.c + phi^T G phi.
template <typename R>
struct ARK {
    using Self = ARK<R>;
    static constexpr bool kDenseCta = false;
    struct Coef { R p0, p1, p2, q0, q1, q2, u0, ru, nm1, l0; };
    template <int GS = kOct>
    __device__ static __forceinline__ void gram_forms(const R* th, const R* rh, int lane, unsigned m,
                                                      const ModelParams& mp, R& q0, R& q1, R& q2,
                                                      R& p0, R& p1, R& p2, R* gphi /*(G phi - c)_lane or null*/) {
        // The sufficient statistics are ALWAYS fp64 (whatever R is) and the forms are accumulated in
        // fp64: sum r^2 = yy - 2 phi.c + phi^T G phi cancels to a few per cent of its terms, which fp32
        // storage cannot carry (D = K + 2 is tiny, so this costs nothing).
        const int K1 = mp.i0 + 1;
        const double* G = reinterpret_cast<const double*>(mp.p0);
        const double* cv = G + K1 * K1;
        const double yy = __ldg(cv + K1);
        double s_pc = 0, s_pGp = 0, s_rGp = 0, s_rGr = 0, s_rc = 0;
        R pp = 0, pr = 0, rr = 0;
        for (int i = lane; i < K1; i += GS) {
            double Gp = 0, Gr = 0;
            for (int k = 0; k < K1; ++k) {
                const double gik = __ldg(G + i * K1 + k);
                Gp += gik * (double)th[k];
                Gr += gik * (double)rh[k];
            }
            const double ci = __ldg(cv + i);
            s_pc += (double)th[i] * ci;
            s_pGp += (double)th[i] * Gp;
            s_rGp += (double)rh[i] * Gp;
            s_rGr += (double)rh[i] * Gr;
            s_rc += (double)rh[i] * ci;
            pp += th[i] * th[i];
            pr += th[i] * rh[i];
            rr += rh[i] * rh[i];
            if (gphi) gphi[i] = (R)(Gp - ci);
        }
        s_pc = grp_sum<GS>(s_pc, m); s_pGp = grp_sum<GS>(s_pGp, m); s_rGp = grp_sum<GS>(s_rGp, m);
        s_rGr = grp_sum<GS>(s_rGr, m); s_rc = grp_sum<GS>(s_rc, m);
        p0 = grp_sum<GS>(pp, m); p1 = grp_sum<GS>(pr, m); p2 = grp_sum<GS>(rr, m);
        q0 = (R)(yy - 2.0 * s_pc + s_pGp);      // sum r^2 at phi
        q1 = (R)(s_rGp - s_rc);                 // 1/2 d/dy sum r^2
        q2 = (R)s_rGr;
    }
    __device__ static __forceinline__ R value(const Coef& c, R y) {
        const R u = c.u0 + y * c.ru;
        return -R(0.5) * (c.p0 + y * (R(2) * c.p1 + y * c.p2)) - R(0.5) * r_exp(R(2) * u) - c.nm1 * u
               - R(0.5) * r_exp(-R(2) * u) * (c.q0 + y * (R(2) * c.q1 + y * c.q2));
    }
    template <int GS = kOct>
    __device__ static Coef setup(const R* th, const R* rh, int lane, unsigned m, const ModelParams& mp) {
        Coef c;
        gram_forms<GS>(th, rh, lane, m, mp, c.q0, c.q1, c.q2, c.p0, c.p1, c.p2, nullptr);
        c.u0 = th[mp.D - 1];
        c.ru = rh[mp.D - 1];
        c.nm1 = (R)(mp.i1 - 1);                 // (T-K) u - u  (likelihood minus Jacobian)
        c.l0 = 0;
        c.l0 = value(c, R(0));
        return c;
    }
    __device__ static __forceinline__ Jet<R> eval(const Coef& c, R y) {
        const R u = c.u0 + y * c.ru;
        const R e2 = r_exp(R(2) * u), em2 = r_exp(-R(2) * u);
        const R S = c.q0 + y * (R(2) * c.q1 + y * c.q2);
        const R S1 = R(2) * (c.q1 + y * c.q2);
        const R S2 = R(2) * c.q2;
        const R l = -R(0.5) * (c.p0 + y * (R(2) * c.p1 + y * c.p2)) - R(0.5) * e2 - c.nm1 * u
                    - R(0.5) * em2 * S - c.l0;
        const R l1 = -(c.p1 + y * c.p2) - c.ru * e2 - c.nm1 * c.ru - R(0.5) * em2 * (S1 - R(2) * c.ru * S);
        const R l2 = -c.p2 - R(2) * c.ru * c.ru * e2
                     - R(0.5) * em2 * (R(4) * c.ru * c.ru * S - R(4) * c.ru * S1 + S2);
        return jet_guard<R>(l, l1, l2);
    }
    KLHR_DEFAULT_EVAL_CLIP
    template <int G = kOct>
    __device__ static R lp_grad(const R* th, R* g, int lane, unsigned m, const ModelParams& mp) {
        // rho := theta is a harmless stand-in for the unused direction sums
        R q0, q1, q2, p0, p1, p2;
        const int K1 = mp.i0 + 1;
        const R u = th[mp.D - 1];
        const R e2 = r_exp(R(2) * u), em2 = r_exp(-R(2) * u);
        gram_forms<G>(th, th, lane, m, mp, q0, q1, q2, p0, p1, p2, g);
        // p0 counted the first K+1 entries only (phi); gphi holds (G phi - c)_i = -(X^T r)_i
        if (g) {
            for (int i = lane; i < K1; i += G) g[i] = -th[i] - em2 * g[i];
            if (lane == 0) g[mp.D - 1] = -e2 + R(1) - (R)mp.i1 + em2 * q0;
        }
        return -R(0.5) * p0 - R(0.5) * e2 + u - (R)mp.i1 * u - R(0.5) * em2 * q0;
    }
};

// ---- stan/earnings.stan:1-17   unconstrained [b1, b2, us = log sigma, ut = log s]
// (the model of the reference's self-tests, klhr.py:238, and relaxation experiment).
// Sufficient statistics (host, fp64) packed as [N, Se, Sh, See, Seh, Shh] with e = earn, h = height:
// SSR(b) = See - 2 b1 Se - 2 b2 Seh + b1^2 N + 2 b1 b2 Sh + b2^2 Shh.
template <typename R>
struct Earnings {
    using Self = Earnings<R>;
    static constexpr bool kDenseCta = false;
    struct Coef { R b1, b2, r1, r2, us0, rs, ut0, rt, S0, S1, S2, nm1, l0; };
    struct Stats { double N, Se, Sh, See, Seh, Shh; };        // always fp64 (dollar-scale sums)
    __device__ static __forceinline__ Stats stats(const ModelParams& mp) {
        const double* p = reinterpret_cast<const double*>(mp.p0);
        Stats s;
        s.N = __ldg(p); s.Se = __ldg(p + 1); s.Sh = __ldg(p + 2);
        s.See = __ldg(p + 3); s.Seh = __ldg(p + 4); s.Shh = __ldg(p + 5);
        return s;
    }
    __device__ static __forceinline__ R student(R w) { return -R(3) * r_log1p(w * w / R(5)); }
    __device__ static __forceinline__ R value(const Coef& c, R y) {
        const R us = c.us0 + y * c.rs, ut = c.ut0 + y * c.rt;
        const R emt = r_exp(-ut);
        const R w1 = (c.b1 + y * c.r1) * emt, w2 = (c.b2 + y * c.r2) * emt;
        const R S = c.S0 + y * (R(2) * c.S1 + y * c.S2);
        return -R(0.01) * r_exp(ut) - ut + student(w1) + student(w2) - R(0.1) * r_exp(us) - c.nm1 * us
               - R(0.5) * r_exp(-R(2) * us) * S;
    }
    // D = 4: every lane computes the same coefficients, no reductions needed
    template <int GS = kOct>
    __device__ static Coef setup(const R* th, const R* rh, int lane, unsigned m, const ModelParams& mp) {
        const Stats s = stats(mp);
        Coef c;
        c.b1 = th[0]; c.b2 = th[1]; c.us0 = th[2]; c.ut0 = th[3];
        c.r1 = rh[0]; c.r2 = rh[1]; c.rs = rh[2]; c.rt = rh[3];
        const double b1 = c.b1, b2 = c.b2, r1 = c.r1, r2 = c.r2;
        c.S0 = (R)(s.See - 2.0 * b1 * s.Se - 2.0 * b2 * s.Seh + b1 * b1 * s.N + 2.0 * b1 * b2 * s.Sh + b2 * b2 * s.Shh);
        // X^T r with r = e - b1 - b2 h
        const double xr1 = s.Se - b1 * s.N - b2 * s.Sh;
        const double xr2 = s.Seh - b1 * s.Sh - b2 * s.Shh;
        c.S1 = (R)(-(r1 * xr1 + r2 * xr2));
        c.S2 = (R)(r1 * r1 * s.N + 2.0 * r1 * r2 * s.Sh + r2 * r2 * s.Shh);
        c.nm1 = (R)(s.N - 1.0);
        c.l0 = 0;
        c.l0 = value(c, R(0));
        return c;
    }
    __device__ static __forceinline__ Jet<R> eval(const Coef& c, R y) {
        const R us = c.us0 + y * c.rs, ut = c.ut0 + y * c.rt;
        const R et = r_exp(ut), emt = R(1) / et, es = r_exp(us), em2 = R(1) / (es * es);
        const R S = c.S0 + y * (R(2) * c.S1 + y * c.S2);
        const R Sp = R(2) * (c.S1 + y * c.S2), Spp = R(2) * c.S2;
        R l = -R(0.01) * et - ut - R(0.1) * es - c.nm1 * us - R(0.5) * em2 * S - c.l0;
        R l1 = -R(0.01) * c.rt * et - c.rt - R(0.1) * c.rs * es - c.nm1 * c.rs - R(0.5) * em2 * (Sp - R(2) * c.rs * S);
        R l2 = -R(0.01) * c.rt * c.rt * et - R(0.1) * c.rs * c.rs * es
               - R(0.5) * em2 * (R(4) * c.rs * c.rs * S - R(4) * c.rs * Sp + Spp);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const R bk = k == 0 ? c.b1 + y * c.r1 : c.b2 + y * c.r2;
            const R rk = k == 0 ? c.r1 : c.r2;
            const R w = bk * emt;
            const R wp = rk * emt - c.rt * w;
            const R wpp = -c.rt * rk * emt - c.rt * wp;
            const R den = R(5) + w * w;
            const R f1 = -R(6) * w / den;
            const R f2 = -R(6) * (R(5) - w * w) / (den * den);
            l += student(w);
            l1 += f1 * wp;
            l2 += f2 * wp * wp + f1 * wpp;
        }
        return jet_guard<R>(l, l1, l2);
    }
    KLHR_DEFAULT_EVAL_CLIP
    template <int G = kOct>
    __device__ static R lp_grad(const R* th, R* g, int lane, unsigned m, const ModelParams& mp) {
        const Stats s = stats(mp);
        const R b1 = th[0], b2 = th[1], us = th[2], ut = th[3];
        const R et = r_exp(ut), em2t = r_exp(-R(2) * ut), es = r_exp(us), em2 = r_exp(-R(2) * us);
        const double d1 = b1, d2 = b2;
        const R ssr = (R)(s.See - 2.0 * d1 * s.Se - 2.0 * d2 * s.Seh + d1 * d1 * s.N + 2.0 * d1 * d2 * s.Sh + d2 * d2 * s.Shh);
        const R q1 = b1 * b1 * em2t, q2 = b2 * b2 * em2t;
        const R nN = (R)s.N;
        if (g && lane == 0) {
            g[0] = -R(6) * b1 * em2t / (R(5) + q1) + em2 * (R)(s.Se - d1 * s.N - d2 * s.Sh);
            g[1] = -R(6) * b2 * em2t / (R(5) + q2) + em2 * (R)(s.Seh - d1 * s.Sh - d2 * s.Shh);
            g[2] = -R(0.1) * es + R(1) - nN + em2 * ssr;
            g[3] = -R(0.01) * et - R(1) + R(6) * q1 / (R(5) + q1) + R(6) * q2 / (R(5) + q2);
        }
        return -R(0.01) * et - ut - R(3) * (r_log1p(q1 / R(5)) + r_log1p(q2 / R(5))) - R(0.1) * es + us - nN * us
               - R(0.5) * em2 * ssr;
    }
};

// ------------------------------------------------------------------ eight schools (hierarchical normal)
// Data (both parametrisations): i0 = J, data0 = [y_1..J | w_1..J] in R, w_j = 1 / sigma_j^2.  u = log tau.
//
// The half-Cauchy prior on tau, on the unconstrained scale, is -log1p(tau^2 / 25) = -softplus(z), z = 2u - log 25.
// log1p(exp(2u) / 25) overflows from u ~ 355 (fp64) or ~ 45 (fp32), long before the line searches of the fit stop
// visiting such u; the stable form max(z, 0) + log1p(e^-|z|) is finite wherever z is, and its derivatives come from
// the logistic function sigma(z) = d softplus / dz.  e^-|z| is formed from the model's own exponential (e^{2u} / 25
// or its reciprocal), so an evaluation costs one exponential and one log1p.
template <typename R>
struct Softplus { R sp, sg, sg1; };          // softplus(z), sigma(z), sigma(z) (1 - sigma(z))

template <typename R>
__device__ __forceinline__ Softplus<R> softplus_q(R z, R q /* e^-|z| */) {
    Softplus<R> s;
    const R inv = R(1) / (R(1) + q);
    s.sp = r_max(z, R(0)) + r_log1p(q);
    s.sg = z >= R(0) ? inv : q * inv;
    s.sg1 = q * inv * inv;
    return s;
}

// e^-|z| for z = 2u - log 25 from e2 = e^{2u}: 25 / e2 above u = log 5, e2 / 25 below
template <typename R>
__device__ __forceinline__ R cauchy_q_from_e2(R z, R e2) { return z >= R(0) ? R(25) / e2 : e2 * R(1.0 / 25.0); }

constexpr double kLog25 = 3.2188758248682006;

// ---- posteriordb eight_schools_noncentered   params [theta_trans_1..J, mu, u = log tau]
//   data { int<lower=0> J; real y[J]; real<lower=0> sigma[J]; }
//   parameters { vector[J] theta_trans; real mu; real<lower=0> tau; }
//   transformed parameters { vector[J] theta = theta_trans * tau + mu; }
//   model { theta_trans ~ normal(0, 1); y ~ normal(theta, sigma); mu ~ normal(0, 5); tau ~ cauchy(0, 5); }
// lp = -1/2 sum tt^2 - 1/2 sum w (y - mu - e^u tt)^2 - mu^2 / 50 - softplus(2u - log 25) + u.
// Line tt = a + t r, mu = m0 + t rm, u = u0 + t ru, c = y - m0, d = c - t rm: with W(f) = sum_j w_j f_j the
// likelihood sum is P(t) - 2 e^u Q(t) + e^{2u} S(t), P = sum w d^2, Q = sum w d tt, S = sum w tt^2, all quadratics
// in t.  Everything but e^u Q - e^{2u} S / 2 - softplus is a quadratic in t, kept as its change b1 t + b2 t^2 from
// t = 0 (the constants W(c^2), sum a^2 cancel, so 11 of the 13 sums are needed).
template <typename R>
struct EightSchoolsNC {
    using Self = EightSchoolsNC<R>;
    static constexpr bool kDenseCta = false;
    struct Coef { R b1, b2, q0, q1, q2, s0, s1, s2, u0, ru, f0; };
    __device__ static __forceinline__ R y_(int j, const ModelParams& mp) { return __ldg(reinterpret_cast<const R*>(mp.p0) + j); }
    __device__ static __forceinline__ R w_(int j, const ModelParams& mp) {
        return __ldg(reinterpret_cast<const R*>(mp.p0) + mp.i0 + j);
    }
    // e^u Q - e^{2u} S / 2 - softplus(z) and its first two t-derivatives
    __device__ static __forceinline__ Jet<R> nonpoly(const Coef& c, R y) {
        const R u = c.u0 + y * c.ru;
        const R E = r_exp(u), e2 = E * E;
        const R z = R(2) * u - R(kLog25);
        const Softplus<R> s = softplus_q(z, cauchy_q_from_e2(z, e2));
        const R Q = c.q0 + y * (c.q1 + y * c.q2), Q1 = c.q1 + R(2) * y * c.q2, Q2 = R(2) * c.q2;
        const R S = c.s0 + y * (c.s1 + y * c.s2), S1 = c.s1 + R(2) * y * c.s2, S2 = R(2) * c.s2;
        Jet<R> j;
        j.l = E * Q - R(0.5) * e2 * S - s.sp;
        j.l1 = E * (c.ru * Q + Q1) - R(0.5) * e2 * (R(2) * c.ru * S + S1) - R(2) * c.ru * s.sg;
        j.l2 = E * (c.ru * c.ru * Q + R(2) * c.ru * Q1 + Q2) - R(0.5) * e2 * (R(4) * c.ru * c.ru * S + R(4) * c.ru * S1 + S2)
               - R(4) * c.ru * c.ru * s.sg1;
        return j;
    }
    template <int GS = kOct>
    __device__ static Coef setup(const R* th, const R* rh, int lane, unsigned m, const ModelParams& mp) {
        const int J = mp.i0;
        const R m0 = th[J], rm = rh[J];
        R W1 = 0, Wc = 0, Wa = 0, Wr = 0, Wca = 0, Wcr = 0, Wa2 = 0, War = 0, Wr2 = 0, ar = 0, r2 = 0;
        for (int j = lane; j < J; j += GS) {
            const R w = w_(j, mp), c = y_(j, mp) - m0, a = th[j], r = rh[j];
            W1 += w; Wc += w * c; Wa += w * a; Wr += w * r;
            Wca += w * c * a; Wcr += w * c * r;
            Wa2 += w * a * a; War += w * a * r; Wr2 += w * r * r;
            ar += a * r; r2 += r * r;
        }
        W1 = grp_sum<GS>(W1, m); Wc = grp_sum<GS>(Wc, m); Wa = grp_sum<GS>(Wa, m); Wr = grp_sum<GS>(Wr, m);
        Wca = grp_sum<GS>(Wca, m); Wcr = grp_sum<GS>(Wcr, m);
        Wa2 = grp_sum<GS>(Wa2, m); War = grp_sum<GS>(War, m); Wr2 = grp_sum<GS>(Wr2, m);
        ar = grp_sum<GS>(ar, m); r2 = grp_sum<GS>(r2, m);
        Coef c;
        c.u0 = th[J + 1];
        c.ru = rh[J + 1];
        // -1/2 sum tt^2 - 1/2 P - mu^2 / 50 + u, less its value at t = 0
        c.b1 = -ar + rm * Wc - m0 * rm * R(1.0 / 25.0) + c.ru;
        c.b2 = -R(0.5) * r2 - R(0.5) * rm * rm * W1 - rm * rm * R(1.0 / 50.0);
        c.q0 = Wca; c.q1 = Wcr - rm * Wa; c.q2 = -rm * Wr;
        c.s0 = Wa2; c.s1 = R(2) * War; c.s2 = Wr2;
        c.f0 = 0;
        c.f0 = nonpoly(c, R(0)).l;
        return c;
    }
    __device__ static __forceinline__ Jet<R> eval(const Coef& c, R y) {
        const Jet<R> f = nonpoly(c, y);
        return jet_guard<R>(y * (c.b1 + y * c.b2) + f.l - c.f0, c.b1 + R(2) * y * c.b2 + f.l1, R(2) * c.b2 + f.l2);
    }
    KLHR_DEFAULT_EVAL_CLIP
    template <int G = kOct>
    __device__ static R lp_grad(const R* th, R* g, int lane, unsigned m, const ModelParams& mp) {
        const int J = mp.i0;
        const R mu = th[J], u = th[J + 1];
        const R E = r_exp(u);
        R acc = 0, swr = 0, swrt = 0;
        for (int j = lane; j < J; j += G) {
            const R tt = th[j], w = w_(j, mp);
            const R res = y_(j, mp) - mu - E * tt;
            acc -= R(0.5) * (tt * tt + w * res * res);
            swr += w * res;
            swrt += w * res * tt;
            if (g) g[j] = -tt + E * w * res;
        }
        acc = grp_sum<G>(acc, m); swr = grp_sum<G>(swr, m); swrt = grp_sum<G>(swrt, m);
        const R z = R(2) * u - R(kLog25);
        const Softplus<R> s = softplus_q(z, cauchy_q_from_e2(z, E * E));
        if (g && lane == 0) {
            g[J] = swr - mu * R(1.0 / 25.0);
            g[J + 1] = E * swrt - R(2) * s.sg + R(1);
        }
        return acc - mu * mu * R(1.0 / 50.0) - s.sp + u;
    }
};

// ---- posteriordb eight_schools_centered   params [mu, u = log tau, theta_1..J]
//   data { int<lower=0> J; real y[J]; real<lower=0> sigma[J]; }
//   parameters { real mu; real<lower=0> tau; real theta[J]; }
//   model { mu ~ normal(0, 5); tau ~ cauchy(0, 5); theta ~ normal(mu, tau); y ~ normal(theta, sigma); }
// lp = -mu^2 / 50 - softplus(2u - log 25) + (1 - J) u - 1/2 e^{-2u} sum (theta - mu)^2 - 1/2 sum w (y - theta)^2.
// Line theta = a + t r, mu = m0 + t rm, u = u0 + t ru: sum (theta - mu)^2 = A0 + 2 A1 t + A2 t^2 and
// sum w (y - theta)^2 = B0 - 2 B1 t + B2 t^2 (B0 cancels in l(t) - l(0)).
template <typename R>
struct EightSchoolsC {
    using Self = EightSchoolsC<R>;
    static constexpr bool kDenseCta = false;
    struct Coef { R b1, b2, A0, A1, A2, u0, ru, f0; };
    __device__ static __forceinline__ R y_(int j, const ModelParams& mp) { return __ldg(reinterpret_cast<const R*>(mp.p0) + j); }
    __device__ static __forceinline__ R w_(int j, const ModelParams& mp) {
        return __ldg(reinterpret_cast<const R*>(mp.p0) + mp.i0 + j);
    }
    // -1/2 e^{-2u} A(t) - softplus(z) and its first two t-derivatives
    __device__ static __forceinline__ Jet<R> nonpoly(const Coef& c, R y) {
        const R u = c.u0 + y * c.ru;
        const R em2 = r_exp(-R(2) * u);
        const R z = R(2) * u - R(kLog25);
        const Softplus<R> s = softplus_q(z, z >= R(0) ? R(25) * em2 : R(1) / (R(25) * em2));
        const R A = c.A0 + y * (R(2) * c.A1 + y * c.A2), A1 = R(2) * (c.A1 + y * c.A2), A2 = R(2) * c.A2;
        Jet<R> j;
        j.l = -R(0.5) * em2 * A - s.sp;
        j.l1 = -R(0.5) * em2 * (A1 - R(2) * c.ru * A) - R(2) * c.ru * s.sg;
        j.l2 = -R(0.5) * em2 * (R(4) * c.ru * c.ru * A - R(4) * c.ru * A1 + A2) - R(4) * c.ru * c.ru * s.sg1;
        return j;
    }
    template <int GS = kOct>
    __device__ static Coef setup(const R* th, const R* rh, int lane, unsigned m, const ModelParams& mp) {
        const int J = mp.i0;
        const R m0 = th[0], rm = rh[0];
        R A0 = 0, A1 = 0, A2 = 0, B1 = 0, B2 = 0;
        for (int j = lane; j < J; j += GS) {
            const R w = w_(j, mp), a = th[2 + j], r = rh[2 + j];
            const R dm = a - m0, dr = r - rm, e = y_(j, mp) - a;
            A0 += dm * dm; A1 += dm * dr; A2 += dr * dr;
            B1 += w * e * r; B2 += w * r * r;
        }
        Coef c;
        c.A0 = grp_sum<GS>(A0, m); c.A1 = grp_sum<GS>(A1, m); c.A2 = grp_sum<GS>(A2, m);
        B1 = grp_sum<GS>(B1, m); B2 = grp_sum<GS>(B2, m);
        c.u0 = th[1];
        c.ru = rh[1];
        // -mu^2 / 50 + (1 - J) u - 1/2 sum w (y - theta)^2, less its value at t = 0
        c.b1 = -m0 * rm * R(1.0 / 25.0) + R(1 - J) * c.ru + B1;
        c.b2 = -rm * rm * R(1.0 / 50.0) - R(0.5) * B2;
        c.f0 = 0;
        c.f0 = nonpoly(c, R(0)).l;
        return c;
    }
    __device__ static __forceinline__ Jet<R> eval(const Coef& c, R y) {
        const Jet<R> f = nonpoly(c, y);
        return jet_guard<R>(y * (c.b1 + y * c.b2) + f.l - c.f0, c.b1 + R(2) * y * c.b2 + f.l1, R(2) * c.b2 + f.l2);
    }
    KLHR_DEFAULT_EVAL_CLIP
    template <int G = kOct>
    __device__ static R lp_grad(const R* th, R* g, int lane, unsigned m, const ModelParams& mp) {
        const int J = mp.i0;
        const R mu = th[0], u = th[1];
        const R em2 = r_exp(-R(2) * u);
        R sd = 0, sd2 = 0, lik = 0;
        for (int j = lane; j < J; j += G) {
            const R tj = th[2 + j], w = w_(j, mp);
            const R d = tj - mu, e = y_(j, mp) - tj;
            sd += d;
            sd2 += d * d;
            lik += w * e * e;
            if (g) g[2 + j] = -em2 * d + w * e;
        }
        sd = grp_sum<G>(sd, m); sd2 = grp_sum<G>(sd2, m); lik = grp_sum<G>(lik, m);
        const R z = R(2) * u - R(kLog25);
        const Softplus<R> s = softplus_q(z, z >= R(0) ? R(25) * em2 : R(1) / (R(25) * em2));
        if (g && lane == 0) {
            g[0] = -mu * R(1.0 / 25.0) + em2 * sd;
            g[1] = -R(2) * s.sg + R(1 - J) + em2 * sd2;
        }
        return -mu * mu * R(1.0 / 50.0) - s.sp + R(1 - J) * u - R(0.5) * em2 * sd2 - R(0.5) * lik;
    }
};

// ------------------------------------------------------------------ logistic regression (a sum over observations)
// ---- Bayesian logistic regression   params [alpha, beta_1..K], D = K + 1
//   data { int<lower=0> N; int<lower=1> K; matrix[N, K] x; array[N] int<lower=0, upper=1> y; }
//   parameters { real alpha; vector[K] beta; }
//   model { alpha ~ normal(0, 2.5); beta ~ normal(0, 2.5); y ~ bernoulli_logit(alpha + x * beta); }
// Data: i0 = N (>= 0), i1 = K, data0 = [X (N x D row-major, X[i][0] = 1) | y (N)] in R.
// lp = -|theta|^2 / 12.5 + sum_i (y_i eta_i - softplus(eta_i)),  eta = X theta.
//
// The restriction to the line theta + t rho has no O(1) form: with a = X theta and b = X rho,
// l(t) = -(|theta|^2 + 2 t theta.rho + t^2 rho.rho) / 12.5 + sum_i (y_i (a_i + t b_i) - softplus(a_i + t b_i)).
// Storing a and b would cost O(N) memory per chain.  eval recomputes both dot products of every row instead (2 D FMAs,
// one exp, one log1p per observation), so the chain state stays O(D) and every kernel runs the model unchanged.  X is
// shared by all chains and the lanes of a warp read the same row at the same time: broadcast loads from L1 / L2.
// So Coef keeps pointers to the chain's theta and rho rows, which must stay valid through the fit (kCoefKeepsRows).
// softplus is formed as max(z, 0) + log1p(e^-|z|) (softplus_q): no |eta| overflows in fp32 or fp64.
template <typename R>
struct LogisticRegression {
    using Self = LogisticRegression<R>;
    static constexpr bool kDenseCta = false;
    static constexpr bool kCoefKeepsRows = true;
    struct Coef { const R* th; const R* rh; const R* X; const R* y; int N, D; R tr, rr, l0; };
    __device__ static __forceinline__ const R* X_(const ModelParams& mp) { return reinterpret_cast<const R*>(mp.p0); }
    template <int GS = kOct>
    __device__ static Coef setup(const R* th, const R* rh, int lane, unsigned m, const ModelParams& mp) {
        Coef c;
        c.th = th; c.rh = rh; c.N = mp.i0; c.D = mp.D;
        c.X = X_(mp);
        c.y = c.X + (size_t)c.N * c.D;
        R tr = 0, rr = 0, l0 = 0;
        for (int k = lane; k < c.D; k += GS) {
            tr += th[k] * rh[k];
            rr += rh[k] * rh[k];
        }
        for (int i = lane; i < c.N; i += GS) {         // the likelihood at t = 0
            const R* x = c.X + (size_t)i * c.D;
            R a = 0;
            for (int k = 0; k < c.D; ++k) a += __ldg(x + k) * th[k];
            const Softplus<R> s = softplus_q(a, r_exp(-r_abs(a)));
            l0 += __ldg(c.y + i) * a - s.sp;
        }
        c.tr = grp_sum<GS>(tr, m);
        c.rr = grp_sum<GS>(rr, m);
        c.l0 = grp_sum<GS>(l0, m);
        return c;
    }
    __device__ static __forceinline__ Jet<R> eval(const Coef& c, R t) {
        R l = 0, l1 = 0, l2 = 0;
        const R* x = c.X;
        for (int i = 0; i < c.N; ++i, x += c.D) {
            R a = 0, b = 0;
            for (int k = 0; k < c.D; ++k) {
                const R xk = __ldg(x + k);
                a += xk * c.th[k];
                b += xk * c.rh[k];
            }
            const R eta = a + t * b;
            const Softplus<R> s = softplus_q(eta, r_exp(-r_abs(eta)));
            const R yi = __ldg(c.y + i);
            l += yi * eta - s.sp;
            l1 += b * (yi - s.sg);
            l2 -= b * b * s.sg1;
        }
        return jet_guard<R>(l - c.l0 - t * (R(2) * c.tr + t * c.rr) * R(1.0 / 12.5),
                            l1 - (c.tr + t * c.rr) * R(1.0 / 6.25), l2 - c.rr * R(1.0 / 6.25));
    }
    KLHR_DEFAULT_EVAL_CLIP
    template <int G = kOct>
    __device__ static R lp_grad(const R* th, R* g, int lane, unsigned m, const ModelParams& mp) {
        const int N = mp.i0, D = mp.D;
        const R* X = X_(mp);
        const R* yv = X + (size_t)N * D;
        R acc = 0;
        for (int k = lane; k < D; k += G) {
            acc -= th[k] * th[k] * R(1.0 / 12.5);
            if (g) g[k] = -th[k] * R(1.0 / 6.25);
        }
        // observations in groups of G, one per lane; then every lane adds x_ik r_i of the whole group to the gradient
        // components it owns (k = lane mod G), with r_i = y_i - sigma(eta_i) broadcast from the lane that formed it
        for (int i0 = 0; i0 < N; i0 += G) {
            const int i = i0 + lane;
            R r = 0;
            if (i < N) {
                const R* x = X + (size_t)i * D;
                R a = 0;
                for (int k = 0; k < D; ++k) a += __ldg(x + k) * th[k];
                const Softplus<R> s = softplus_q(a, r_exp(-r_abs(a)));
                const R yi = __ldg(yv + i);
                acc += yi * a - s.sp;
                r = yi - s.sg;
            }
            if (g) {
                R rl[G];
#pragma unroll
                for (int l = 0; l < G; ++l) rl[l] = G == 1 ? r : __shfl_sync(m, r, l, kOct);
                const int nl = N - i0 < G ? N - i0 : G;
                for (int k = lane; k < D; k += G) {
                    R s = 0;
#pragma unroll
                    for (int l = 0; l < G; ++l)
                        if (l < nl) s += __ldg(X + (size_t)(i0 + l) * D + k) * rl[l];
                    g[k] += s;
                }
            }
        }
        return grp_sum<G>(acc, m);
    }
};

}  // namespace klhr
