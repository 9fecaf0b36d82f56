// klhr_b200 -- forward-mode Taylor arithmetic for user-written targets (klhr_user.cuh).
//
// A user target is one templated device function T log_density(x, data).  The library runs it on three types:
//   R        the value (lp, MH ratios, the line's l(0));
//   Dual<R>  the value and one directional derivative: one pass per gradient component (log_density_gradient);
//   Tay2<R>  the value and the first two derivatives along the line theta + y rho: l(y), l'(y), l''(y) in one pass
//            (every evaluation of the fit and the slice sampler).
// Every operation inlines to straight-line code on a few registers: no arrays, no virtual calls.
//
// The elementary functions reuse the library's own routines and the stable forms the built-in models use, so a user
// restatement of a built-in target matches it to rounding and stays finite where the built-in model does:
//   exp / log / log1p          r_exp, r_log, r_log1p (klhr_common.cuh)
//   log1p_exp, log_inv_logit  softplus_q: max(z, 0) + log1p(e^-|z|), derivatives from the logistic function
//   tanh                       from e^-2|u| (as Arma11::bounded forms tanh(u / 2) from e^-|u|): 1 - tanh^2 is never
//                              formed by cancellation
// For plain R the CUDA math library's functions of the same name are chosen where they exist (exp, log, log1p, expm1,
// sqrt, tanh, fabs): the overloads below are templates, which lose to them on an exact match; pow on plain R is the
// library's.
#pragma once
#include <type_traits>

#include "klhr_models.cuh"

namespace klhr {
namespace ad {

template <typename R> struct Dual { R v, d; };
template <typename R> struct Tay2 { R v, d, s; };

template <typename S> using if_scalar = std::enable_if_t<std::is_arithmetic<S>::value, int>;
template <typename R> using if_real = std::enable_if_t<std::is_floating_point<R>::value, int>;

// f(x) from f0 = f(v), f1 = f'(v), f2 = f''(v): the chain rule to first / second order
template <typename R>
__device__ __forceinline__ Dual<R> lift(const Dual<R>& x, R f0, R f1, R) { return {f0, f1 * x.d}; }
template <typename R>
__device__ __forceinline__ Tay2<R> lift(const Tay2<R>& x, R f0, R f1, R f2) {
    return {f0, f1 * x.d, f1 * x.s + f2 * x.d * x.d};
}

// ------------------------------------------------------------------ arithmetic
template <typename R> __device__ __forceinline__ Dual<R> operator-(const Dual<R>& a) { return {-a.v, -a.d}; }
template <typename R> __device__ __forceinline__ Tay2<R> operator-(const Tay2<R>& a) { return {-a.v, -a.d, -a.s}; }

template <typename R> __device__ __forceinline__ Dual<R> operator+(const Dual<R>& a, const Dual<R>& b) {
    return {a.v + b.v, a.d + b.d};
}
template <typename R> __device__ __forceinline__ Tay2<R> operator+(const Tay2<R>& a, const Tay2<R>& b) {
    return {a.v + b.v, a.d + b.d, a.s + b.s};
}
template <typename R> __device__ __forceinline__ Dual<R> operator-(const Dual<R>& a, const Dual<R>& b) {
    return {a.v - b.v, a.d - b.d};
}
template <typename R> __device__ __forceinline__ Tay2<R> operator-(const Tay2<R>& a, const Tay2<R>& b) {
    return {a.v - b.v, a.d - b.d, a.s - b.s};
}
template <typename R> __device__ __forceinline__ Dual<R> operator*(const Dual<R>& a, const Dual<R>& b) {
    return {a.v * b.v, a.d * b.v + a.v * b.d};
}
template <typename R> __device__ __forceinline__ Tay2<R> operator*(const Tay2<R>& a, const Tay2<R>& b) {
    return {a.v * b.v, a.d * b.v + a.v * b.d, a.s * b.v + R(2) * a.d * b.d + a.v * b.s};
}
// q = a / b: q' = (a' - q b') / b, q'' = (a'' - 2 q' b' - q b'') / b
template <typename R> __device__ __forceinline__ Dual<R> operator/(const Dual<R>& a, const Dual<R>& b) {
    const R q = a.v / b.v;
    return {q, (a.d - q * b.d) / b.v};
}
template <typename R> __device__ __forceinline__ Tay2<R> operator/(const Tay2<R>& a, const Tay2<R>& b) {
    const R ib = R(1) / b.v, q = a.v / b.v, q1 = (a.d - q * b.d) * ib;
    return {q, q1, (a.s - R(2) * q1 * b.d - q * b.s) * ib};
}

// with an arithmetic scalar (a literal, a data value, an integer), converted to R first
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Dual<R> operator+(const Dual<R>& a, S b) { return {a.v + R(b), a.d}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Dual<R> operator+(S b, const Dual<R>& a) { return {R(b) + a.v, a.d}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Dual<R> operator-(const Dual<R>& a, S b) { return {a.v - R(b), a.d}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Dual<R> operator-(S b, const Dual<R>& a) { return {R(b) - a.v, -a.d}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Dual<R> operator*(const Dual<R>& a, S b) { return {a.v * R(b), a.d * R(b)}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Dual<R> operator*(S b, const Dual<R>& a) { return {R(b) * a.v, R(b) * a.d}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Dual<R> operator/(const Dual<R>& a, S b) { return {a.v / R(b), a.d / R(b)}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Dual<R> operator/(S b, const Dual<R>& a) { return Dual<R>{R(b), R(0)} / a; }

template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Tay2<R> operator+(const Tay2<R>& a, S b) { return {a.v + R(b), a.d, a.s}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Tay2<R> operator+(S b, const Tay2<R>& a) { return {R(b) + a.v, a.d, a.s}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Tay2<R> operator-(const Tay2<R>& a, S b) { return {a.v - R(b), a.d, a.s}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Tay2<R> operator-(S b, const Tay2<R>& a) { return {R(b) - a.v, -a.d, -a.s}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Tay2<R> operator*(const Tay2<R>& a, S b) { return {a.v * R(b), a.d * R(b), a.s * R(b)}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Tay2<R> operator*(S b, const Tay2<R>& a) { return {R(b) * a.v, R(b) * a.d, R(b) * a.s}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Tay2<R> operator/(const Tay2<R>& a, S b) { return {a.v / R(b), a.d / R(b), a.s / R(b)}; }
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Tay2<R> operator/(S b, const Tay2<R>& a) { return Tay2<R>{R(b), R(0), R(0)} / a; }

// compound assignment (sums over observations in a loop)
template <typename A, typename B> __device__ __forceinline__ Dual<A>& operator+=(Dual<A>& a, const B& b) { return a = a + b; }
template <typename A, typename B> __device__ __forceinline__ Dual<A>& operator-=(Dual<A>& a, const B& b) { return a = a - b; }
template <typename A, typename B> __device__ __forceinline__ Dual<A>& operator*=(Dual<A>& a, const B& b) { return a = a * b; }
template <typename A, typename B> __device__ __forceinline__ Dual<A>& operator/=(Dual<A>& a, const B& b) { return a = a / b; }
template <typename A, typename B> __device__ __forceinline__ Tay2<A>& operator+=(Tay2<A>& a, const B& b) { return a = a + b; }
template <typename A, typename B> __device__ __forceinline__ Tay2<A>& operator-=(Tay2<A>& a, const B& b) { return a = a - b; }
template <typename A, typename B> __device__ __forceinline__ Tay2<A>& operator*=(Tay2<A>& a, const B& b) { return a = a * b; }
template <typename A, typename B> __device__ __forceinline__ Tay2<A>& operator/=(Tay2<A>& a, const B& b) { return a = a / b; }

// ------------------------------------------------------------------ elementary functions
__device__ __forceinline__ double r_expm1(double x) { return ::expm1(x); }
__device__ __forceinline__ float r_expm1(float x) { return expm1f(x); }
__device__ __forceinline__ double r_pow(double x, double c) { return ::pow(x, c); }
__device__ __forceinline__ float r_pow(float x, float c) { return powf(x, c); }

// e^-|z| -> softplus(z) = log(1 + e^z), sigma(z), sigma(z) (1 - sigma(z))
template <typename R> __device__ __forceinline__ Softplus<R> softplus_of(R z) { return softplus_q(z, r_exp(-r_abs(z))); }
// tanh(u), 1 - tanh^2(u) = 4 e / (1 + e)^2 with e = e^-2|u|
template <typename R> struct TanhQ { R t, q; };
template <typename R> __device__ __forceinline__ TanhQ<R> tanh_q(R u) {
    const R e = r_exp(R(-2) * r_abs(u));
    const R inv = R(1) / (R(1) + e);
    const R p = (R(1) - e) * inv;
    return {u < R(0) ? -p : p, R(4) * e * inv * inv};
}

#define KLHR_AD_UNARY(name, ...)                                                                      \
    template <typename R> __device__ __forceinline__ Dual<R> name(const Dual<R>& x) {                 \
        const R v = x.v;                                                                              \
        __VA_ARGS__                                                                                   \
        return lift(x, f0, f1, f2);                                                                   \
    }                                                                                                 \
    template <typename R> __device__ __forceinline__ Tay2<R> name(const Tay2<R>& x) {                 \
        const R v = x.v;                                                                              \
        __VA_ARGS__                                                                                   \
        return lift(x, f0, f1, f2);                                                                   \
    }

KLHR_AD_UNARY(exp, const R f0 = r_exp(v), f1 = f0, f2 = f0;)
KLHR_AD_UNARY(log, const R f0 = r_log(v), f1 = R(1) / v, f2 = -f1 * f1;)
KLHR_AD_UNARY(log1p, const R f0 = r_log1p(v), f1 = R(1) / (R(1) + v), f2 = -f1 * f1;)
KLHR_AD_UNARY(expm1, const R f0 = r_expm1(v), f1 = r_exp(v), f2 = f1;)
KLHR_AD_UNARY(sqrt, const R f0 = r_sqrt(v), f1 = R(0.5) / f0, f2 = -R(0.5) * f1 / v;)
KLHR_AD_UNARY(square, const R f0 = v * v, f1 = R(2) * v, f2 = R(2);)
KLHR_AD_UNARY(fabs, const R sg = v < R(0) ? R(-1) : R(1); const R f0 = r_abs(v), f1 = sg, f2 = R(0);)
KLHR_AD_UNARY(tanh, const TanhQ<R> h = tanh_q(v); const R f0 = h.t, f1 = h.q, f2 = R(-2) * h.t * h.q;)
KLHR_AD_UNARY(log1p_exp, const Softplus<R> s = softplus_of(v); const R f0 = s.sp, f1 = s.sg, f2 = s.sg1;)
// log sigma(z) = -softplus(-z): derivative sigma(-z), second derivative -sigma(z) sigma(-z)
KLHR_AD_UNARY(log_inv_logit, const Softplus<R> s = softplus_of(-v); const R f0 = -s.sp, f1 = s.sg, f2 = -s.sg1;)
#undef KLHR_AD_UNARY

// x^c for a constant exponent c
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Dual<R> pow(const Dual<R>& x, S c) {
    const R cr = R(c);
    return lift(x, r_pow(x.v, cr), cr * r_pow(x.v, cr - R(1)), R(0));
}
template <typename R, typename S, if_scalar<S> = 0> __device__ __forceinline__ Tay2<R> pow(const Tay2<R>& x, S c) {
    const R cr = R(c);
    return lift(x, r_pow(x.v, cr), cr * r_pow(x.v, cr - R(1)), cr * (cr - R(1)) * r_pow(x.v, cr - R(2)));
}

// the same names on plain R (those without a CUDA math library counterpart matter: the rest resolve to the library)
template <typename R, if_real<R> = 0> __device__ __forceinline__ R exp(R x) { return r_exp(x); }
template <typename R, if_real<R> = 0> __device__ __forceinline__ R log(R x) { return r_log(x); }
template <typename R, if_real<R> = 0> __device__ __forceinline__ R log1p(R x) { return r_log1p(x); }
template <typename R, if_real<R> = 0> __device__ __forceinline__ R expm1(R x) { return r_expm1(x); }
template <typename R, if_real<R> = 0> __device__ __forceinline__ R sqrt(R x) { return r_sqrt(x); }
template <typename R, if_real<R> = 0> __device__ __forceinline__ R fabs(R x) { return r_abs(x); }
template <typename R, if_real<R> = 0> __device__ __forceinline__ R tanh(R x) { return tanh_q(x).t; }
template <typename R, if_real<R> = 0> __device__ __forceinline__ R square(R x) { return x * x; }
template <typename R, if_real<R> = 0> __device__ __forceinline__ R log1p_exp(R x) { return softplus_of(x).sp; }
template <typename R, if_real<R> = 0> __device__ __forceinline__ R log_inv_logit(R x) { return -softplus_of(-x).sp; }

// the value of any of the three types (for branches on the point, e.g. a piecewise density)
template <typename R, if_real<R> = 0> __device__ __forceinline__ R value(R x) { return x; }
template <typename R> __device__ __forceinline__ R value(const Dual<R>& x) { return x.v; }
template <typename R> __device__ __forceinline__ R value(const Tay2<R>& x) { return x.v; }

}  // namespace ad
}  // namespace klhr
