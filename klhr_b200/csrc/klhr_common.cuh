// klhr_b200 -- device-side building blocks shared by all kernels (sm_100a).
//
// Execution shapes.  An OCTET (8 consecutive lanes of a warp) cooperates on one chain for
// everything that walks the D-vector (direction, line setup, update): 8 interleaved slices,
// 3-level xor-shuffle reductions confined to the octet.  The line fit runs either on the same
// octet (klhr_step.cuh: the 8 lanes are the 8 Gauss-Hermite nodes of klhr.py:110-117 and the 8
// back-tracking candidates of the mode search) or thread-per-chain (klhr_tile.cuh,
// klhr_chain.cuh: a warp owns 32 chains, lane 8o+j fits the chain octet o handled in pass j).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "klhr_math.cuh"

namespace klhr {

constexpr int kOct = 8;                 // lanes per chain
constexpr int kMaxNodes = 32;           // quadrature nodes supported (reference default N = 8)

__device__ __forceinline__ unsigned oct_mask() {
    return 0xFFu << ((threadIdx.x & 31u) & 24u);
}

template <typename R>
__device__ __forceinline__ R oct_sum(R v, unsigned m) {
    v += __shfl_xor_sync(m, v, 1);
    v += __shfl_xor_sync(m, v, 2);
    v += __shfl_xor_sync(m, v, 4);
    return v;
}

// sum over the G lanes that cooperate on one chain: G = 8 an octet, G = 1 a single thread (no shuffle)
template <int G, typename R>
__device__ __forceinline__ R grp_sum(R v, unsigned m) {
    if constexpr (G == kOct) return oct_sum(v, m);
    else return v;
}

// broadcast from lane `src` (0..7) of this octet
template <typename R>
__device__ __forceinline__ R oct_bcast(R v, int src, unsigned m) {
    return __shfl_sync(m, v, src, kOct);
}

// ------------------------------------------------------------------ Real traits
template <typename R> struct Num;
template <> struct Num<double> {
    static constexpr double eps = 2.220446049250313e-16;
    __device__ static __forceinline__ double inf() { return __longlong_as_double(0x7ff0000000000000LL); }
    __device__ static __forceinline__ double nan() { return __longlong_as_double(0x7ff8000000000000LL); }
};
template <> struct Num<float> {
    static constexpr float eps = 1.1920929e-07f;
    __device__ static __forceinline__ float inf() { return __int_as_float(0x7f800000); }
    __device__ static __forceinline__ float nan() { return __int_as_float(0x7fc00000); }
};

__device__ __forceinline__ double r_exp(double x) { return exp_c(x); }
__device__ __forceinline__ float r_exp(float x) { return expf(x); }
__device__ __forceinline__ double r_log(double x) { return log_c(x); }
__device__ __forceinline__ float r_log(float x) { return logf(x); }
__device__ __forceinline__ double r_log1p(double x) { return log1p(x); }
__device__ __forceinline__ float r_log1p(float x) { return log1pf(x); }
__device__ __forceinline__ double r_sqrt(double x) { return sqrt(x); }
__device__ __forceinline__ double r_rsqrt(double x) { return rsqrt(x); }
__device__ __forceinline__ float r_rsqrt(float x) { return rsqrtf(x); }
__device__ __forceinline__ float r_sqrt(float x) { return sqrtf(x); }
// 1 / x for a finite, normal x whose reciprocal is normal too: hardware seed (20 bits) + two Newton steps, no
// special-case branches (the IEEE division spends ~25 dependent instructions on them); within 1 ulp
__device__ __forceinline__ double r_rcp_normal(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-x, y, 1.0);
    y = fma(y, e, y);
    e = fma(-x, y, 1.0);
    return fma(y, e, y);
}
__device__ __forceinline__ float r_rcp_normal(float x) { return 1.0f / x; }
__device__ __forceinline__ double r_abs(double x) { return fabs(x); }
__device__ __forceinline__ float r_abs(float x) { return fabsf(x); }
__device__ __forceinline__ double r_sinh(double x) { return sinh(x); }
__device__ __forceinline__ float r_sinh(float x) { return sinhf(x); }
__device__ __forceinline__ double r_cosh(double x) { return cosh(x); }
__device__ __forceinline__ float r_cosh(float x) { return coshf(x); }
__device__ __forceinline__ double r_tanh(double x) { return tanh(x); }
__device__ __forceinline__ float r_tanh(float x) { return tanhf(x); }
__device__ __forceinline__ double r_asinh(double x) { return asinh(x); }
__device__ __forceinline__ float r_asinh(float x) { return asinhf(x); }
__device__ __forceinline__ bool r_finite(double x) { return isfinite(x); }
__device__ __forceinline__ bool r_finite(float x) { return isfinite(x); }
template <typename R> __device__ __forceinline__ R r_clamp(R v, R lo, R hi) { return v < lo ? lo : (v > hi ? hi : v); }
template <typename R> __device__ __forceinline__ R r_max(R a, R b) { return a > b ? a : b; }

// ------------------------------------------------------------------ line restriction value
// (l(y) - l(0), l'(y), l''(y)); non-finite anywhere -> (-inf, 0, 0): the batched form of the
// reference wrapper's "failure => -inf / zero gradient" (bsmodel.py:15-30).
template <typename R> struct Jet { R l, l1, l2; };

template <typename R>
__device__ __forceinline__ Jet<R> jet_guard(R l, R l1, R l2) {
    Jet<R> j;
    const bool ok = r_finite(l) && r_finite(l1) && r_finite(l2);
    j.l = ok ? l : -Num<R>::inf();
    j.l1 = ok ? l1 : R(0);
    j.l2 = ok ? l2 : R(0);
    return j;
}

// ------------------------------------------------------------------ elementwise gradient clip (sinh family)
struct ModelParams;
constexpr int kClipMaxD = 16;

template <typename R>
struct ClipCtx {
    R c;                     // clip threshold; <= 0: off
    const R* th;             // theta row of the chain (shared or global memory)
    const R* rh;             // rho row
    const ModelParams* mp;
    int D;
    __device__ __forceinline__ bool on() const { return c > R(0); }
};

template <typename R>
__device__ __forceinline__ ClipCtx<R> clip_off() {
    ClipCtx<R> cc;
    cc.c = R(0); cc.th = nullptr; cc.rh = nullptr; cc.mp = nullptr; cc.D = 0;
    return cc;
}

template <typename R, typename Model>
__device__ __noinline__ R clip_l1_slow(R y, R l1, const ClipCtx<R>& cc) {
    R pt[kClipMaxD], g[kClipMaxD];
    for (int i = 0; i < cc.D; ++i) pt[i] = cc.th[i] + y * cc.rh[i];
    Model::template lp_grad<1>(pt, g, 0, 0u, *cc.mp);
    bool any = false;
    R acc = 0;
    for (int i = 0; i < cc.D; ++i) {
        const R gi = g[i];
        const R ci = r_clamp(gi, -cc.c, cc.c);
        any = any || (ci != gi);
        acc += ci * cc.rh[i];
    }
    return any ? acc : l1;
}

// default Model::eval_clip: full gradient wherever the evaluation is finite (models with a cheap test for "no
// component can exceed c" specialise it, see Funnel)
template <typename R, typename Model>
__device__ __forceinline__ Jet<R> eval_clip_generic(const typename Model::Coef& cf, R y, const ClipCtx<R>& cc, R& l1c) {
    const Jet<R> J = Model::eval(cf, y);
    l1c = J.l1;
    if (r_finite(J.l)) l1c = clip_l1_slow<R, Model>(y, J.l1, cc);
    return J;
}

// ------------------------------------------------------------------ Philox4x32-10
// Counter-based generator (Salmon et al. 2011): zero bytes of RNG state per chain.
// counter = (chain_lo, chain_hi, draw, slot), key = (seed_lo, seed_hi).
struct Philox {
    static constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
    static constexpr uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    __host__ __device__ static inline void block(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                 uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            const uint64_t p0 = (uint64_t)M0 * c0;
            const uint64_t p1 = (uint64_t)M1 * c2;
            const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
            const uint32_t n1 = (uint32_t)p1;
            const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
            const uint32_t n3 = (uint32_t)p0;
            c0 = n0; c1 = n1; c2 = n2; c3 = n3;
            k0 += W0; k1 += W1;
        }
        out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
    }
    // NB blocks whose counters differ only in c3 = slot0 + stride * b, advanced round by round
    // so that the 8 independent multiplies per round overlap (one block alone is a serial chain).
    template <int NB>
    __device__ static __forceinline__ void blockN(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t slot0,
                                                   uint32_t stride, uint32_t k0, uint32_t k1, uint32_t out[NB][4]) {
        uint32_t s[NB][4];
#pragma unroll
        for (int b = 0; b < NB; ++b) { s[b][0] = c0; s[b][1] = c1; s[b][2] = c2; s[b][3] = slot0 + stride * b; }
#pragma unroll
        for (int r = 0; r < 10; ++r) {
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                const uint64_t p0 = (uint64_t)M0 * s[b][0];
                const uint64_t p1 = (uint64_t)M1 * s[b][2];
                const uint32_t n0 = (uint32_t)(p1 >> 32) ^ s[b][1] ^ k0;
                const uint32_t n2 = (uint32_t)(p0 >> 32) ^ s[b][3] ^ k1;
                s[b][0] = n0; s[b][1] = (uint32_t)p1; s[b][2] = n2; s[b][3] = (uint32_t)p0;
            }
            k0 += W0; k1 += W1;
        }
#pragma unroll
        for (int b = 0; b < NB; ++b)
#pragma unroll
            for (int q = 0; q < 4; ++q) out[b][q] = s[b][q];
    }
};

// slots of one (chain, draw) stream
constexpr uint32_t kSlotScalarA = 0;   // w0: direction-column uniform; w2,w3: z_init pair
constexpr uint32_t kSlotProposal = 1;  // w0..w3: two 53-bit uniforms -> Box-Muller -> z_prop
constexpr uint32_t kSlotAccept = 2;    // w0,w1: 53-bit accept uniform
constexpr uint32_t kSlotInit4 = 3;     // w0..w3: two Box-Muller pairs -> init4[2], init4[3] (sinh)
constexpr uint32_t kSlotDir = 8;       // direction element i: slot kSlotDir + (i % 8) + 8 ((i % 128) / 32) + 32 (i / 128), word (i % 32) / 8

// uniform from the top 24 bits: (x >> 8 + 0.5) / 2^24, rounded to fp32.  The range is [2^-25, 1], not (0, 1): from
// 1/2 up the lattice points fall halfway between fp32 neighbours and round to even, the top one (x >= 0xFFFFFF00,
// probability 2^-24) to exactly 1.0.  Where this uniform is used that is harmless: a Box-Muller radius of 0 (one zero
// normal), the last direction column, a rejected draw (log u = 0), a slice candidate at the bracket end, a binomial
// trial P(u < u0) off u0 by at most 2^-24.  Exponentials must not be formed from it: see exp1_32.
__device__ __forceinline__ float u01_32(uint32_t x) { return fmaf((float)(x >> 8), 1.0f / 16777216.0f, 0.5f / 16777216.0f); }
// -log u of the same lattice point u = (x >> 8 + 0.5) / 2^24, an Exp(1) variate: -log u below 1/2, where u is exact
// in fp32, and -log1p(-(1 - u)) from 1/2 up, where 1 - u is the lattice point of ~x, exact as well.  So it is never 0
// and keeps fp32 relative accuracy (logf, log1pf: 1 ulp) down to its smallest value 2^-25.
__device__ __forceinline__ float exp1_32(uint32_t x) {
    return x < 0x80000000u ? -logf(u01_32(x)) : -log1pf(-u01_32(~x));
}
// uniform in (0,1) from 53 of 64 bits
__device__ __forceinline__ double u01_53(uint32_t hi, uint32_t lo) {
    const uint64_t v = (((uint64_t)hi << 32) | lo) >> 11;
    return ((double)v + 0.5) * (1.0 / 9007199254740992.0);
}

// Box-Muller, single precision, fast intrinsics: direction normals only need to be a valid
// random direction law (any rho is a valid hit-and-run direction), not 1-ulp accurate.
__device__ __forceinline__ void box_muller_f32(uint32_t a, uint32_t b, float& z0, float& z1) {
    const float u = u01_32(a);
    // -2 ln u = (-2 ln 2) lg2 u ; MUFU.LG2, MUFU.SQRT, MUFU.SIN/COS (approximate units are fine
    // for a direction law; the proposal normal uses box_muller_f64)
    // u >= 2^-25 is never denormal: the .ftz forms skip the denormal fix-up __log2f would add
    float lg, rad;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(u));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad) : "f"(-1.3862943611198906f * lg));
    const float ang = (float)b * 1.4629180792671596e-09f;       // 2 pi / 2^32 * b
    z0 = rad * __cosf(ang);
    z1 = rad * __sinf(ang);
}

// z0 of box_muller_f32 alone (same operations, same bits), where the sine branch has no coordinate to go to
__device__ __forceinline__ float box_muller_f32_cos(uint32_t a, uint32_t b) {
    const float u = u01_32(a);
    float lg, rad;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(u));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad) : "f"(-1.3862943611198906f * lg));
    const float ang = (float)b * 1.4629180792671596e-09f;
    return rad * __cosf(ang);
}

// One fp64 normal from two 53-bit uniforms (the proposal variate): only the cosine branch is ever used
__device__ __forceinline__ double box_muller_f64(double u, double v) {
    return sqrt(-2.0 * log_c(u)) * cospi(2.0 * v);
}

}  // namespace klhr
