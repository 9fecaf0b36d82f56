// klhr_b200 -- univariate slice sampling along KLHR's adapted random directions (reference
// slice.py:12-176, one of the algorithms of experiment_accuracy.py:56-64), on the same batch engine:
// octet per chain, theta and rho in shared memory for the whole launch, the direction law of
// klhr_step.cuh (slice.py:148-158 == klhr.py:143-153), and the target seen only through the closed-form
// line restriction g(x) = lp(theta + x rho) - lp(theta) (Model::setup once per draw, O(1) per test).
//
// Per draw (Slice._uni_slice, slice.py:84-146, the reference's working configuration m = inf):
//   log y = g(0) - e, e ~ Exp(1); u ~ U(0, w); L = -u, R = w - u;
//   stepping out: L -= w while L > lower and g(L) > log y; R += w while R < upper and g(R) > log y;
//   shrinkage:    x1 = L + (R - L) U(0,1) until g(x1) >= log y, replacing R (x1 > 0) or L by x1;
//   theta += x1 rho  (every draw moves: acceptance_probability -> 1, slice.py:143-144).
// Variates: e from Philox slot 1, u from slot 2, shrinkage uniforms from slots 0xC0000000 + q (two 53-bit
// uniforms per block in fp64, four 24-bit ones in fp32), or injected in replay mode.
#pragma once
#include "klhr_step.cuh"

namespace klhr {

constexpr uint32_t kSlotSlice = 0xC0000000u;
constexpr int kSliceMaxIter = 1 << 16;     // safety bound of each data-dependent loop (never reached on a proper target)

struct SliceArgs {
    ModelParams mp;
    klhr_slice_t sp;
    void* theta;
    long long B;
    int Dpad;
    double tol;
    // replay inputs
    const void* rho;        // [B][D]
    const void* e;          // [B]
    const void* u0;         // [B]
    const void* shrink_u;   // [B][sp.cap], NaN = not available
    // free-running
    klhr_direction_t dir;
    long long chain_offset, draw_offset;
    int n_steps;
    unsigned long long seed;
    klhr_accum_t acc;
    klhr_trace_t tr;        // zp <- x1, evals, rho, z_init <- e, u <- u0, slice_u, slice_n, accept <- 1
};

template <typename R, typename Model, bool kReplay>
__global__ void __launch_bounds__(kThreadsMax) slice_kernel(const __grid_constant__ SliceArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int D = a.mp.D, Dpad = a.Dpad;
    const int cpb = blockDim.x / kOct;
    const int o = threadIdx.x / kOct, lane = threadIdx.x & (kOct - 1);
    const unsigned om = oct_mask();
    R* sm = reinterpret_cast<R*>(smem_raw);
    R* th = sm + (size_t)o * Dpad;
    R* rh = sm + (size_t)(cpb + o) * Dpad;
    R* s_sd = sm + (size_t)2 * cpb * Dpad;             // [D]
    R* s_mean = s_sd + D;                              // [n stored cols][D]
    if constexpr (!kReplay) {
        const R* g_sd = reinterpret_cast<const R*>(a.dir.sd);
        const R* g_mean = reinterpret_cast<const R*>(a.dir.mean_cols);
        for (int i = threadIdx.x; i < D; i += blockDim.x) s_sd[i] = g_sd ? g_sd[i] : R(1);
        if (g_mean)
            for (int i = threadIdx.x; i < (a.dir.n_cols - a.dir.n_zero_cols) * D; i += blockDim.x) s_mean[i] = g_mean[i];
    }
    const long long c = (long long)blockIdx.x * cpb + o;
    const bool valid = c < a.B;
    R* g_theta = reinterpret_cast<R*>(a.theta);
    if (valid)
        for (int i = lane; i < D; i += kOct) th[i] = g_theta[c * D + i];
    __syncthreads();
    if (!valid) return;

    const R w = (R)a.sp.w, lower = (R)a.sp.lower, upper = (R)a.sp.upper, tol = (R)a.tol;
    const int cap = a.sp.cap;
    const unsigned long long cid = (unsigned long long)(a.chain_offset + c);
    const uint32_t c0 = (uint32_t)cid, c1 = (uint32_t)(cid >> 32);
    const uint32_t k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
    unsigned long long n_evals = 0;

    for (int step = 0; step < a.n_steps; ++step) {
        const long long row = (long long)step * a.B + c;
        const unsigned long long draw = (unsigned long long)(a.draw_offset + step);
        const uint32_t d0 = (uint32_t)draw, k1d = k1 ^ (uint32_t)(draw >> 32);
        R e, u0;
        // ------------------------------------------------------------------ direction + scalar variates
        if constexpr (kReplay) {
            const R* g_rho = reinterpret_cast<const R*>(a.rho);
            for (int i = lane; i < D; i += kOct) rh[i] = g_rho[c * D + i];
            e = reinterpret_cast<const R*>(a.e)[c];
            u0 = reinterpret_cast<const R*>(a.u0)[c];
        } else {
            R sv = 0;
            {
                uint32_t wd[4];
                Philox::block(c0, c1, d0, (uint32_t)(lane & 3), k0, k1d, wd);
                if ((lane & 3) == 0) sv = (R)u01_32(wd[0]);                         // direction column (slot 0)
                else if ((lane & 3) == 1) sv = (R)(-log(u01_53(wd[0], wd[1])));     // e ~ Exp(1)      (slot 1)
                else if ((lane & 3) == 2) sv = sizeof(R) == 8 ? (R)u01_53(wd[0], wd[1]) : (R)u01_32(wd[0]);   // (slot 2)
            }
            const R u_col = oct_bcast(sv, 0, om);
            e = oct_bcast(sv, 1, om);
            u0 = oct_bcast(sv, 2, om);
            octet_direction<R>(a.dir, s_sd, s_mean, rh, D, tol, u_col, c0, c1, d0, k0, k1d, lane, om);
        }
        __syncwarp(om);
        if (a.tr.rho) {
            R* g = reinterpret_cast<R*>(a.tr.rho) + row * D;
            for (int i = lane; i < D; i += kOct) g[i] = rh[i];
        }
        // ------------------------------------------------------------------ line restriction
        const typename Model::Coef cf = Model::setup(th, rh, lane, om, a.mp);
        // ------------------------------------------------------------------ slice (all 8 lanes in lock step)
        const R logy = -e;                                  // g(0) = 0 on the line restriction (slice.py:89-90)
        const R off = w * u0;                               // rng.uniform(0, w), slice.py:92
        R L = R(0) - off, Rr = R(0) + (w - off);
        int evals = 1;
        for (int it = 0; it < kSliceMaxIter; ++it) {        // slice.py:96-101
            if (L <= lower) break;
            const R gl = Model::eval(cf, L).l;
            ++evals;
            if (!(gl > logy)) break;                // NaN counts as -inf (bsmodel.py:15-21)
            L -= w;
        }
        for (int it = 0; it < kSliceMaxIter; ++it) {        // slice.py:102-107
            if (Rr >= upper) break;
            const R gr = Model::eval(cf, Rr).l;
            ++evals;
            if (!(gr > logy)) break;
            Rr += w;
        }
        if (L < lower) L = lower;                           // slice.py:127-128
        if (Rr > upper) Rr = upper;
        R x1 = 0;
        int n_shrink = 0;
        bool done = false;
        uint32_t wq[4];
        int have = 0;
        uint32_t q = 0;
        R* t_su = a.tr.slice_u && !kReplay ? reinterpret_cast<R*>(a.tr.slice_u) + row * cap : nullptr;
        const R* in_su = kReplay ? reinterpret_cast<const R*>(a.shrink_u) + c * cap : nullptr;
        const int max_shrink = kReplay ? cap : kSliceMaxIter;
        while (n_shrink < max_shrink) {                     // slice.py:131-139
            R uk;
            if constexpr (kReplay) {
                uk = in_su[n_shrink];
                if (uk != uk) break;                        // tape exhausted
            } else {
                if (have == 0) {
                    Philox::block(c0, c1, d0, kSlotSlice + q, k0, k1d, wq);
                    ++q;
                    have = sizeof(R) == 8 ? 2 : 4;
                }
                if (sizeof(R) == 8) uk = (R)u01_53(wq[4 - 2 * have], wq[5 - 2 * have]);
                else uk = (R)u01_32(wq[4 - have]);
                --have;
                if (t_su && n_shrink < cap && lane == 0) t_su[n_shrink] = uk;
            }
            ++n_shrink;
            const R cand = L + (Rr - L) * uk;               // rng.uniform(L, R)
            const R gc = Model::eval(cf, cand).l;
            ++evals;
            if (gc >= logy) { x1 = cand; done = true; break; }
            if (cand > R(0)) Rr = cand; else L = cand;
        }
        if (!done) n_shrink = max_shrink + 1;               // stays put (x1 = 0): tape ran out / safety bound
        if (t_su && lane == 0)
            for (int k = n_shrink; k < cap; ++k) t_su[k] = Num<R>::nan();
        for (int i = lane; i < D; i += kOct) th[i] = th[i] + x1 * rh[i];     // slice.py:142
        n_evals += (unsigned long long)evals;
        __syncwarp(om);
        if (lane == 0) {
            if (a.tr.zp) reinterpret_cast<R*>(a.tr.zp)[row] = x1;
            if (a.tr.evals) a.tr.evals[row] = evals;
            if (a.tr.accept) a.tr.accept[row] = 1;
            if (a.tr.slice_n) a.tr.slice_n[row] = n_shrink;
            if (!kReplay && a.tr.z_init) reinterpret_cast<R*>(a.tr.z_init)[row] = e;
            if (!kReplay && a.tr.u) reinterpret_cast<R*>(a.tr.u)[row] = u0;
        }
        if (a.acc.draws) {
            const long long gdraw = a.acc.thin_offset + step + 1;
            if (gdraw % a.acc.thin == 0) {
                R* g = reinterpret_cast<R*>(a.acc.draws) + ((gdraw / a.acc.thin - 1) * a.B + c) * D;
                for (int i = lane; i < D; i += kOct) g[i] = th[i];
            }
        }
        if (a.acc.chain_s1) {
            const R* sh = reinterpret_cast<const R*>(a.acc.shift);
            for (int i = lane; i < D; i += kOct) {
                const double d = (double)th[i] - (sh ? (double)sh[i] : 0.0);
                a.acc.chain_s1[c * D + i] += d;
                if (a.acc.chain_s2) a.acc.chain_s2[c * D + i] += d * d;
            }
        }
    }
    for (int i = lane; i < D; i += kOct) g_theta[c * D + i] = th[i];
    if (lane == 0) {
        if (a.acc.accept_count) a.acc.accept_count[c] += a.n_steps;
        if (a.acc.evals_total) atomicAdd(a.acc.evals_total, n_evals);
    }
}

template <typename R, typename Model>
int launch_slice_typed(const SliceArgs& args_in, bool replay, cudaStream_t st) {
    SliceArgs a = args_in;
    a.Dpad = pad_dim(a.mp.D, (int)sizeof(R));
    const int n_cols = (!replay && a.dir.mean_cols) ? a.dir.n_cols - a.dir.n_zero_cols : 0;
    int threads = kThreadsMax;
    size_t smem = 0;
    for (; threads >= 32; threads /= 2) {
        smem = ((size_t)2 * (threads / kOct) * a.Dpad + (size_t)a.mp.D * (1 + n_cols)) * sizeof(R);
        if (smem <= 100 * 1024 || threads == 32) break;
    }
    if (smem > 227 * 1024) return -20;
    const void* fn = replay ? (const void*)slice_kernel<R, Model, true> : (const void*)slice_kernel<R, Model, false>;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int cpb = threads / kOct;
    const long long grid = (a.B + cpb - 1) / cpb;
    if (grid <= 0) return 0;
    void* kargs[] = {(void*)&a};
    return (int)cudaLaunchKernel(fn, dim3((unsigned)grid), dim3((unsigned)threads), kargs, smem, st);
}

#define KLHR_DECLARE_MODEL_SLICE(name) int launch_slice_##name(const SliceArgs& a, int dtype, bool replay, cudaStream_t st);
#define KLHR_DEFINE_MODEL_SLICE(name, M64, M32)                                                    \
    int launch_slice_##name(const SliceArgs& a, int dtype, bool replay, cudaStream_t st) {         \
        return dtype == KLHR_F64 ? launch_slice_typed<double, M64>(a, replay, st)                  \
                                 : launch_slice_typed<float, M32>(a, replay, st);                  \
    }

KLHR_DECLARE_MODEL_SLICE(normal)
KLHR_DECLARE_MODEL_SLICE(ill_normal)
KLHR_DECLARE_MODEL_SLICE(funnel)
KLHR_DECLARE_MODEL_SLICE(corr_normal)
KLHR_DECLARE_MODEL_SLICE(ar1)
KLHR_DECLARE_MODEL_SLICE(ark)
KLHR_DECLARE_MODEL_SLICE(rosenbrock)
KLHR_DECLARE_MODEL_SLICE(earnings)
KLHR_DECLARE_MODEL_SLICE(eight_schools_nc)
KLHR_DECLARE_MODEL_SLICE(eight_schools_c)
KLHR_DECLARE_MODEL_SLICE(logistic_regression)

}  // namespace klhr
