// klhr_b200 -- the step kernel: every chain advances by whole KLHR draws per launch.
//
// One octet (8 lanes) per chain, kThreads/8 chains per CTA.  Chain state theta and the
// direction rho live in shared memory for the whole launch (n_steps draws): HBM sees one
// read and one write of theta per launch, not per draw.  Per draw (reference
// KLHR.draw klhr.py:196-201):
//   1. direction   Philox4x32-10 -> Box-Muller -> x = mean_j + sd z -> rho = x/||x+tol||
//                  (klhr.py:143-153), or the injected rho in replay mode;
//   2. line setup  Model::setup -> closed-form coefficients of l(y) = lp(theta + y rho);
//   3. fit         stage 1 + stage 2 (klhr_fit.cuh);
//   4. MH          proposal, ratio, accept, theta += zp rho (klhr.py:175-190);
//   5. accumulate  Welford-equivalent raw sums for the pooled adaptation
//                  (onlinemoments.py:10-15 -> raw sums, klhr.py:216-218), thinned draws.
#pragma once
#include "klhr_fit.cuh"
#include "klhr_models.cuh"
#include "klhr_dense.cuh"

namespace klhr {

constexpr int kThreadsMax = 256;
// resident 256-thread CTAs per SM the register budget aims for: 3 (<= 80 registers) measured +7..10% over 2
// on ar1 / ill-normal / funnel; the dense DMMA path keeps 64 accumulator registers and needs 128
#ifndef KLHR_MIN_CTAS
#define KLHR_MIN_CTAS 3
#endif
template <typename R, typename Model>
constexpr int step_min_ctas() { return (Model::kDenseCta && sizeof(R) == 8) ? (kDenseMaxChains > 16 ? 1 : 2) : KLHR_MIN_CTAS; }

struct StepArgs {
    ModelParams mp;
    FitParams fp;
    void* theta;
    long long B;
    int Dpad;
    int serial_d;      // chain kernel: thread-per-chain D-phase (small D), set by its launcher
    // replay inputs
    const void* rho;
    const void* z_init;
    const void* init4;
    const void* z_prop;
    const void* u;
    // free-running
    klhr_direction_t dir;
    long long chain_offset, draw_offset;
    int n_steps;
    unsigned long long seed;
    klhr_accum_t acc;
    klhr_trace_t tr;
};

struct LaunchInfo {
    int threads, smem, regs, ctas_per_sm;
};

__host__ __device__ inline int pad_dim(int D, int real_bytes) {
    // row stride such that the octets of a warp hit disjoint shared-memory banks:
    // stride = 8 (mod 16) doubles, = 8 (mod 32) floats
    const int mod = real_bytes == 8 ? 16 : 32;
    int p = ((D + mod - 1) / mod) * mod + 8;
    if (p - mod >= D) p -= mod;
    return p;
}

// Direction of one chain, by its octet (reference _random_direction, klhr.py:143-153): mean column
// j = searchsorted(cdf, u_col, 'right'), x = mean_j + sd z with z from the chain's Philox stream,
// rho = x / ||x + tol|| left in rh[0..D).  Element i = g0 + lane + 32 t + 8 r  <->  Philox slot
// kSlotDir + lane + 8 t + g0 / 4, word r; x is formed in fp32 (same stream and rounding as the tile kernel).
template <typename R>
__device__ __forceinline__ void octet_direction(const klhr_direction_t& dir, const R* s_sd, const R* s_mean, R* rh,
                                                int D, R tol, R u_col, uint32_t c0, uint32_t c1, uint32_t d0,
                                                uint32_t k0, uint32_t k1d, int lane, unsigned om) {
    const R* mcol = nullptr;
    if (dir.mean_cols) {
        int j = 0;
        if (dir.n_cols > 1) {
            const R* cdf = reinterpret_cast<const R*>(dir.cdf);
            while (j < dir.n_cols - 1 && u_col >= cdf[j]) ++j;
        }
        mcol = j < dir.n_cols - dir.n_zero_cols ? s_mean + (size_t)j * D : nullptr;   // zero column
    }
    R ss = 0;
    for (int g0 = 0; g0 < D; g0 += 128) {
        for (int t = 0; t < 4 && g0 + 32 * t < D; ++t) {
            uint32_t w[4];
            Philox::block(c0, c1, d0, kSlotDir + (uint32_t)(lane + 8 * t) + (uint32_t)(g0 / 4), k0, k1d, w);
            float z[4];
            box_muller_f32(w[0], w[1], z[0], z[1]);
            box_muller_f32(w[2], w[3], z[2], z[3]);
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
                const int i = g0 + lane + 32 * t + 8 * rr;
                if (i < D) {
                    const R x = (R)fmaf((float)s_sd[i], z[rr], mcol ? (float)mcol[i] : 0.0f);
                    rh[i] = x;
                    const R xt = x + tol;
                    ss += xt * xt;
                }
            }
        }
    }
    ss = oct_sum(ss, om);
    const R inv = R(1) / r_sqrt(ss);
    for (int i = lane; i < D; i += kOct) rh[i] *= inv;
}

template <typename R, typename Model, int NE, bool kReplay, bool kAccum>
__global__ void __launch_bounds__(kThreadsMax, step_min_ctas<R, Model>()) step_kernel(const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int D = a.mp.D;
    const int Dpad = a.Dpad;
    const int cpb = blockDim.x / kOct;                 // chains per CTA
    const int o = threadIdx.x / kOct;                  // octet (chain slot) in the CTA
    const int lane = threadIdx.x & (kOct - 1);
    const unsigned om = oct_mask();
    R* sm = reinterpret_cast<R*>(smem_raw);
    R* th = sm + (size_t)o * Dpad;
    R* rh = sm + (size_t)(cpb + o) * Dpad;
    R* a1 = kAccum ? sm + (size_t)(2 * cpb + o) * Dpad : nullptr;
    R* a2 = kAccum ? sm + (size_t)(3 * cpb + o) * Dpad : nullptr;
    R* shared_tail = sm + (size_t)(kAccum ? 4 : 2) * cpb * Dpad;
    R* s_sd = shared_tail;                             // [D]
    R* s_mean = shared_tail + D;                       // [n_cols][D]
    R* s_shift = s_mean + (size_t)(kReplay ? 0 : (a.dir.mean_cols ? a.dir.n_cols : 0)) * D;   // [D]
    __shared__ unsigned long long cta_evals;
    // dense targets in fp64: line coefficients for all chains of the CTA at once on the FP64
    // tensor cores (klhr_dense.cuh); every thread takes part, so the draw loop runs CTA-uniform
    constexpr bool kDense = Model::kDenseCta && sizeof(R) == 8;
    __shared__ double dense_red[kDense ? 8 : 1][kDenseMaxChains][2];

    const long long c = (long long)blockIdx.x * cpb + o;
    const bool valid = c < a.B;
    R* g_theta = reinterpret_cast<R*>(a.theta);

    if (threadIdx.x == 0) cta_evals = 0ull;
    if constexpr (!kReplay) {
        const R* g_sd = reinterpret_cast<const R*>(a.dir.sd);
        const R* g_mean = reinterpret_cast<const R*>(a.dir.mean_cols);
        for (int i = threadIdx.x; i < D; i += blockDim.x) s_sd[i] = g_sd ? g_sd[i] : R(1);
        if (g_mean)
            for (int i = threadIdx.x; i < (a.dir.n_cols - a.dir.n_zero_cols) * D; i += blockDim.x) s_mean[i] = g_mean[i];
    }
    if constexpr (kAccum) {
        const R* g_shift = reinterpret_cast<const R*>(a.acc.shift);
        for (int i = threadIdx.x; i < D; i += blockDim.x) s_shift[i] = g_shift ? g_shift[i] : R(0);
    }
    if (valid) {
        for (int i = lane; i < D; i += kOct) {
            th[i] = g_theta[c * D + i];
            if constexpr (kAccum) { a1[i] = 0; a2[i] = 0; }
        }
    } else if (kDense) {
        for (int i = lane; i < D; i += kOct) { th[i] = 0; rh[i] = 0; }
    }
    __syncthreads();

    long long n_acc = 0;
    unsigned long long n_evals = 0;
    const R tol = (R)a.fp.tol;
    const unsigned long long cid = (unsigned long long)(a.chain_offset + c);

    {
        for (int step = 0; step < a.n_steps; ++step) {
            const long long row = (long long)step * a.B + c;      // trace row
            R z_init = 0, z_prop = 0, u = 0, init2 = 0, init3 = 0;
            if (valid) {
            // ---------------------------------------------------------------- 1. direction
            if constexpr (kReplay) {
                const R* g_rho = reinterpret_cast<const R*>(a.rho);
                for (int i = lane; i < D; i += kOct) rh[i] = g_rho[c * D + i];
                z_init = reinterpret_cast<const R*>(a.z_init)[c];
                z_prop = reinterpret_cast<const R*>(a.z_prop)[c];
                u = reinterpret_cast<const R*>(a.u)[c];
                if (NE == 4) {
                    init2 = reinterpret_cast<const R*>(a.init4)[c * 4 + 2];
                    init3 = reinterpret_cast<const R*>(a.init4)[c * 4 + 3];
                }
            } else {
                const unsigned long long draw = (unsigned long long)(a.draw_offset + step);
                const uint32_t c0 = (uint32_t)cid, c1 = (uint32_t)(cid >> 32);
                const uint32_t k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
                // NOTE: draw index uses 32 bits of the counter; the upper draw bits perturb the key
                const uint32_t d0 = (uint32_t)draw, k1d = k1 ^ (uint32_t)(draw >> 32);
                // scalar variates: lanes 0..3 each expand one slot, then broadcast
                R sv0 = 0, sv1 = 0;
                {
                    uint32_t w[4];
                    Philox::block(c0, c1, d0, (uint32_t)(lane & 3), k0, k1d, w);
                    if ((lane & 3) == 0) {            // slot 0: column uniform, z_init
                        float z0, z1;
                        box_muller_f32(w[2], w[3], z0, z1);
                        sv0 = (R)u01_32(w[0]);
                        sv1 = (R)z0;
                    } else if ((lane & 3) == 1) {     // slot 1: z_prop
                        if (sizeof(R) == 8) {
                            const double z0 = box_muller_f64(u01_53(w[0], w[1]), u01_53(w[2], w[3]));
                            sv0 = (R)z0;
                        } else {
                            float z0, z1;
                            box_muller_f32(w[0], w[2], z0, z1);
                            sv0 = (R)z0;
                        }
                    } else if ((lane & 3) == 2) {     // slot 2: accept uniform
                        sv0 = sizeof(R) == 8 ? (R)u01_53(w[0], w[1]) : (R)u01_32(w[0]);
                    } else {                          // slot 3: sinh start values
                        float z0, z1;
                        box_muller_f32(w[0], w[1], z0, z1);
                        sv0 = (R)z0;
                        sv1 = (R)z1;
                    }
                }
                const R u_col = oct_bcast(sv0, 0, om);
                z_init = oct_bcast(sv1, 0, om);
                z_prop = oct_bcast(sv0, 1, om);
                u = oct_bcast(sv0, 2, om);
                init2 = oct_bcast(sv0, 3, om);
                init3 = oct_bcast(sv1, 3, om);
                octet_direction<R>(a.dir, s_sd, s_mean, rh, D, tol, u_col, c0, c1, d0, k0, k1d, lane, om);
                if (a.tr.z_init) {
                    if (lane == 0) {
                        reinterpret_cast<R*>(a.tr.z_init)[row] = z_init;
                        reinterpret_cast<R*>(a.tr.z_prop)[row] = z_prop;
                        reinterpret_cast<R*>(a.tr.u)[row] = u;
                        if (a.tr.init4) {
                            R* i4 = reinterpret_cast<R*>(a.tr.init4) + row * 4;
                            i4[0] = 0; i4[1] = 0; i4[2] = init2; i4[3] = init3;
                        }
                    }
                }
            }
            __syncwarp(om);
            if (a.tr.rho) {
                R* g = reinterpret_cast<R*>(a.tr.rho) + row * D;
                for (int i = lane; i < D; i += kOct) g[i] = rh[i];
            }
            }   // valid
            // ---------------------------------------------------------------- 2. line setup
            typename Model::Coef cf;
            if constexpr (kDense) {
                double A, Bq;
                dense_cta_quadratic(reinterpret_cast<const double*>(sm), reinterpret_cast<const double*>(sm) + (size_t)cpb * Dpad,
                                    reinterpret_cast<const double*>(a.mp.p0), D, Dpad, cpb, dense_red, o, A, Bq);
                cf.A = (R)A;
                cf.Bq = (R)Bq;
            } else {
                if (valid) cf = Model::setup(th, rh, lane, om, a.mp);
            }
            if (!valid) continue;
            // ---------------------------------------------------------------- 3.+4. fit, propose, MH
            StepOut<R> so;
            OrCtx<R> oc;
            oc.K = a.fp.or_K;
            oc.inject = kReplay;
            oc.r = 0;
            oc.v = 1;
            if (oc.K > 0) {
                if constexpr (kReplay) {
                    oc.r = a.tr.or_r[c];
                    oc.v = reinterpret_cast<const R*>(a.tr.or_v)[c];
                } else {
                    const unsigned long long ocid = (unsigned long long)(a.chain_offset + c);
                    const unsigned long long odraw = (unsigned long long)(a.draw_offset + step);
                    oc.c0 = (uint32_t)ocid; oc.c1 = (uint32_t)(ocid >> 32); oc.d0 = (uint32_t)odraw;
                    oc.k0 = (uint32_t)a.seed; oc.k1d = (uint32_t)(a.seed >> 32) ^ (uint32_t)(odraw >> 32);
                }
            }
            const ClipCtx<R> cc = clip_ctx<R>(a.fp, a.mp, D, th, rh);        // klhr_sinh.py:158-161 (sinh family only)
            fit_and_propose<kOct, R, Model, NE>(cf, a.fp, lane, om, z_init, init2, init3, z_prop, u, so, oc, cc);
            if (!kReplay && oc.K > 0 && a.tr.or_r && lane == 0) {
                a.tr.or_r[row] = oc.r;
                reinterpret_cast<R*>(a.tr.or_v)[row] = oc.v;
            }

            if (so.accept) {
                for (int i = lane; i < D; i += kOct) th[i] = th[i] + so.zp * rh[i];
                ++n_acc;
            }
            n_evals += (unsigned long long)so.evals;
            __syncwarp(om);
            // ---------------------------------------------------------------- traces
            if (lane == 0) {
                if (a.tr.eta) {
                    R* e = reinterpret_cast<R*>(a.tr.eta) + row * NE;
#pragma unroll
                    for (int k = 0; k < NE; ++k) e[k] = so.eta[k];
                }
                if (a.tr.zp) reinterpret_cast<R*>(a.tr.zp)[row] = so.zp;
                if (a.tr.r) reinterpret_cast<R*>(a.tr.r)[row] = so.r;
                if (a.tr.accept) a.tr.accept[row] = so.accept ? 1 : 0;
                if (a.tr.evals) a.tr.evals[row] = so.evals;
            }
            // ---------------------------------------------------------------- 5. accumulate
            if constexpr (kAccum) {
                const bool closure = a.acc.skip_accum_last && step == a.n_steps - 1;
                if (!closure) {
                    for (int i = lane; i < D; i += kOct) {
                        const R d = th[i] - s_shift[i];
                        a1[i] += d;
                        a2[i] += d * d;
                    }
                }
            }
            if (a.acc.draws) {
                const long long gdraw = a.acc.thin_offset + step + 1;
                if (gdraw % a.acc.thin == 0) {
                    R* g = reinterpret_cast<R*>(a.acc.draws) + ((gdraw / a.acc.thin - 1) * a.B + c) * D;
                    for (int i = lane; i < D; i += kOct) g[i] = th[i];
                }
            }
        }
    }
    if (valid) {
        // ------------------------------------------------------------------ write back
        for (int i = lane; i < D; i += kOct) g_theta[c * D + i] = th[i];
        if (lane == 0) {
            if (a.acc.accept_count) a.acc.accept_count[c] += n_acc;
            if (a.acc.evals_total) atomicAdd(&cta_evals, n_evals);
        }
        if constexpr (kAccum) {
            if (a.acc.chain_s1)
                for (int i = lane; i < D; i += kOct) a.acc.chain_s1[c * D + i] += (double)a1[i];
            if (a.acc.chain_s2)
                for (int i = lane; i < D; i += kOct) a.acc.chain_s2[c * D + i] += (double)a2[i];
        }
    }
    __syncthreads();
    if (threadIdx.x == 0 && a.acc.evals_total && cta_evals) atomicAdd(a.acc.evals_total, cta_evals);
    if constexpr (kAccum) {
        if (a.acc.pooled_s1) {
            long long left = a.B - (long long)blockIdx.x * cpb;
            const int nv = left < cpb ? (int)left : cpb;
            for (int i = threadIdx.x; i < D; i += blockDim.x) {
                double t1 = 0, t2 = 0;
                for (int k = 0; k < nv; ++k) {
                    t1 += (double)sm[(size_t)(2 * cpb + k) * Dpad + i];
                    t2 += (double)sm[(size_t)(3 * cpb + k) * Dpad + i];
                }
                atomicAdd(a.acc.pooled_s1 + i, t1);
                atomicAdd(a.acc.pooled_s2 + i, t2);
            }
        }
    }
}

// ------------------------------------------------------------------ full-D model evaluation
template <typename R, typename Model>
__global__ void __launch_bounds__(kThreadsMax) eval_kernel(ModelParams mp, const R* __restrict__ theta,
                                                           R* __restrict__ lp, R* __restrict__ grad,
                                                           long long B, int Dpad) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int D = mp.D;
    const int cpb = blockDim.x / kOct;
    const int o = threadIdx.x / kOct;
    const int lane = threadIdx.x & (kOct - 1);
    const unsigned om = oct_mask();
    R* sm = reinterpret_cast<R*>(smem_raw);
    R* th = sm + (size_t)o * Dpad;
    R* g = grad ? sm + (size_t)(cpb + o) * Dpad : nullptr;
    const long long c = (long long)blockIdx.x * cpb + o;
    if (c >= B) return;
    for (int i = lane; i < D; i += kOct) th[i] = theta[c * D + i];
    __syncwarp(om);
    R v = Model::lp_grad(th, g, lane, om, mp);
    __syncwarp(om);
    // failure semantics of the reference wrapper (bsmodel.py:15-30): -inf and a zero gradient
    bool ok = r_finite(v);
    if (g) {
        bool gok = true;
        for (int i = lane; i < D; i += kOct) gok = gok && r_finite(g[i]);
        ok = ok && (__all_sync(om, gok) != 0);
    }
    if (lane == 0) lp[c] = ok ? v : -Num<R>::inf();
    if (g)
        for (int i = lane; i < D; i += kOct) grad[c * D + i] = ok ? g[i] : R(0);
}

// ------------------------------------------------------------------ KL objective at a given eta
// The reference's KL(eta, rho) (klhr.py:106-120, klhr_sinh.py:163-176) for every chain: value and gradient in
// the reference's own coordinates (m, log s[, log d, e]) -- the fit works in m / s -- plus the Hessian the
// Newton iteration uses.  lp(theta) is added back: the kernels work with l(y) - l(0).
struct KlArgs {
    ModelParams mp;
    FitParams fp;
    const void* theta;   // [B][D]
    const void* rho;     // [B][D]
    const void* eta;     // [B][NE]
    void* f;             // [B]
    void* grad;          // [B][NE]
    void* hess;          // [B][NE][NE] or null
    long long B;
    int Dpad;
    int serial_d;      // chain kernel: thread-per-chain D-phase (small D), set by its launcher
};

template <typename R, typename Model, int NE>
__global__ void __launch_bounds__(kThreadsMax) kl_eval_kernel(const __grid_constant__ KlArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int D = a.mp.D, Dpad = a.Dpad;
    const int cpb = blockDim.x / kOct;
    const int o = threadIdx.x / kOct, lane = threadIdx.x & (kOct - 1);
    const unsigned om = oct_mask();
    R* sm = reinterpret_cast<R*>(smem_raw);
    R* th = sm + (size_t)o * Dpad;
    R* rh = sm + (size_t)(cpb + o) * Dpad;
    const long long c = (long long)blockIdx.x * cpb + o;
    if (c >= a.B) return;
    for (int i = lane; i < D; i += kOct) {
        th[i] = reinterpret_cast<const R*>(a.theta)[c * D + i];
        rh[i] = reinterpret_cast<const R*>(a.rho)[c * D + i];
    }
    __syncwarp(om);
    const typename Model::Coef cf = Model::setup(th, rh, lane, om, a.mp);
    const R lp0 = Model::lp_grad(th, nullptr, lane, om, a.mp);
    R eta[NE];
#pragma unroll
    for (int k = 0; k < NE; ++k) eta[k] = reinterpret_cast<const R*>(a.eta)[c * NE + k];
    KLState<R, NE> S;
    R s;
    if constexpr (NE == 2) {
        kl_gauss<kOct, R, Model>(cf, eta, a.fp, lane, om, S);
        const R clip = (R)a.fp.scale_clip;
        s = r_exp(r_clamp(eta[1], -clip, clip));
    } else {
        kl_sinh<kOct, R, Model>(cf, eta, a.fp, lane, om, S, clip_ctx<R>(a.fp, a.mp, D, th, rh));
        s = sinh_unpack<R>(eta, a.fp).s;
    }
    if (lane != 0) return;
    const R is = R(1) / s;
    reinterpret_cast<R*>(a.f)[c] = S.f - lp0;
    R* g = reinterpret_cast<R*>(a.grad) + c * NE;
#pragma unroll
    for (int k = 0; k < NE; ++k) g[k] = k == 0 ? S.g[0] * is : S.g[k];
    if (a.hess) {
        R* H = reinterpret_cast<R*>(a.hess) + c * NE * NE;
#pragma unroll
        for (int i = 0; i < NE; ++i)
#pragma unroll
            for (int j = 0; j < NE; ++j) H[i * NE + j] = S.H[i][j] * (i == 0 ? is : R(1)) * (j == 0 ? is : R(1));
    }
}

template <typename R, typename Model>
int launch_kl_typed(const KlArgs& args_in, int family, cudaStream_t st) {
    KlArgs a = args_in;
    a.Dpad = pad_dim(a.mp.D, (int)sizeof(R));
    int threads = kThreadsMax;
    size_t smem = 0;
    for (; threads >= 32; threads /= 2) {
        smem = (size_t)2 * (threads / kOct) * a.Dpad * sizeof(R);
        if (smem <= 100 * 1024 || threads == 32) break;
    }
    if (smem > 227 * 1024) return -20;
    const void* fn = family == KLHR_FAMILY_GAUSS ? (const void*)kl_eval_kernel<R, Model, 2>
                                                 : (const void*)kl_eval_kernel<R, Model, 4>;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int cpb = threads / kOct;
    const long long grid = (a.B + cpb - 1) / cpb;
    if (grid <= 0) return 0;
    void* kargs[] = {(void*)&a};
    return (int)cudaLaunchKernel(fn, dim3((unsigned)grid), dim3((unsigned)threads), kargs, smem, st);
}

// ------------------------------------------------------------------ launch helpers
struct LaunchPlan {
    int threads;
    size_t smem;
};

inline LaunchPlan plan_step(int D, int real_bytes, bool accum, int n_cols, bool replay, int max_threads = kThreadsMax,
                            size_t smem_target = 100 * 1024) {
    const int Dpad = pad_dim(D, real_bytes);
    LaunchPlan p;
    for (int threads = max_threads; threads >= 32; threads /= 2) {
        const int cpb = threads / kOct;
        const size_t rows = (size_t)(accum ? 4 : 2) * cpb;
        const size_t tail = (size_t)D * (1 + (replay ? 0 : n_cols) + 1);
        p.threads = threads;
        p.smem = (rows * Dpad + tail) * real_bytes;
        // default target: >= 2 CTAs per SM when possible
        if (p.smem <= smem_target || threads == 32) break;
    }
    return p;
}

template <typename R, typename Model>
int launch_step_typed(const StepArgs& args_in, int family, bool replay, bool accum, cudaStream_t st,
                      LaunchInfo* info) {
    StepArgs a = args_in;
    const int n_cols = a.dir.mean_cols ? a.dir.n_cols : 0;
    // dense DMMA path: as many chains per CTA as fit (every chain sharing the CTA reuses the P fragments)
    constexpr bool dense = Model::kDenseCta && sizeof(R) == 8;
    const LaunchPlan p = plan_step(a.mp.D, (int)sizeof(R), accum, n_cols, replay, dense ? 8 * kDenseMaxChains : kThreadsMax,
                                   dense && kDenseMaxChains > 16 ? (size_t)200 * 1024 : (size_t)100 * 1024);
    if (p.smem > 227 * 1024) return -20;
    a.Dpad = pad_dim(a.mp.D, (int)sizeof(R));
    const void* fn = nullptr;
#define KLHR_PICK(NE, RP, AC) fn = (const void*)step_kernel<R, Model, NE, RP, AC>
    if (family == KLHR_FAMILY_GAUSS) {
        if (replay) KLHR_PICK(2, true, false);
        else if (accum) KLHR_PICK(2, false, true);
        else KLHR_PICK(2, false, false);
    } else {
        if (replay) KLHR_PICK(4, true, false);
        else if (accum) KLHR_PICK(4, false, true);
        else KLHR_PICK(4, false, false);
    }
#undef KLHR_PICK
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem);
    if (e != cudaSuccess) return (int)e;
    if (info) {
        cudaFuncAttributes fa;
        e = cudaFuncGetAttributes(&fa, fn);
        if (e != cudaSuccess) return (int)e;
        int nb = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, p.threads, p.smem);
        if (e != cudaSuccess) return (int)e;
        info->threads = p.threads;
        info->smem = (int)p.smem;
        info->regs = fa.numRegs;
        info->ctas_per_sm = nb;
        return 0;
    }
    const int cpb = p.threads / kOct;
    const long long grid = (a.B + cpb - 1) / cpb;
    if (grid <= 0) return 0;
    void* kargs[] = {(void*)&a};
    e = cudaLaunchKernel(fn, dim3((unsigned)grid), dim3((unsigned)p.threads), kargs, p.smem, st);
    return (int)e;
}

template <typename R, typename Model>
int launch_eval_typed(const ModelParams& mp, const void* theta, void* lp, void* grad, long long B,
                      cudaStream_t st) {
    const int Dpad = pad_dim(mp.D, (int)sizeof(R));
    int threads = kThreadsMax;
    size_t smem = 0;
    for (; threads >= 32; threads /= 2) {
        smem = (size_t)(grad ? 2 : 1) * (threads / kOct) * Dpad * sizeof(R);
        if (smem <= 100 * 1024 || threads == 32) break;
    }
    if (smem > 227 * 1024) return -20;
    const void* fn = (const void*)eval_kernel<R, Model>;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int cpb = threads / kOct;
    const long long grid = (B + cpb - 1) / cpb;
    if (grid <= 0) return 0;
    eval_kernel<R, Model><<<(unsigned)grid, threads, smem, st>>>(
        mp, reinterpret_cast<const R*>(theta), reinterpret_cast<R*>(lp), reinterpret_cast<R*>(grad), B, Dpad);
    return (int)cudaGetLastError();
}

}  // namespace klhr
