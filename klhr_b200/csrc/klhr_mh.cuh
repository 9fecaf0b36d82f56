// klhr_b200 -- random-walk Metropolis (reference mh.py:7-37), the comparison sampler of the
// reference's accuracy experiment (experiment_accuracy.py:69), on the same batch engine:
// octet per chain, theta and the proposal staged in shared memory for the whole launch,
// xi ~ N(0, I) from the chain's Philox stream (same element <-> counter mapping as the KLHR
// direction), theta' = theta + stepsize xi, accept iff log u < min(0, lp(theta') - lp(theta))
// (the two proposal-density terms of mh.py:26-27 cancel exactly: the proposal is symmetric).
#pragma once
#include "klhr_step.cuh"

namespace klhr {

struct MhArgs {
    ModelParams mp;
    void* theta;
    long long B;
    int Dpad;
    double stepsize;
    long long chain_offset, draw_offset;
    int n_steps;
    unsigned long long seed;
    klhr_accum_t acc;
    klhr_trace_t tr;       // rho <- xi, r, accept, u
};

template <typename R, typename Model>
__global__ void __launch_bounds__(kThreadsMax) mh_kernel(const __grid_constant__ MhArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int D = a.mp.D, Dpad = a.Dpad;
    const int cpb = blockDim.x / kOct;
    const int o = threadIdx.x / kOct, lane = threadIdx.x & (kOct - 1);
    const unsigned om = oct_mask();
    R* sm = reinterpret_cast<R*>(smem_raw);
    R* th = sm + (size_t)o * Dpad;
    R* tp = sm + (size_t)(cpb + o) * Dpad;
    const long long c = (long long)blockIdx.x * cpb + o;
    if (c >= a.B) return;
    R* g_theta = reinterpret_cast<R*>(a.theta);
    for (int i = lane; i < D; i += kOct) th[i] = g_theta[c * D + i];
    __syncwarp(om);
    R lp = Model::lp_grad(th, nullptr, lane, om, a.mp);
    if (!r_finite(lp)) lp = -Num<R>::inf();                       // mcmc.py:25-29 / bsmodel.py:15-21
    const unsigned long long cid = (unsigned long long)(a.chain_offset + c);
    const uint32_t c0 = (uint32_t)cid, c1 = (uint32_t)(cid >> 32);
    const uint32_t k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
    const R step = (R)a.stepsize;
    long long n_acc = 0;
    for (int s = 0; s < a.n_steps; ++s) {
        const unsigned long long draw = (unsigned long long)(a.draw_offset + s);
        const uint32_t d0 = (uint32_t)draw, k1d = k1 ^ (uint32_t)(draw >> 32);
        const long long row = (long long)s * a.B + c;
        R u;
        {
            uint32_t w[4];
            Philox::block(c0, c1, d0, kSlotAccept, k0, k1d, w);
            u = sizeof(R) == 8 ? (R)u01_53(w[0], w[1]) : (R)u01_32(w[0]);
        }
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
                        const R xi = (R)z[rr];
                        tp[i] = th[i] + xi * step;                // mh.py:22
                        if (a.tr.rho) reinterpret_cast<R*>(a.tr.rho)[row * D + i] = xi;
                    }
                }
            }
        }
        __syncwarp(om);
        R lpp = Model::lp_grad(tp, nullptr, lane, om, a.mp);
        if (!r_finite(lpp)) lpp = -Num<R>::inf();
        const R r = lpp - lp;                                     // mh.py:24-27
        const R rm = r < R(0) ? r : R(0);
        const bool acc = (r == r) && (r_log(u) < rm);             // mh.py:29
        if (acc) {
            for (int i = lane; i < D; i += kOct) th[i] = tp[i];
            lp = lpp;
            ++n_acc;
        }
        __syncwarp(om);
        if (lane == 0) {
            if (a.tr.r) reinterpret_cast<R*>(a.tr.r)[row] = r;
            if (a.tr.accept) a.tr.accept[row] = acc ? 1 : 0;
            if (a.tr.u) reinterpret_cast<R*>(a.tr.u)[row] = u;
        }
        if (a.acc.draws) {
            const long long gdraw = a.acc.thin_offset + s + 1;
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
    if (lane == 0 && a.acc.accept_count) a.acc.accept_count[c] += n_acc;
}

template <typename R, typename Model>
int launch_mh_typed(const MhArgs& args_in, cudaStream_t st) {
    MhArgs a = args_in;
    a.Dpad = pad_dim(a.mp.D, (int)sizeof(R));
    int threads = kThreadsMax;
    size_t smem = 0;
    for (; threads >= 32; threads /= 2) {
        smem = (size_t)2 * (threads / kOct) * a.Dpad * sizeof(R);
        if (smem <= 100 * 1024 || threads == 32) break;
    }
    if (smem > 227 * 1024) return -20;
    const void* fn = (const void*)mh_kernel<R, Model>;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int cpb = threads / kOct;
    const long long grid = (a.B + cpb - 1) / cpb;
    if (grid <= 0) return 0;
    void* kargs[] = {(void*)&a};
    return (int)cudaLaunchKernel(fn, dim3((unsigned)grid), dim3((unsigned)threads), kargs, smem, st);
}

#define KLHR_DECLARE_MODEL_MH(name) int launch_mh_##name(const MhArgs& a, int dtype, cudaStream_t st);
#define KLHR_DEFINE_MODEL_MH(name, M64, M32)                                             \
    int launch_mh_##name(const MhArgs& a, int dtype, cudaStream_t st) {                  \
        return dtype == KLHR_F64 ? launch_mh_typed<double, M64>(a, st) : launch_mh_typed<float, M32>(a, st); \
    }

KLHR_DECLARE_MODEL_MH(normal)
KLHR_DECLARE_MODEL_MH(ill_normal)
KLHR_DECLARE_MODEL_MH(funnel)
KLHR_DECLARE_MODEL_MH(corr_normal)
KLHR_DECLARE_MODEL_MH(ar1)
KLHR_DECLARE_MODEL_MH(ark)
KLHR_DECLARE_MODEL_MH(rosenbrock)
KLHR_DECLARE_MODEL_MH(earnings)
KLHR_DECLARE_MODEL_MH(eight_schools_nc)
KLHR_DECLARE_MODEL_MH(eight_schools_c)
KLHR_DECLARE_MODEL_MH(logistic_regression)

}  // namespace klhr
