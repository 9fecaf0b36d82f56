// klhr_b200 -- the CHAIN kernel: general thread-per-chain fit for every target and both families.
//
// Same two-shape schedule as the tile kernel (klhr_tile.cuh) but with the model-generic line
// setup of the octet kernel:
//   D-phase   8 passes; in pass p octet o handles chain slot 4p+o cooperatively: stage the theta
//             row in shared memory (applying and writing back the previous draw's accepted
//             move), draw rho (Philox -> Box-Muller -> normalise) into the warp's rho tile, and
//             reduce the row pair to the model's line coefficients with Model::setup;
//   fit-phase lane 8o+j owns chain slot 4j+o and runs stage 1 / stage 2 / proposal / MH with
//             G = 1: no shuffles, no 8-fold redundant scalar work, one KL evaluation per trip of
//             the lock-step state machine for 32 chains at once.
// For the non-Gaussian targets (funnel, rosenbrock, arK) and the sinh-arcsinh family the step is
// dominated by the fit, which is why this shape wins over the octet kernel there.
// Small D (<= kChainSerialMaxD: funnel 2 / 11, rosenbrock 4, earnings 4, arK 7): an octet has more lanes than a
// row has elements, and 8 passes of octet reductions cost more than the rows are worth -- the D-phase is then
// thread-per-chain too (a.serial_d): every lane stages its own theta row, draws its own direction (the same
// (slot, word) -> element map, so the same streams) and reduces it with Model::setup<1>, no shuffles.
#pragma once
#include <cstdlib>
#include "klhr_tile.cuh"

namespace klhr {

constexpr int kChainSerialMaxD = 16;

#ifndef KLHR_CHAIN_MINCTAS
#define KLHR_CHAIN_MINCTAS 16   // 128 registers: the extra resident warps beat the small spills (measured, funnel)
#endif

// kDraws: thinned-draw output (MCMCBase.sample rows) as a separate instantiation, like the tile kernel
template <typename R, typename Model, int NE, bool kReplay, bool kDraws>
__global__ void __launch_bounds__(kWarp, KLHR_CHAIN_MINCTAS) chain_kernel(const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int kPasses = 8;
    const int D = a.mp.D;
    const int Dp = a.Dpad;
    const int L = threadIdx.x;
    const int o = L >> 3, j = L & 7;
    const unsigned om = oct_mask();
    const int n_cols = (!kReplay && a.dir.mean_cols) ? a.dir.n_cols : 0;
    const int n_stored = n_cols ? n_cols - a.dir.n_zero_cols : 0;
    // shared memory: th_s[4][Dp] | rho[32][Dp] | sd[D] | mean[n_stored][D] | cdf[n_cols]   (all R)
    // serial D-phase: th[32][Do] | rho[32][Do] | ...  with rows owned by lanes and an ODD pitch Do (conflict-free)
    const bool serial = a.serial_d != 0;
    const int Do = D | 1;
    R* th_all = reinterpret_cast<R*>(smem_raw);
    R* th_s = th_all + (size_t)o * Dp;
    R* rho_all = th_all + (serial ? (size_t)32 * Do : (size_t)4 * Dp);
    R* s_sd = rho_all + (serial ? (size_t)32 * Do : (size_t)32 * Dp);
    R* s_mean = s_sd + D;
    R* s_cdf = s_mean + (size_t)n_stored * D;

    const long long tile0 = (long long)blockIdx.x * 32;
    const long long c_own = tile0 + 4 * j + o;
    const bool own_valid = c_own < a.B;
    R* g_theta = reinterpret_cast<R*>(a.theta);

    if constexpr (!kReplay) {
        const R* g_sd = reinterpret_cast<const R*>(a.dir.sd);
        const R* g_mean = reinterpret_cast<const R*>(a.dir.mean_cols);
        for (int i = L; i < D; i += kWarp) s_sd[i] = g_sd ? g_sd[i] : R(1);
        for (int i = L; i < n_stored * D; i += kWarp) s_mean[i] = g_mean[i];
        if (n_cols > 1)
            for (int i = L; i < n_cols; i += kWarp) s_cdf[i] = reinterpret_cast<const R*>(a.dir.cdf)[i];
    }
    __syncwarp();

    const R tol = (R)a.fp.tol;
    const uint32_t k0 = (uint32_t)a.seed, k1 = (uint32_t)(a.seed >> 32);
    R c_pend = 0;
    long long n_acc = 0;
    unsigned long long n_evals = 0;

    for (int step = 0; step <= a.n_steps; ++step) {
        const bool last = step == a.n_steps;              // extra trip: only flush pending moves
        const unsigned long long draw = (unsigned long long)(a.draw_offset + step);
        const uint32_t d0 = (uint32_t)draw, k1d = k1 ^ (uint32_t)(draw >> 32);
        R u_col = 0, z_init = 0, z_prop = 0, u = 0, init2 = 0, init3 = 0;
        int jcol = 0;
        if (!last) {
            if constexpr (kReplay) {
                if (own_valid) {
                    z_init = reinterpret_cast<const R*>(a.z_init)[c_own];
                    z_prop = reinterpret_cast<const R*>(a.z_prop)[c_own];
                    u = reinterpret_cast<const R*>(a.u)[c_own];
                    if (NE == 4) {
                        init2 = reinterpret_cast<const R*>(a.init4)[c_own * 4 + 2];
                        init3 = reinterpret_cast<const R*>(a.init4)[c_own * 4 + 3];
                    }
                }
            } else {
                const unsigned long long cid = (unsigned long long)(a.chain_offset + c_own);
                chain_scalars<R>((uint32_t)cid, (uint32_t)(cid >> 32), d0, k0, k1d, u_col, z_init, z_prop, u);
                if (NE == 4) {                            // sinh start values, slot 3 (klhr_sinh.py:191)
                    uint32_t w[4];
                    Philox::block((uint32_t)cid, (uint32_t)(cid >> 32), d0, kSlotInit4, k0, k1d, w);
                    float f0, f1;
                    box_muller_f32(w[0], w[1], f0, f1);
                    init2 = (R)f0;
                    init3 = (R)f1;
                }
                if (n_cols > 1)                           // searchsorted(cdf, u, 'right'), klhr.py:147
                    while (jcol < n_cols - 1 && u_col >= s_cdf[jcol]) ++jcol;
            }
        }
        typename Model::Coef my_cf;
        // thinned output: the state after draw g = thin_offset + step (1-based) is staged at the top of the
        // NEXT trip (the extra last trip covers the final draw), so that is where it is written
        const long long g_prev = a.acc.thin_offset + step;
        const bool emit_rt = kDraws && step > 0 && g_prev % a.acc.thin == 0;
        // -------------------------------------------------------------------- D-phase
        if (serial) {
            R* th_row = th_all + (size_t)L * Do;
            R* rh = rho_all + (size_t)L * Do;
            const R cp = c_pend;
            if (own_valid && !(last && cp == R(0) && !emit_rt)) {
                R* row = g_theta + c_own * D;
                R* drow = nullptr;
                if constexpr (kDraws)
                    if (emit_rt) drow = reinterpret_cast<R*>(a.acc.draws) + ((g_prev / a.acc.thin - 1) * a.B + c_own) * D;
                // theta row -> shared, with the pending move of the previous draw applied
                for (int i = 0; i < D; ++i) {
                    R t0 = row[i];
                    if (cp != R(0)) {
                        t0 = t0 + cp * rh[i];
                        row[i] = t0;
                    }
                    th_row[i] = t0;
                    if constexpr (kDraws)
                        if (drow) drow[i] = t0;
                }
            }
            if (!last && own_valid) {
                if constexpr (kReplay) {
                    const R* g_rho = reinterpret_cast<const R*>(a.rho);
                    for (int i = 0; i < D; ++i) rh[i] = g_rho[c_own * D + i];
                } else {
                    const unsigned long long cid = (unsigned long long)(a.chain_offset + c_own);
                    const uint32_t c0 = (uint32_t)cid, c1 = (uint32_t)(cid >> 32);
                    const R* mcol = jcol < n_stored ? s_mean + (size_t)jcol * D : nullptr;
                    R ss = 0;
                    // element i = b + 8 r  <->  Philox slot kSlotDir + b, word r (D <= 16: r = 0, 1 = the two
                    // normals of the block's first Box-Muller pair)
                    for (int b0 = 0; b0 < D && b0 < 8; b0 += 4) {
                        uint32_t w[4][4];
                        Philox::blockN<4>(c0, c1, d0, kSlotDir + (uint32_t)b0, 1u, k0, k1d, w);
#pragma unroll
                        for (int bb = 0; bb < 4; ++bb) {
                            const int i = b0 + bb;
                            if (i < D) {
                                float z0, z1 = 0.0f;
                                if (i + 8 < D) box_muller_f32(w[bb][0], w[bb][1], z0, z1);
                                else z0 = box_muller_f32_cos(w[bb][0], w[bb][1]);
                                const R x = (R)fmaf((float)s_sd[i], z0, mcol ? (float)mcol[i] : 0.0f);
                                rh[i] = x;
                                const R xt = x + tol;
                                ss += xt * xt;
                                if (i + 8 < D) {
                                    const R x1 = (R)fmaf((float)s_sd[i + 8], z1, mcol ? (float)mcol[i + 8] : 0.0f);
                                    rh[i + 8] = x1;
                                    const R xt1 = x1 + tol;
                                    ss += xt1 * xt1;
                                }
                            }
                        }
                    }
                    const R inv = R(1) / r_sqrt(ss);      // rho = x / ||x + tol||  (klhr.py:153)
                    for (int i = 0; i < D; ++i) rh[i] *= inv;
                }
                if (a.tr.rho) {
                    R* g = reinterpret_cast<R*>(a.tr.rho) + ((long long)step * a.B + c_own) * D;
                    for (int i = 0; i < D; ++i) g[i] = rh[i];
                }
                my_cf = Model::template setup<1>(th_row, rh, 0, 0u, a.mp);
            }
            __syncwarp();
        } else
#pragma unroll 1
        for (int p = 0; p < kPasses; ++p) {
            const int cs = 4 * p + o;
            const long long c = tile0 + cs;
            const R cp = oct_bcast(c_pend, p, om);
            const int col = oct_bcast(jcol, p, om);
            if (c >= a.B) continue;                       // octet-uniform
            if (last && cp == R(0) && !emit_rt) continue;
            R* row = g_theta + c * D;
            R* rh = rho_all + (size_t)cs * Dp;
            R* drow = nullptr;
            if constexpr (kDraws)
                if (emit_rt) drow = reinterpret_cast<R*>(a.acc.draws) + ((g_prev / a.acc.thin - 1) * a.B + c) * D;
            // theta row -> shared, with the pending move of the previous draw applied
            for (int i = j; i < D; i += kOct) {
                R t0 = row[i];
                if (cp != R(0)) {
                    t0 = t0 + cp * rh[i];
                    row[i] = t0;
                }
                th_s[i] = t0;
                if constexpr (kDraws)
                    if (drow) drow[i] = t0;
            }
            if (last) continue;
            if constexpr (kReplay) {
                const R* g_rho = reinterpret_cast<const R*>(a.rho);
                for (int i = j; i < D; i += kOct) rh[i] = g_rho[c * D + i];
            } else {
                const unsigned long long cid = (unsigned long long)(a.chain_offset + c);
                const uint32_t c0 = (uint32_t)cid, c1 = (uint32_t)(cid >> 32);
                const R* mcol = col < n_stored ? s_mean + (size_t)col * D : nullptr;
                R ss = 0;
                // element i = g0 + j + 32 t + 8 r  <->  Philox slot kSlotDir + j + 8 t + g0 / 4, word r
                for (int g0 = 0; g0 < D; g0 += 128) {
                    for (int t = 0; t < 4 && g0 + 32 * t < D; ++t) {
                        uint32_t w[4];
                        Philox::block(c0, c1, d0, kSlotDir + (uint32_t)(j + 8 * t) + (uint32_t)(g0 / 4), k0, k1d, w);
                        float z[4];
                        box_muller_f32(w[0], w[1], z[0], z[1]);
                        box_muller_f32(w[2], w[3], z[2], z[3]);
#pragma unroll
                        for (int rr = 0; rr < 4; ++rr) {
                            const int i = g0 + j + 32 * t + 8 * rr;
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
                const R inv = R(1) / r_sqrt(ss);          // rho = x / ||x + tol||  (klhr.py:153)
                for (int i = j; i < D; i += kOct) rh[i] *= inv;
            }
            __syncwarp(om);
            if (a.tr.rho) {
                R* g = reinterpret_cast<R*>(a.tr.rho) + ((long long)step * a.B + c) * D;
                for (int i = j; i < D; i += kOct) g[i] = rh[i];
            }
            // th_s is the next pass's staging row: a model whose Coef keeps its rows reads the chain's global row,
            // which holds the same values (written above, ordered by the __syncwarp) and stays put through the fit
            const R* th_set = CoefKeepsRows<Model>::value ? row : th_s;
            const typename Model::Coef cf = Model::setup(th_set, rh, j, om, a.mp);
            if (j == p) my_cf = cf;
            __syncwarp(om);                               // th_s is reused by the next pass
        }
        if (last) break;
        // -------------------------------------------------------------------- fit phase (thread per chain)
        if (own_valid) {
            StepOut<R> so;
            OrCtx<R> oc;
            oc.K = a.fp.or_K;
            oc.inject = kReplay;
            oc.r = 0;
            oc.v = 1;
            if (oc.K > 0) {
                if constexpr (kReplay) {
                    oc.r = a.tr.or_r[c_own];
                    oc.v = reinterpret_cast<const R*>(a.tr.or_v)[c_own];
                } else {
                    const unsigned long long ocid = (unsigned long long)(a.chain_offset + c_own);
                    const unsigned long long odraw = (unsigned long long)(a.draw_offset + step);
                    oc.c0 = (uint32_t)ocid; oc.c1 = (uint32_t)(ocid >> 32); oc.d0 = (uint32_t)odraw;
                    oc.k0 = (uint32_t)a.seed; oc.k1d = (uint32_t)(a.seed >> 32) ^ (uint32_t)(odraw >> 32);
                }
            }
            // sinh family: elementwise gradient clip of klhr_sinh.py:158-161 (theta row: global memory, already
            // carrying the previous draw's move; rho row: this chain's slot of the warp tile)
            const ClipCtx<R> cc = clip_ctx<R>(a.fp, a.mp, D, g_theta + c_own * D,
                                              serial ? rho_all + (size_t)L * Do : rho_all + (size_t)(4 * j + o) * Dp);
            fit_and_propose<1, R, Model, NE>(my_cf, a.fp, 0, 0u, z_init, init2, init3, z_prop, u, so, oc, cc);
            if (!kReplay && oc.K > 0 && a.tr.or_r) {
                a.tr.or_r[(long long)step * a.B + c_own] = oc.r;
                reinterpret_cast<R*>(a.tr.or_v)[(long long)step * a.B + c_own] = oc.v;
            }

            c_pend = so.accept ? so.zp : R(0);
            n_acc += so.accept ? 1 : 0;
            n_evals += (unsigned long long)so.evals;
            const long long trow = (long long)step * a.B + c_own;
            if (a.tr.eta) {
                R* e = reinterpret_cast<R*>(a.tr.eta) + trow * NE;
#pragma unroll
                for (int k = 0; k < NE; ++k) e[k] = so.eta[k];
            }
            if (a.tr.zp) reinterpret_cast<R*>(a.tr.zp)[trow] = so.zp;
            if (a.tr.r) reinterpret_cast<R*>(a.tr.r)[trow] = so.r;
            if (a.tr.accept) a.tr.accept[trow] = so.accept ? 1 : 0;
            if (a.tr.evals) a.tr.evals[trow] = so.evals;
            if (!kReplay && a.tr.z_init) {
                reinterpret_cast<R*>(a.tr.z_init)[trow] = z_init;
                reinterpret_cast<R*>(a.tr.z_prop)[trow] = z_prop;
                reinterpret_cast<R*>(a.tr.u)[trow] = u;
                if (a.tr.init4) {
                    R* i4 = reinterpret_cast<R*>(a.tr.init4) + trow * 4;
                    i4[0] = 0; i4[1] = 0; i4[2] = init2; i4[3] = init3;
                }
            }
        } else {
            c_pend = 0;
        }
        __syncwarp();
    }
    if (own_valid && a.acc.accept_count) a.acc.accept_count[c_own] += n_acc;
    if (a.acc.evals_total) {
        unsigned long long tot = own_valid ? n_evals : 0ull;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, off);
        if (L == 0 && tot) atomicAdd(a.acc.evals_total, tot);
    }
}

// thread-per-chain D-phase for small D; KLHR_CHAIN_SERIAL=0 in the environment keeps the octet D-phase (measurements)
inline bool chain_serial_d(int D) {
    static const bool on = [] { const char* e = std::getenv("KLHR_CHAIN_SERIAL"); return !(e && e[0] == '0'); }();
    return on && D <= kChainSerialMaxD;
}

inline size_t chain_smem_bytes(const StepArgs& a, int real_bytes, bool replay) {
    const int n_cols = (!replay && a.dir.mean_cols) ? a.dir.n_cols : 0;
    const int n_stored = n_cols ? n_cols - a.dir.n_zero_cols : 0;
    const int Dp = pad_dim(a.mp.D, real_bytes);
    const size_t rows = chain_serial_d(a.mp.D) ? (size_t)64 * (a.mp.D | 1) : (size_t)36 * Dp;
    return (rows + (size_t)(1 + n_stored) * a.mp.D + n_cols) * real_bytes;
}

template <typename R, typename Model>
int launch_chain_typed(const StepArgs& args_in, int family, bool replay, cudaStream_t st, LaunchInfo* info) {
    StepArgs a = args_in;
    a.Dpad = pad_dim(a.mp.D, (int)sizeof(R));
    a.serial_d = chain_serial_d(a.mp.D) ? 1 : 0;
    const size_t smem = chain_smem_bytes(a, (int)sizeof(R), replay);
    if (smem > 227 * 1024) return -20;
    const void* fn;
    const bool draws = !replay && a.acc.draws != nullptr;
    if (family == KLHR_FAMILY_GAUSS)
        fn = replay ? (const void*)chain_kernel<R, Model, 2, true, false>
                    : (draws ? (const void*)chain_kernel<R, Model, 2, false, true>
                             : (const void*)chain_kernel<R, Model, 2, false, false>);
    else
        fn = replay ? (const void*)chain_kernel<R, Model, 4, true, false>
                    : (draws ? (const void*)chain_kernel<R, Model, 4, false, true>
                             : (const void*)chain_kernel<R, Model, 4, false, false>);
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    if (info) {
        cudaFuncAttributes fa;
        e = cudaFuncGetAttributes(&fa, fn);
        if (e != cudaSuccess) return (int)e;
        int nb = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, kWarp, smem);
        if (e != cudaSuccess) return (int)e;
        info->threads = kWarp;
        info->smem = (int)smem;
        info->regs = fa.numRegs;
        info->ctas_per_sm = nb;
        return 0;
    }
    const long long grid = (a.B + 31) / 32;
    if (grid <= 0) return 0;
    void* kargs[] = {(void*)&a};
    e = cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(kWarp), kargs, smem, st);
    return (int)e;
}

}  // namespace klhr
