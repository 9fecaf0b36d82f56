// klhr_b200 -- the DENSE kernel: stan/corr-normal.stan (dense precision), Gaussian line family, fp64,
// D = 128 or 256; chain state resident in shared memory for the whole launch, 32 chains per CTA.
//
// The line restriction of a Gaussian target needs A = rho' P rho and Bq = -theta' P rho per chain and draw
// (reference klhr.py:106-124 evaluates lp through the full D-vector at every node instead).  With the Cholesky
// factor P = L L' (host, fp64, BSModel) both are inner products of TRIANGULAR images:
//     V = L' rho,   A = V.V,   Bq = -(L' theta).V
// and w = L' theta follows the chain by the same V: theta' = theta + zp rho  =>  w' = w + zp V.  So one
// triangular product per draw (D^2 flops per chain instead of the 2 D^2 of P rho) gives everything, and w never
// has to be recomputed inside a launch (it is rebuilt from theta by the same product when a launch starts).
//
// Shape.  A CTA of 8 warps owns 32 chains.  X (the un-normalised directions, 32 x D) and theta live in shared
// memory; V = X L runs on mma.sync.m8n8k4.f64: warp w owns the column tiles {w, 15-w, 16+w, 31-w} of L (equal
// DMMA counts for every warp although tile n only needs k >= 8 n), its accumulator fragments ARE V for those
// columns, and the matching fragments of w stay in registers for the whole launch -- V and w are never written
// to memory.  The B fragments of L stream L2 -> shared memory through a per-warp cp.async ring 8 k-steps deep
// (the factor is packed on the host in consumption order: each lane copies exactly the 16 bytes it will consume), so the L2 latency sits
// behind 8 x 16 DMMAs.  The fit of a quadratic target is closed form (quad_fit_closed, klhr_lane.cuh); chains
// whose premises fail take the generic iteration of klhr_fit.cuh, so every path returns the same iterates.
// Variate streams are the same function of (seed, chain, draw, element) as in every other kernel.
#pragma once
#ifdef KLHR_DENSE_TIMING
#include <cstdio>
#endif
#include "klhr_lane.cuh"

namespace klhr {

#ifndef KLHR_DENSEK_CHAINS
#define KLHR_DENSEK_CHAINS 32
#endif
// chains per CTA.  Measured on B200 (D = 256, 16 384 chains): 32 chains, one CTA per SM 2.30e8 draws/s; 16 chains, two CTAs
// per SM (their tensor-core and scalar phases interleave, but every L fragment feeds half as many DMMAs and the
// k-loop overhead per DMMA doubles) 2.09e8
constexpr int kDkChains = KLHR_DENSEK_CHAINS;
constexpr int kDkThreads = 256;
constexpr int kDkWarps = kDkThreads / 32;
constexpr int kDkDepth = kDkChains == 16 ? 2 : 4;  // k-PAIRS (8 rows of L) in flight per warp (two CTAs per SM need <= 113 KB each)
constexpr int kDkMT = kDkChains / 8;              // m8 row tiles
constexpr int kDkLpc = kDkThreads / kDkChains;    // lanes per chain in the vector phases (8 or 16)
static_assert(kDkChains == 16 || kDkChains == 32, "dense kernel: 16 or 32 chains per CTA");

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// column tile q (0..NT-1) of warp w: ascending in q, and sum_q tile = const for every warp
__host__ __device__ __forceinline__ int dk_tile(int q, int w) { return (q & 1) ? 8 * (q - 1) + 15 - w : 8 * q + w; }

// The Cholesky factor arrives PACKED in the order the tensor warps consume it (klhr_corr_pack_cholesky, klhr_api.cu;
// klhr_model_t.data1): for column tile nt = 0 .. D/8 - 1, for k-pair p = nt .. D/8 - 1 (rows 8 p .. 8 p + 7: tile nt of
// the lower-triangular L is zero above), for lane = 0 .. 31 (r8 = lane / 4, k4 = lane % 4) the two B-fragment values
//     L[8 p + k4][8 nt + r8],  L[8 p + 4 + k4][8 nt + r8]
// i.e. one 16-byte cp.async and one 128-bit shared load per lane feed the DMMAs of two k-steps, and the stream of a
// tile is contiguous.  Offset of tile nt: 64 (nt T - nt (nt - 1) / 2) doubles, T = D / 8.
__host__ __device__ __forceinline__ long long dk_pack_offset(int nt, int T) { return 64LL * ((long long)nt * T - (long long)nt * (nt - 1) / 2); }
__host__ __device__ __forceinline__ long long dk_pack_doubles(int D) { return dk_pack_offset(D / 8, D / 8); }

// acc[m][q][e] (m < MT row tiles) = sum_k rows[8 m + r8][k] * L[k][8 tile_q + 2 k4 + e]   (k >= 8 tile_q: L is lower triangular)
// rows: [8 MT][S] (double or float) in shared memory; Lp: the packed factor; ring: this warp's [DEPTH][NT][32][2] staging doubles.
template <int MT, int NT, typename XT = double, int DEPTH = kDkDepth>
__device__ __forceinline__ void dk_tri_product(const XT* __restrict__ rows, int S, const double* __restrict__ Lp, int D,
                                               double* ring, int warp, int lane, double (&acc)[MT][NT][2]) {
    const int r8 = lane >> 2, k4 = lane & 3;
#pragma unroll
    for (int m = 0; m < MT; ++m)
#pragma unroll
        for (int q = 0; q < NT; ++q) acc[m][q][0] = acc[m][q][1] = 0.0;
    const int T = D >> 3;
    const int t0 = dk_tile(0, warp);
    int ist[NT];                                       // first k-pair (relative to this warp's first tile) of tile q
    const double* gp[NT];                              // source of tile q for the NEXT k-pair to issue (runs from before its stream)
#pragma unroll
    for (int q = 0; q < NT; ++q) {
        ist[q] = dk_tile(q, warp) - t0;
        gp[q] = Lp + dk_pack_offset(dk_tile(q, warp), T) + 2 * lane - (long long)ist[q] * 64;
    }
    const int n_pairs = T - t0;
    double* my_ring = ring + 2 * lane;
    int i_issue = 0, slot_w = 0;
    auto issue = [&]() {                               // k-pair i_issue into ring slot i_issue % DEPTH
        if (i_issue < n_pairs) {
            double* dst = my_ring + slot_w * (NT * 64);
#pragma unroll
            for (int q = 0; q < NT; ++q)
                if (i_issue >= ist[q]) cp_async16(dst + q * 64, gp[q]);
        }
#pragma unroll
        for (int q = 0; q < NT; ++q) gp[q] += 64;
        cp_async_commit();
        ++i_issue;
        slot_w = (slot_w + 1) & (DEPTH - 1);
    };
#pragma unroll
    for (int i = 0; i < DEPTH - 1; ++i) issue();
    const XT* ar = rows + (size_t)r8 * S + k4 + 8 * t0;
    const size_t s8 = (size_t)8 * S;
    int slot_r = 0;
    auto segment = [&](auto na_tag, int i_begin, int i_end) {
        constexpr int NA = decltype(na_tag)::value;
        for (int i = i_begin; i < i_end; ++i) {
            issue();
            cp_async_wait<DEPTH - 1>();
            const double* slot = my_ring + slot_r * (NT * 64);
            slot_r = (slot_r + 1) & (DEPTH - 1);
            double a0[MT], a1[MT];
            double2 bv[NA];
#pragma unroll
            for (int m = 0; m < MT; ++m) {
                a0[m] = (double)ar[m * s8];
                a1[m] = (double)ar[m * s8 + 4];
            }
            ar += 8;
#pragma unroll
            for (int q = 0; q < NA; ++q) bv[q] = *reinterpret_cast<const double2*>(slot + q * 64);
#pragma unroll
            for (int q = 0; q < NA; ++q)
#pragma unroll
                for (int m = 0; m < MT; ++m) dmma_m8n8k4(acc[m][q][0], acc[m][q][1], a0[m], bv[q].x);
#pragma unroll
            for (int q = 0; q < NA; ++q)
#pragma unroll
                for (int m = 0; m < MT; ++m) dmma_m8n8k4(acc[m][q][0], acc[m][q][1], a1[m], bv[q].y);
        }
    };
    // segment s: tiles 0..s active, k-pairs [ist[s], ist[s+1])
    if constexpr (NT == 2) {
        segment(std::integral_constant<int, 1>{}, 0, ist[1]);
        segment(std::integral_constant<int, 2>{}, ist[1], n_pairs);
    } else {
        segment(std::integral_constant<int, 1>{}, 0, ist[1]);
        segment(std::integral_constant<int, 2>{}, ist[1], ist[2]);
        segment(std::integral_constant<int, 3>{}, ist[2], ist[3]);
        segment(std::integral_constant<int, 4>{}, ist[3], n_pairs);
    }
    cp_async_wait<0>();
}

// sum over the kDkLpc consecutive lanes that share a chain
// gmask: the lanes of the chain's group only -- the groups of a ragged last CTA that hold no chain skip the call
__device__ __forceinline__ double dk_grp_sum(double v, unsigned gmask) {
#pragma unroll
    for (int off = 1; off < kDkLpc; off <<= 1) v += __shfl_xor_sync(gmask, v, off);
    return v;
}

template <int NT, bool kReplay, bool kDraws>
__global__ void __launch_bounds__(kDkThreads, 32 / kDkChains) dense_kernel(const __grid_constant__ StepArgs a) {
    using R = double;
    using Model = CorrNormal<R>;
    constexpr int CH = kDkChains, MT = kDkMT, LPC = kDkLpc;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int D = a.mp.D;                              // 64 NT
    const int S = D + 4;                               // row pitch: = 4 (mod 16) doubles -> conflict-free A fragments
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int o = tid / LPC, j = tid % LPC;            // chain slot o, lane j of the chain's group
    const int r8 = lane >> 2, k4 = lane & 3;
    const int n_cols = (!kReplay && a.dir.mean_cols) ? a.dir.n_cols : 0;
    const int n_stored = n_cols ? n_cols - a.dir.n_zero_cols : 0;
    // shared memory (doubles first): th[CH][S] | xs[CH][S] | ring[8][depth][NT][32] | red[8][CH][2] | s_inv[CH] | s_c[CH]
    //   | s_zi[CH] | s_zp[CH] | s_lu[CH] | s_u[CH] | (floats) sd[D] | mean[n_stored][D] | cdf[n_cols]
    R* th_all = reinterpret_cast<R*>(smem_raw);
    R* xs_all = th_all + (size_t)CH * S;
    R* ring_all = xs_all + (size_t)CH * S;
    R* red = ring_all + (size_t)kDkWarps * kDkDepth * NT * 64;
    R* s_inv = red + kDkWarps * CH * 2;
    R* s_c = s_inv + CH;
    R* s_zi = s_c + CH;
    R* s_zp = s_zi + CH;
    R* s_lu = s_zp + CH;
    R* s_u = s_lu + CH;
    float* s_sd = reinterpret_cast<float*>(s_u + CH);
    float* s_mean = s_sd + D;
    float* s_cdf = s_mean + (size_t)n_stored * D;
    R* th = th_all + (size_t)o * S;
    R* xs = xs_all + (size_t)o * S;
    R* ring = ring_all + (size_t)warp * kDkDepth * NT * 64;

    const long long c = (long long)blockIdx.x * CH + o;             // chain of this lane group
    const bool valid = c < a.B;
    const long long c_fit = (long long)blockIdx.x * CH + tid;       // chain fitted by thread tid < CH
    R* g_theta = reinterpret_cast<R*>(a.theta);
    const R* Lm = reinterpret_cast<const R*>(a.mp.p1);

    if constexpr (!kReplay) {
        const R* g_sd = reinterpret_cast<const R*>(a.dir.sd);
        const R* g_mean = reinterpret_cast<const R*>(a.dir.mean_cols);
        for (int i = tid; i < D; i += kDkThreads) s_sd[i] = g_sd ? (float)g_sd[i] : 1.0f;
        for (int i = tid; i < n_stored * D; i += kDkThreads) s_mean[i] = (float)g_mean[i];
        for (int i = tid; i < n_cols; i += kDkThreads) s_cdf[i] = n_cols > 1 ? (float)reinterpret_cast<const R*>(a.dir.cdf)[i] : 1.0f;
    }
    for (int i = j; i < S; i += LPC) {
        th[i] = (valid && i < D) ? g_theta[c * D + i] : R(0);
        xs[i] = R(0);
    }
    __syncthreads();

    // w = L' theta for this thread's fragment positions (rows 8 m + r8, columns 8 tile_q + 2 k4 + e)
    double wf[MT][NT][2];
    dk_tri_product<MT, NT>(th_all, S, Lm, D, ring, warp, lane, wf);

    const R tol = (R)a.fp.tol;
    const uint32_t k0s = (uint32_t)a.seed, k1s = (uint32_t)(a.seed >> 32);
    const unsigned long long cid = (unsigned long long)(a.chain_offset + c);
    const uint32_t c0 = (uint32_t)cid, c1 = (uint32_t)(cid >> 32);
    long long n_acc = 0;
    unsigned long long n_evals = 0;

    for (int step = 0; step < a.n_steps; ++step) {
        const long long row = (long long)step * a.B + c;
#ifdef KLHR_DENSE_TIMING
        const long long tq0 = clock64();
#endif
        // ---------------------------------------------------------------- A. variates and direction (LPC lanes per chain)
        __syncwarp();                                          // the move below read x elements that other lanes of the group redraw here
        if (valid) {
            if constexpr (kReplay) {
                const R* g_rho = reinterpret_cast<const R*>(a.rho);
                for (int i = j; i < D; i += LPC) xs[i] = g_rho[c * D + i];
                if (j == 0) {
                    const R u = reinterpret_cast<const R*>(a.u)[c];
                    s_inv[o] = R(1);
                    s_zi[o] = reinterpret_cast<const R*>(a.z_init)[c];
                    s_zp[o] = reinterpret_cast<const R*>(a.z_prop)[c];
                    s_u[o] = u;
                    s_lu[o] = r_log(u);
                }
            } else {
                const unsigned long long draw = (unsigned long long)(a.draw_offset + step);
                const uint32_t d0 = (uint32_t)draw, k1d = k1s ^ (uint32_t)(draw >> 32);
                // scalar variates (slots 0..2, same mapping and arithmetic as chain_scalars): lanes 0..2 expand one slot
                // each.  Lanes 1 and 2 both need the logarithm of the 53-bit uniform in (w0, w1): ONE convergent call --
                // as divergent branches these long dependent fp64 chains would run one after the other (a quarter of
                // this phase); only lane 1's square root and cosine remain on their own
                R sv0 = 0;
                if (j < 3) {
                    uint32_t wv[4];
                    Philox::block(c0, c1, d0, (uint32_t)j, k0s, k1d, wv);
                    const R u53 = u01_53(wv[0], wv[1]);
                    const R lg = r_log(u53);
                    float z0, z1;
                    box_muller_f32(wv[2], wv[3], z0, z1);
                    if (j == 0) {
                        sv0 = (R)u01_32(wv[0]);
                        s_zi[o] = (R)z0;
                    } else if (j == 1) {
                        s_zp[o] = sqrt(-2.0 * lg) * cospi(2.0 * u01_53(wv[2], wv[3]));     // = box_muller_f64
                    } else {
                        s_u[o] = u53;
                        s_lu[o] = lg;                          // log of the accept uniform, off the critical path of the fit
                    }
                }
                // group mask, not the full warp: in a ragged last CTA a warp can hold valid and invalid chains, and
                // only the valid groups get here
                const unsigned gmask = (LPC == 32 ? 0xffffffffu : ((1u << LPC) - 1u)) << (LPC * (lane / LPC));
                const R u_col = __shfl_sync(gmask, sv0, 0, LPC);
                int jcol = 0;
                if (n_cols > 1)                                // searchsorted(cdf, u, 'right'), klhr.py:147
                    while (jcol < n_cols - 1 && (float)u_col >= s_cdf[jcol]) ++jcol;
                const float* mcol = (n_cols && jcol < n_stored) ? s_mean + (size_t)jcol * D : nullptr;
                // element i = g0 + j8 + 32 t + 8 r  <->  Philox slot kSlotDir + j8 + 8 t + g0 / 4, word r
                const int j8 = j & 7;
                R ss = 0;
                for (int g0 = 128 * (j >> 3); g0 < D; g0 += 128 * (LPC / 8)) {
                    uint32_t wv[4][4];
                    Philox::blockN<4>(c0, c1, d0, kSlotDir + (uint32_t)j8 + (uint32_t)(g0 / 4), 8u, k0s, k1d, wv);
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        float z[4];
                        box_muller_f32(wv[t][0], wv[t][1], z[0], z[1]);
                        box_muller_f32(wv[t][2], wv[t][3], z[2], z[3]);
#pragma unroll
                        for (int rr = 0; rr < 4; ++rr) {
                            const int i = g0 + j8 + 32 * t + 8 * rr;
                            const R x = (R)fmaf(s_sd[i], z[rr], mcol ? mcol[i] : 0.0f);
                            xs[i] = x;
                            const R xt = x + tol;
                            ss += xt * xt;
                        }
                    }
                }
                ss = dk_grp_sum(ss, gmask);
                if (j == 0) s_inv[o] = R(1) / r_sqrt(ss);      // rho = x / ||x + tol||  (klhr.py:153)
            }
        }
#ifdef KLHR_DENSE_TIMING
        const long long tq1 = clock64();
#endif
        __syncthreads();
#ifdef KLHR_DENSE_TIMING
        const long long tq2 = clock64();
#endif
        // ---------------------------------------------------------------- B. V = X L on the FP64 tensor cores
        double vf[MT][NT][2];
        dk_tri_product<MT, NT>(xs_all, S, Lm, D, ring, warp, lane, vf);
#ifdef KLHR_DENSE_TIMING
        const long long tq3 = clock64();
#endif
#pragma unroll
        for (int m = 0; m < MT; ++m) {
            double pa = 0, pb = 0;
#pragma unroll
            for (int q = 0; q < NT; ++q)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    pa = fma(vf[m][q][e], vf[m][q][e], pa);
                    pb = fma(wf[m][q][e], vf[m][q][e], pb);
                }
            pa += __shfl_xor_sync(0xffffffffu, pa, 1);
            pa += __shfl_xor_sync(0xffffffffu, pa, 2);
            pb += __shfl_xor_sync(0xffffffffu, pb, 1);
            pb += __shfl_xor_sync(0xffffffffu, pb, 2);
            if (k4 == 0) {
                red[(warp * CH + 8 * m + r8) * 2 + 0] = pa;
                red[(warp * CH + 8 * m + r8) * 2 + 1] = pb;
            }
        }
#ifdef KLHR_DENSE_TIMING
        const long long tq4 = clock64();
#endif
        __syncthreads();
#ifdef KLHR_DENSE_TIMING
        const long long tq5 = clock64();
#endif
        // ---------------------------------------------------------------- C. fit, proposal, MH (thread per chain)
        if (tid < CH) {
            R cmove = 0;
            if (c_fit < a.B) {
                double sA = 0, sB = 0;
#pragma unroll
                for (int w8 = 0; w8 < kDkWarps; ++w8) {        // fixed order: deterministic
                    sA += red[(w8 * CH + tid) * 2 + 0];
                    sB += red[(w8 * CH + tid) * 2 + 1];
                }
                const R inv = s_inv[tid];
                typename Model::Coef cf;
                cf.A = __dmul_rn(__dmul_rn(sA, inv), inv);
                cf.Bq = __dmul_rn(-sB, inv);
                const R z_init = s_zi[tid], z_prop = s_zp[tid];
                StepOut<R> so;
                if (!quad_fit_closed(cf.A, cf.Bq, z_init, z_prop, s_lu[tid], a.fp, a.tr.eta != nullptr, so)) {
                    OrCtx<R> oc;
                    oc.K = 0; oc.inject = false; oc.r = 0; oc.v = 1;
                    fit_and_propose<1, R, Model, 2>(cf, a.fp, 0, 0u, z_init, R(0), R(0), z_prop, s_u[tid], so, oc);
                }
                cmove = so.accept ? __dmul_rn(so.zp, inv) : R(0);
                n_acc += so.accept ? 1 : 0;
                n_evals += (unsigned long long)so.evals;
                const long long trow = (long long)step * a.B + c_fit;
                if (a.tr.eta) {
                    R* e = reinterpret_cast<R*>(a.tr.eta) + trow * 2;
                    e[0] = so.eta[0];
                    e[1] = so.eta[1];
                }
                if (a.tr.zp) reinterpret_cast<R*>(a.tr.zp)[trow] = so.zp;
                if (a.tr.r) reinterpret_cast<R*>(a.tr.r)[trow] = so.r;
                if (a.tr.accept) a.tr.accept[trow] = so.accept ? 1 : 0;
                if (a.tr.evals) a.tr.evals[trow] = so.evals;
                if (!kReplay && a.tr.z_init) {
                    reinterpret_cast<R*>(a.tr.z_init)[trow] = z_init;
                    reinterpret_cast<R*>(a.tr.z_prop)[trow] = z_prop;
                    reinterpret_cast<R*>(a.tr.u)[trow] = s_u[tid];
                }
            }
            s_c[tid] = cmove;
        }
#ifdef KLHR_DENSE_TIMING
        const long long tq6 = clock64();
#endif
        __syncthreads();
#ifdef KLHR_DENSE_TIMING
        const long long tq7 = clock64();
#endif
        // ---------------------------------------------------------------- D. move: theta += c x, w += c V
#pragma unroll
        for (int m = 0; m < MT; ++m) {
            const R cm = s_c[8 * m + r8];
#pragma unroll
            for (int q = 0; q < NT; ++q) {
                wf[m][q][0] = fma(cm, vf[m][q][0], wf[m][q][0]);
                wf[m][q][1] = fma(cm, vf[m][q][1], wf[m][q][1]);
            }
        }
        if (valid) {
            if (a.tr.rho) {                                    // rho = x / ||x + tol|| (tests)
                R* g = reinterpret_cast<R*>(a.tr.rho) + row * D;
                const R inv = s_inv[o];
                for (int i = j; i < D; i += LPC) g[i] = xs[i] * inv;
            }
            const R cm = s_c[o];
            if (cm != R(0)) {                                  // 128-bit accesses: the rows are 16-byte aligned (S even)
                double2* t2 = reinterpret_cast<double2*>(th);
                const double2* x2 = reinterpret_cast<const double2*>(xs);
                for (int i = j; i < D / 2; i += LPC) {
                    double2 t = t2[i];
                    const double2 x = x2[i];
                    t.x = fma(cm, x.x, t.x);
                    t.y = fma(cm, x.y, t.y);
                    t2[i] = t;
                }
            }
            if constexpr (kDraws) {
                const long long gdraw = a.acc.thin_offset + step + 1;
                if (gdraw % a.acc.thin == 0) {
                    R* g = reinterpret_cast<R*>(a.acc.draws) + ((gdraw / a.acc.thin - 1) * a.B + c) * D;
                    for (int i = j; i < D; i += LPC) g[i] = th[i];
                }
            }
        }
        // no barrier: phase A of the next draw writes only this group's own xs row and scalars, which nobody
        // else reads before the barrier that follows it; s_c / red are rewritten two barriers from here
#ifdef KLHR_DENSE_TIMING
        if (blockIdx.x == 0 && lane == 0 && step == 40)
            printf("plain warp %d: A %lld | wait %lld | product %lld | fold %lld | wait %lld | C %lld | wait %lld | D %lld\n", warp, tq1 - tq0,
                   tq2 - tq1, tq3 - tq2, tq4 - tq3, tq5 - tq4, tq6 - tq5, tq7 - tq6, clock64() - tq7);
#endif
    }
    if (valid)
        for (int i = j; i < D; i += LPC) g_theta[c * D + i] = th[i];
    if (tid < 32) {
        const bool mine = tid < CH && c_fit < a.B;
        if (mine && a.acc.accept_count) a.acc.accept_count[c_fit] += n_acc;
        if (a.acc.evals_total) {
            unsigned long long tot = mine ? n_evals : 0ull;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, off);
            if (tid == 0 && tot) atomicAdd(a.acc.evals_total, tot);
        }
    }
}

__host__ inline size_t densek_smem_bytes(const StepArgs& a, bool replay) {
    const int D = a.mp.D, S = D + 4, NT = D / 64;
    const int n_cols = (!replay && a.dir.mean_cols) ? a.dir.n_cols : 0;
    const int n_stored = n_cols ? n_cols - a.dir.n_zero_cols : 0;
    size_t b = (size_t)2 * kDkChains * S * 8;                                  // theta, x
    b += (size_t)kDkWarps * kDkDepth * NT * 64 * 8;                            // cp.async rings
    b += (size_t)(kDkWarps * kDkChains * 2 + 6 * kDkChains) * 8;               // red, inv, c, z_init, z_prop, log u, u
    b += (size_t)(D + (size_t)n_stored * D + ((n_cols + 3) & ~3)) * 4;         // sd, mean columns, cdf
    return b;
}
// fp64, Gaussian family, no in-kernel accumulators, standard proposals, Cholesky factor supplied, D = 128 | 256
__host__ inline bool densek_applies(const StepArgs& a, int dtype, int family, bool replay, bool accum, int flags) {
    return !(flags & KLHR_FIT_FORCE_OCTET) && dtype == KLHR_F64 && family == KLHR_FAMILY_GAUSS && !accum &&
           a.fp.or_K == 0 && a.mp.id == KLHR_MODEL_CORR_NORMAL && a.mp.p1 != nullptr &&
           (a.mp.D == 128 || a.mp.D == 256) && densek_smem_bytes(a, replay) <= (size_t)227 * 1024;
}

template <int NT>
int launch_densek_nt(const StepArgs& a, bool replay, cudaStream_t st, LaunchInfo* info) {
    const size_t smem = densek_smem_bytes(a, replay);
    const bool draws = !replay && a.acc.draws != nullptr;
    const void* fn = replay ? (const void*)dense_kernel<NT, true, false>
                            : (draws ? (const void*)dense_kernel<NT, false, true> : (const void*)dense_kernel<NT, false, false>);
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    if (info) {
        cudaFuncAttributes fa;
        e = cudaFuncGetAttributes(&fa, fn);
        if (e != cudaSuccess) return (int)e;
        int nb = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, kDkThreads, smem);
        if (e != cudaSuccess) return (int)e;
        info->threads = kDkThreads;
        info->smem = (int)smem;
        info->regs = fa.numRegs;
        info->ctas_per_sm = nb;
        return 0;
    }
    const long long grid = (a.B + kDkChains - 1) / kDkChains;
    if (grid <= 0) return 0;
    void* kargs[] = {(void*)&a};
    e = cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(kDkThreads), kargs, smem, st);
    return (int)e;
}

// defined in klhr_densek.cu
int launch_densek(const StepArgs& a, bool replay, cudaStream_t st, LaunchInfo* info);

}  // namespace klhr
