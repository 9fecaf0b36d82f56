// klhr_b200 -- extern "C" entry points of libklhr_sm100.so (include/klhr_sm100.h).
// Validation, error strings and dispatch only; the kernels are in klhr_step.cuh and the
// per-model translation units.
#include <atomic>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <mutex>
#include <string>

#include "klhr_chain.cuh"
#include "klhr_lane.cuh"
#include "klhr_densek.cuh"
#include "klhr_mh.cuh"
#include "klhr_slice.cuh"

namespace klhr {

static thread_local std::string g_last_error;

static int fail(int code, const char* msg) {
    g_last_error = msg;
    return code;
}

static int cuda_fail(int e, const char* where) {
    if (e > 0) {
        g_last_error = std::string(where) + ": " + cudaGetErrorString((cudaError_t)e);
    } else if (e == -20) {
        g_last_error = std::string(where) + ": dimension too large for the shared-memory staged step";
    }
    return e;
}

// ------------------------------------------------------------------ user targets
// Launcher tables of the user target libraries registered in this process (klhr_user_register).  A slot is written
// once, before the count that publishes it, and never changes, so the dispatchers read it without the lock.
constexpr int kUserSlots = 64;
static klhr_user_table_t g_user[kUserSlots];
static std::atomic<int> g_user_count{0};
static std::mutex g_user_mutex;

// ------------------------------------------------------------------ built-in targets
// Launcher tables of the built-in targets (klhr_model_*.cu), indexed by model id.
extern const klhr_user_table_t kNormalLaunchers, kIllNormalLaunchers, kFunnelLaunchers, kCorrNormalLaunchers,
    kAr1Launchers, kArkLaunchers, kRosenbrockLaunchers, kEarningsLaunchers, kEightSchoolsNCLaunchers,
    kEightSchoolsCLaunchers, kLogisticRegressionLaunchers, kArma11Launchers;

struct BuiltinTargets { const klhr_user_table_t* t[KLHR_MODEL_USER]; };

constexpr BuiltinTargets builtin_targets() {
    BuiltinTargets b{};
    b.t[KLHR_MODEL_NORMAL] = &kNormalLaunchers;
    b.t[KLHR_MODEL_ILL_NORMAL] = &kIllNormalLaunchers;
    b.t[KLHR_MODEL_FUNNEL] = &kFunnelLaunchers;
    b.t[KLHR_MODEL_CORR_NORMAL] = &kCorrNormalLaunchers;
    b.t[KLHR_MODEL_AR1] = &kAr1Launchers;
    b.t[KLHR_MODEL_ARK] = &kArkLaunchers;
    b.t[KLHR_MODEL_ROSENBROCK] = &kRosenbrockLaunchers;
    b.t[KLHR_MODEL_EARNINGS] = &kEarningsLaunchers;
    b.t[KLHR_MODEL_EIGHT_SCHOOLS_NC] = &kEightSchoolsNCLaunchers;
    b.t[KLHR_MODEL_EIGHT_SCHOOLS_C] = &kEightSchoolsCLaunchers;
    b.t[KLHR_MODEL_LOGISTIC_REGRESSION] = &kLogisticRegressionLaunchers;
    b.t[KLHR_MODEL_ARMA11] = &kArma11Launchers;
    return b;
}

constexpr BuiltinTargets kBuiltin = builtin_targets();

constexpr bool every_id_has_a_table(const BuiltinTargets& b) {
    for (const klhr_user_table_t* t : b.t)
        if (!t) return false;
    return true;
}
static_assert(every_id_has_a_table(kBuiltin), "a model id below KLHR_MODEL_USER has no launcher table");

// The launchers of a descriptor that passed check_model.
static const klhr_user_table_t& launchers(const ModelParams& mp) {
    return mp.id == KLHR_MODEL_USER ? g_user[mp.i0] : *kBuiltin.t[mp.id];
}

static int check_model(const klhr_model_t* m, ModelParams& mp) {
    if (!m) return fail(-1, "model is NULL");
    if (m->id < 0 || m->id >= KLHR_MODEL_COUNT)
        return fail(-2, "unknown model id: no device implementation (there is no CPU fallback)");
    if (m->dim <= 0) return fail(-3, "model dim must be positive");
    mp.id = m->id; mp.D = m->dim; mp.i0 = m->i0; mp.i1 = m->i1;
    mp.s0 = m->s0; mp.s1 = m->s1; mp.p0 = m->data0; mp.p1 = m->data1;
    switch (m->id) {
        case KLHR_MODEL_ILL_NORMAL:
            if (!m->data0) return fail(-4, "ill-normal needs data0 = inv_s2[D]");
            break;
        case KLHR_MODEL_CORR_NORMAL:
            if (!m->data0) return fail(-4, "corr-normal needs data0 = P[D*D]");
            break;
        case KLHR_MODEL_FUNNEL:
            if (m->i0 != m->dim - 1) return fail(-5, "funnel: dim must equal i0 + 1");
            break;
        case KLHR_MODEL_ARK:
            if (!m->data0 || m->i0 < 0 || m->dim != m->i0 + 2 || m->i1 <= 0)
                return fail(-5, "arK: need data0 = [G|c|yy], dim = K + 2, i1 = T - K > 0");
            break;
        case KLHR_MODEL_ROSENBROCK:
            if (m->dim != 2 * m->i0) return fail(-5, "rosenbrock: dim must equal 2 * i0");
            break;
        case KLHR_MODEL_AR1:
            if (!(m->s1 > 0)) return fail(-5, "ar1: s1 = 1/beta^2 must be positive");
            break;
        case KLHR_MODEL_EARNINGS:
            if (!m->data0 || m->dim != 4) return fail(-5, "earnings: need data0 = [N,Se,Sh,See,Seh,Shh], dim = 4");
            break;
        case KLHR_MODEL_EIGHT_SCHOOLS_NC:
        case KLHR_MODEL_EIGHT_SCHOOLS_C:
            if (!m->data0 || m->i0 < 1 || m->dim != m->i0 + 2)
                return fail(-5, "eight schools: need data0 = [y|w], i0 = J >= 1, dim = J + 2");
            break;
        case KLHR_MODEL_LOGISTIC_REGRESSION:
            if (m->i0 < 0) return fail(-5, "logistic regression: i0 = N must be >= 0");
            if (m->i1 < 1) return fail(-5, "logistic regression: i1 = K must be >= 1");
            if (m->dim != m->i1 + 1) return fail(-5, "logistic regression: dim must equal i1 + 1 = K + 1");
            if (!m->data0 && m->i0 > 0) return fail(-5, "logistic regression: need data0 = [X|y] when N > 0");
            break;
        case KLHR_MODEL_ARMA11:
            if (m->i0 < 1) return fail(-5, "arma11: i0 = T must be >= 1");
            if (m->dim != 4) return fail(-5, "arma11: dim must be 4 ([mu, a, b, v])");
            if (!m->data0) return fail(-5, "arma11: need data0 = y[T]");
            break;
        case KLHR_MODEL_USER:
            if (m->i0 < 0 || m->i0 >= g_user_count.load(std::memory_order_acquire))
                return fail(-5, "user target: i0 is not a registered slot (klhr_user_register)");
            if (m->i1 < 0) return fail(-5, "user target: i1 = number of data fields must be >= 0");
            if (m->i1 > 0 && (!m->data0 || !m->data1))
                return fail(-5, "user target: data fields declared (i1 > 0) need data0 = values and data1 = field table");
            break;
        default: break;
    }
    return 0;
}

static int check_fit(const klhr_fit_t* f, FitParams& fp) {
    if (!f) return fail(-1, "fit is NULL");
    if (f->family != KLHR_FAMILY_GAUSS && f->family != KLHR_FAMILY_SINH) return fail(-6, "unknown family");
    if (f->n_nodes < 1 || f->n_nodes > KLHR_MAX_NODES) return fail(-7, "n_nodes out of range");
    if (f->n1 < 0 || f->n2 < 0 || f->nb < 1) return fail(-8, "iteration budgets out of range");
    fp.family = f->family; fp.N = f->n_nodes; fp.n1 = f->n1; fp.n2 = f->n2; fp.nb = f->nb;
    fp.kmax = (f->kmax > 0 && f->kmax < 1 + f->n2 * f->nb) ? f->kmax : 1 + f->n2 * f->nb;
    if (f->overrelax_K < 0 || f->overrelax_K > 50) return fail(-8, "overrelax_K must be in 0..50 (klhr.py:213)");
    fp.or_K = f->overrelax_K;
    fp.fix_d = (f->flags & KLHR_FIT_FIX_D) ? 1 : 0;
    fp.initscale = f->initscale; fp.tol = f->tol; fp.scale_clip = f->scale_clip;
    fp.gtol1 = f->gtol1; fp.gtol2 = f->gtol2; fp.step_cap = f->step_cap; fp.c1 = f->c1; fp.basin = f->basin;
    if (f->grad_clip < 0) return fail(-8, "grad_clip must be >= 0 (0 = no clip)");
    fp.grad_clip = f->grad_clip;
    for (int i = 0; i < kMaxNodes; ++i) {
        fp.x[i] = i < f->n_nodes ? f->x[i] : 0.0;
        fp.w[i] = i < f->n_nodes ? f->w[i] : 0.0;
        fp.cx[i] = std::asinh(fp.x[i]);
    }
    return 0;
}

// The tile kernel covers: diagonal-Gaussian targets, Gaussian family, no in-kernel moment accumulators
// (thinned draws are written by a second instantiation).  Everything else runs on the chain or octet kernel.
// The lane kernel (thread per chain, theta resident in shared memory, closed-form quadratic fit) takes the
// free-running fp64 launches of the same cases whenever at least 4 one-warp CTAs fit per SM (D <= ~115 with two
// stored mean columns); replay, fp32, over-relaxed proposals and larger D stay on the tile kernel.
static bool lane_applies(const StepArgs& a, int dtype, int family, bool replay, bool accum, int flags) {
    return !(flags & (KLHR_FIT_FORCE_OCTET | KLHR_FIT_FORCE_TILE)) && !replay && dtype == KLHR_F64 &&
           family == KLHR_FAMILY_GAUSS && !accum && a.fp.or_K == 0 &&
           (a.mp.id == KLHR_MODEL_NORMAL || a.mp.id == KLHR_MODEL_ILL_NORMAL) &&
           lane_smem_bytes(a) + 1024 <= (size_t)(228 * 1024) / 4;
}

static bool tile_applies(const StepArgs& a, int family, bool accum, int flags) {
    // at most 2 stored direction-mean columns: they live in the tile's shared memory (J = 2 default)
    const int n_stored = a.dir.mean_cols ? a.dir.n_cols - a.dir.n_zero_cols : 0;
    // the warp's x tile (32 x D fp32) must stay small enough for several one-warp CTAs per SM;
    // beyond D ~ 250 the octet kernel (theta resident in shared memory, fewer chains per CTA) takes over
    const bool small = (size_t)kTileChains * pad_dim(a.mp.D, 4) * 4 <= 32 * 1024;
    return !(flags & KLHR_FIT_FORCE_OCTET) && family == KLHR_FAMILY_GAUSS && !accum && small &&
           (a.mp.id == KLHR_MODEL_NORMAL || a.mp.id == KLHR_MODEL_ILL_NORMAL) && n_stored <= 2;
}

// The chain kernel (thread-per-chain fit, model-generic line setup) covers every target and both
// families as long as its rho tile fits a modest shared-memory budget; like the tile kernel it
// has no in-kernel accumulators (thinned draws are written by a second instantiation).
static bool chain_applies(const StepArgs& a, int dtype, bool replay, bool accum, int flags) {
    return !(flags & KLHR_FIT_FORCE_OCTET) && !accum &&
           chain_smem_bytes(a, dtype == KLHR_F64 ? 8 : 4, replay) <= 20 * 1024;   // larger D: the octet kernel keeps theta resident
}

static int dispatch_step(const StepArgs& a, int dtype, int family, bool replay, bool accum, cudaStream_t st,
                         LaunchInfo* info, int flags) {
    if (lane_applies(a, dtype, family, replay, accum, flags)) return launch_lane(a, st, info);
    if (densek_applies(a, dtype, family, replay, accum, flags)) return launch_densek(a, replay, st, info);
    if (tile_applies(a, family, accum, flags)) return launch_tile(a, dtype, replay, st, info);
    if (chain_applies(a, dtype, replay, accum, flags)) return launchers(a.mp).chain(&a, dtype, family, replay, st, info);
    return launchers(a.mp).step(&a, dtype, family, replay, accum, st, info);
}

// ------------------------------------------------------------------ pooled outer products
// outer[i][j] += sum_c (theta_ci - shift_i)(theta_cj - shift_j): a tall-skinny SYRK on the FP64 tensor cores.
// Each CTA owns a 32x32 tile of the output (upper triangle only) and a slice of the chains.  32 chains at a
// time are staged in shared memory (shift subtracted, promoted to fp64); the tile is 4x4 m8n8 fragments: warp w
// accumulates row fragment w / 2 against column fragments 2 (w % 2) and 2 (w % 2) + 1 with mma.sync.m8n8k4.f64,
// three 64-bit shared loads per two DMMAs (row pitch 36 doubles: conflict-free fragment reads).
template <typename R>
__global__ void __launch_bounds__(256) outer_kernel(const R* __restrict__ theta, const R* __restrict__ shift,
                                                    double* __restrict__ outer, double* __restrict__ s1,
                                                    long long B, int D, int chains_per_cta,
                                                    double* __restrict__ scratch) {
    constexpr int kPitch = 36;
    __shared__ double ta[32][kPitch], tb[32][kPitch];
    const int ti = blockIdx.x * 32, tj = blockIdx.y * 32;
    if (tj < ti) return;                                 // upper triangle only; mirrored below
    const long long c_begin = (long long)blockIdx.z * chains_per_cta;
    const long long c_end = c_begin + chains_per_cta < B ? c_begin + chains_per_cta : B;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // 32 lanes x 8 warps
    const int r8 = tx >> 2, k4 = tx & 3;                         // fragment coordinates
    const int fm = ty >> 1, fn = 2 * (ty & 1);                   // row fragment, first of two column fragments
    double acc[2][2] = {{0, 0}, {0, 0}};
    double colsum = 0;
    const double sa = (shift && ti + tx < D) ? (double)shift[ti + tx] : 0.0;
    const double sb = (shift && tj + tx < D) ? (double)shift[tj + tx] : 0.0;
    for (long long c0 = c_begin; c0 < c_end; c0 += 32) {
        // stage 32 chains x 32 dims of both tiles (rows of absent chains / dims are zero)
        for (int r = ty; r < 32; r += 8) {
            const long long c = c0 + r;
            const int ia = ti + tx, ib = tj + tx;
            double va = 0, vb = 0;
            if (c < c_end) {
                if (ia < D) va = (double)theta[c * D + ia] - sa;
                if (ib < D) vb = (double)theta[c * D + ib] - sb;
            }
            ta[r][tx] = va;
            tb[r][tx] = vb;
        }
        __syncthreads();
#pragma unroll
        for (int k0 = 0; k0 < 32; k0 += 4) {
            const double a = ta[k0 + k4][8 * fm + r8];           // A[i][k] = ta[k][i]
            const double b0 = tb[k0 + k4][8 * fn + r8];          // B[k][j] = tb[k][j]
            const double b1 = tb[k0 + k4][8 * fn + 8 + r8];
            dmma_m8n8k4(acc[0][0], acc[0][1], a, b0);
            dmma_m8n8k4(acc[1][0], acc[1][1], a, b1);
        }
        if (s1 && blockIdx.y == blockIdx.x && ty == 0)
            for (int k = 0; k < 32; ++k) colsum += ta[k][tx];
        __syncthreads();
    }
    // C fragment: row r8, columns 2 k4 + {0, 1} of fragment (fm, fn + q)
    double* plane = scratch ? scratch + (size_t)blockIdx.z * ((size_t)D * D + D) : nullptr;
#pragma unroll
    for (int q = 0; q < 2; ++q)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int i = ti + 8 * fm + r8, j = tj + 8 * (fn + q) + 2 * k4 + e;
            if (i < D && j < D) {
                if (plane) {
                    // deterministic mode: every chain slice ADDS its partial tile to its own scratch plane
                    // [slice][D*D + D] (one owner thread per entry); klhr_outer_reduce folds the planes with a
                    // canonical tree at the window closure
                    plane[(size_t)i * D + j] += acc[q][e];
                    if (ti != tj) plane[(size_t)j * D + i] += acc[q][e];
                } else {
                    atomicAdd(outer + (size_t)i * D + j, acc[q][e]);
                    if (ti != tj) atomicAdd(outer + (size_t)j * D + i, acc[q][e]);
                }
            }
        }
    if (blockIdx.y == blockIdx.x && ty == 0 && ti + tx < D) {
        if (plane) plane[(size_t)D * D + ti + tx] += colsum;
        else if (s1) atomicAdd(s1 + ti + tx, colsum);
    }
}

// Adds the per-slice planes with a CANONICAL pairwise tree over the slice index (slice = 1024 consecutive chains):
// (((p0 + p1) + (p2 + p3)) + ...).  The tree of an aligned power-of-two run of slices is a subtree of the tree
// of the whole range, so ranks that own such runs and combine their results pairwise in rank order
// (adaptation.allreduce_adaptation) reproduce the single-process sum BIT FOR BIT.
__global__ void outer_reduce_kernel(double* __restrict__ scratch, double* __restrict__ outer,
                                    double* __restrict__ s1, int D, int slices) {
    const size_t plane = (size_t)D * D + D;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= plane) return;
    double stack[32];                       // stack[k]: sum of a complete aligned run of 2^k slices
    int n = 0;                              // slices consumed; bit k of n <=> stack[k] is occupied
    for (int s = 0; s < slices; ++s) {
        double v = scratch[(size_t)s * plane + idx];
        scratch[(size_t)s * plane + idx] = 0.0;          // ready for the next window
        int k = 0;
        while ((n >> k) & 1) { v = stack[k] + v; ++k; }
        stack[k] = v;
        ++n;
    }
    double t = 0;
    bool have = false;
    for (int k = 0; k < 32; ++k)            // ragged tail: fold the remaining runs from the smallest up
        if ((n >> k) & 1) { t = have ? stack[k] + t : stack[k]; have = true; }
    if (idx < (size_t)D * D) outer[idx] += t;
    else if (s1) s1[idx - (size_t)D * D] += t;
}

}  // namespace klhr

using namespace klhr;

extern "C" {

int klhr_abi_version(void) { return KLHR_ABI_VERSION; }

int klhr_user_register(const klhr_user_table_t* t) {
    if (!t) return fail(-1, "klhr_user_register: table is NULL");
    if (t->abi_version != KLHR_ABI_VERSION)
        return fail(-17, "klhr_user_register: the user library was built for another ABI version");
    if (t->sizeof_step_args != (int32_t)sizeof(StepArgs) || t->sizeof_slice_args != (int32_t)sizeof(SliceArgs) ||
        t->sizeof_mh_args != (int32_t)sizeof(MhArgs) || t->sizeof_kl_args != (int32_t)sizeof(KlArgs) ||
        t->sizeof_model_params != (int32_t)sizeof(ModelParams))
        return fail(-17, "klhr_user_register: argument struct layout mismatch (the user library was built against other headers)");
    if (!t->step || !t->chain || !t->eval || !t->kl || !t->mh || !t->slice)
        return fail(-1, "klhr_user_register: a launcher of the table is NULL");
    std::lock_guard<std::mutex> lock(g_user_mutex);
    const int n = g_user_count.load(std::memory_order_relaxed);
    for (int k = 0; k < n; ++k)
        if (std::memcmp(&g_user[k], t, sizeof(*t)) == 0) return k;
    if (n == kUserSlots) return fail(-18, "klhr_user_register: registry full (64 user targets per process)");
    g_user[n] = *t;
    g_user_count.store(n + 1, std::memory_order_release);
    return n;
}

size_t klhr_last_error(char* buf, size_t len) {
    if (!buf || len == 0) return g_last_error.size();
    const size_t n = g_last_error.size() < len - 1 ? g_last_error.size() : len - 1;
    std::memcpy(buf, g_last_error.data(), n);
    buf[n] = 0;
    return n;
}

int klhr_model_eval(const klhr_model_t* model, int dtype, const void* theta_dev, void* lp_dev, void* grad_dev,
                    int64_t n_chains, void* stream) {
    ModelParams mp;
    if (int e = check_model(model, mp)) return e;
    if (dtype != KLHR_F64 && dtype != KLHR_F32) return fail(-9, "dtype must be KLHR_F64 or KLHR_F32");
    if (n_chains < 0) return fail(-10, "n_chains must be non-negative");
    if (n_chains == 0) return 0;
    if (!theta_dev || !lp_dev) return fail(-1, "theta and lp must not be NULL");
    return cuda_fail(launchers(mp).eval(&mp, dtype, theta_dev, lp_dev, grad_dev, n_chains, stream), "klhr_model_eval");
}

int klhr_step_replay(const klhr_model_t* model, const klhr_fit_t* fit, int dtype, void* theta_dev,
                     const void* rho_dev, const void* z_init_dev, const void* init4_dev, const void* z_prop_dev,
                     const void* u_dev, const klhr_trace_t* trace, int64_t n_chains, void* stream) {
    StepArgs a;
    std::memset(&a, 0, sizeof(a));
    if (int e = check_model(model, a.mp)) return e;
    if (int e = check_fit(fit, a.fp)) return e;
    if (dtype != KLHR_F64 && dtype != KLHR_F32) return fail(-9, "dtype must be KLHR_F64 or KLHR_F32");
    if (n_chains == 0) return 0;
    if (!theta_dev || !rho_dev || !z_init_dev || !z_prop_dev || !u_dev)
        return fail(-1, "theta, rho, z_init, z_prop, u must not be NULL");
    if (fit->family == KLHR_FAMILY_SINH && !init4_dev) return fail(-1, "sinh family needs init4");
    if (n_chains < 0) return fail(-10, "n_chains must be non-negative");
    a.theta = theta_dev; a.B = n_chains;
    a.rho = rho_dev; a.z_init = z_init_dev; a.init4 = init4_dev; a.z_prop = z_prop_dev; a.u = u_dev;
    a.n_steps = 1;
    a.acc.thin = 1;
    if (trace) a.tr = *trace;
    a.tr.z_init = a.tr.z_prop = a.tr.u = a.tr.init4 = nullptr;   // inputs in this mode
    if (fit->overrelax_K > 0 && (!a.tr.or_r || !a.tr.or_v))
        return fail(-1, "over-relaxed replay needs trace.or_r and trace.or_v as inputs");
    return cuda_fail(dispatch_step(a, dtype, fit->family, true, false, (cudaStream_t)stream, nullptr, fit->flags),
                     "klhr_step_replay");
}

static int fill_run(StepArgs& a, const klhr_model_t* model, const klhr_fit_t* fit, const klhr_direction_t* dir,
                    int dtype, int64_t n_chains, const klhr_accum_t* accum, const klhr_trace_t* trace, bool& use_acc) {
    std::memset(&a, 0, sizeof(a));
    if (int e = check_model(model, a.mp)) return e;
    if (int e = check_fit(fit, a.fp)) return e;
    if (dtype != KLHR_F64 && dtype != KLHR_F32) return fail(-9, "dtype must be KLHR_F64 or KLHR_F32");
    if (n_chains < 0) return fail(-10, "n_chains must be non-negative");
    if (dir) {
        a.dir = *dir;
        if (a.dir.mean_cols && a.dir.n_cols < 1) return fail(-11, "direction: n_cols must be >= 1 with mean_cols");
        if (a.dir.n_zero_cols < 0 || a.dir.n_zero_cols > 1 || (a.dir.mean_cols && a.dir.n_zero_cols >= a.dir.n_cols))
            return fail(-11, "direction: n_zero_cols must be 0 or 1 and smaller than n_cols");
        if (a.dir.mean_cols && a.dir.n_cols > 1 && !a.dir.cdf) return fail(-11, "direction: cdf needed when n_cols > 1");
        if (!a.dir.mean_cols) a.dir.n_cols = 0;
    }
    a.acc.thin = 1;
    use_acc = false;
    if (accum) {
        a.acc = *accum;
        if (a.acc.thin < 1) a.acc.thin = 1;
        if ((a.acc.pooled_s1 == nullptr) != (a.acc.pooled_s2 == nullptr))
            return fail(-12, "pooled_s1 and pooled_s2 must be given together");
        use_acc = a.acc.pooled_s1 || a.acc.chain_s1 || a.acc.chain_s2;
    }
    if (trace) {
        a.tr = *trace;
        if (a.tr.z_init && (!a.tr.z_prop || !a.tr.u)) return fail(-13, "trace: z_init, z_prop, u go together");
    }
    a.B = n_chains;
    return 0;
}

int klhr_run(const klhr_model_t* model, const klhr_fit_t* fit, const klhr_direction_t* dir, int dtype,
             void* theta_dev, int64_t n_chains, int64_t chain_offset, int64_t draw_offset, int32_t n_steps,
             uint64_t seed, const klhr_accum_t* accum, const klhr_trace_t* trace, void* stream) {
    StepArgs a;
    bool use_acc;
    if (int e = fill_run(a, model, fit, dir, dtype, n_chains, accum, trace, use_acc)) return e;
    if (n_steps < 0 || chain_offset < 0 || draw_offset < 0) return fail(-10, "negative count or offset");
    if (n_steps == 0 || n_chains == 0) return 0;
    if (!theta_dev) return fail(-1, "theta must not be NULL");
    a.theta = theta_dev;
    a.chain_offset = chain_offset; a.draw_offset = draw_offset; a.n_steps = n_steps; a.seed = seed;
    return cuda_fail(dispatch_step(a, dtype, fit->family, false, use_acc, (cudaStream_t)stream, nullptr, fit->flags),
                     "klhr_run");
}

int klhr_mh_run(const klhr_model_t* model, int dtype, void* theta_dev, double stepsize, int64_t n_chains,
                int64_t chain_offset, int64_t draw_offset, int32_t n_steps, uint64_t seed, const klhr_accum_t* accum,
                const klhr_trace_t* trace, void* stream) {
    MhArgs a;
    std::memset(&a, 0, sizeof(a));
    if (int e = check_model(model, a.mp)) return e;
    if (dtype != KLHR_F64 && dtype != KLHR_F32) return fail(-9, "dtype must be KLHR_F64 or KLHR_F32");
    if (n_chains < 0 || n_steps < 0 || chain_offset < 0 || draw_offset < 0) return fail(-10, "negative count or offset");
    if (!(stepsize > 0)) return fail(-14, "stepsize must be positive");
    a.acc.thin = 1;
    if (accum) {
        a.acc = *accum;
        if (a.acc.thin < 1) a.acc.thin = 1;
        if (a.acc.pooled_s1 || a.acc.pooled_s2) return fail(-12, "klhr_mh_run: pooled in-kernel moments are not supported");
        if (a.acc.chain_s2 && !a.acc.chain_s1) return fail(-12, "chain_s2 needs chain_s1");
    }
    if (trace) a.tr = *trace;
    if (n_chains == 0 || n_steps == 0) return 0;
    if (!theta_dev) return fail(-1, "theta must not be NULL");
    a.theta = theta_dev; a.B = n_chains; a.stepsize = stepsize;
    a.chain_offset = chain_offset; a.draw_offset = draw_offset; a.n_steps = n_steps; a.seed = seed;
    return cuda_fail(launchers(a.mp).mh(&a, dtype, stream), "klhr_mh_run");
}

static int check_slice(const klhr_slice_t* sp) {
    if (!sp) return fail(-1, "slice must not be NULL");
    if (!(sp->w > 0) || !std::isfinite(sp->w)) return fail(-15, "slice: w must be positive and finite");
    if (!(sp->lower <= 0.0) || !(sp->upper >= 0.0)) return fail(-15, "slice: need lower <= 0 <= upper (the current point is line coordinate 0)");
    if (!(sp->tol >= 0)) return fail(-15, "slice: tol must be non-negative");
    if (sp->cap < 1) return fail(-15, "slice: cap must be >= 1");
    return 0;
}

int klhr_slice_run(const klhr_model_t* model, const klhr_slice_t* slice, const klhr_direction_t* dir, int dtype,
                   void* theta_dev, int64_t n_chains, int64_t chain_offset, int64_t draw_offset, int32_t n_steps,
                   uint64_t seed, const klhr_accum_t* accum, const klhr_trace_t* trace, void* stream) {
    SliceArgs a;
    std::memset(&a, 0, sizeof(a));
    if (int e = check_model(model, a.mp)) return e;
    if (int e = check_slice(slice)) return e;
    if (dtype != KLHR_F64 && dtype != KLHR_F32) return fail(-9, "dtype must be KLHR_F64 or KLHR_F32");
    if (n_chains < 0 || n_steps < 0 || chain_offset < 0 || draw_offset < 0) return fail(-10, "negative count or offset");
    if (dir) {
        a.dir = *dir;
        if (a.dir.mean_cols && a.dir.n_cols < 1) return fail(-11, "direction: n_cols must be >= 1 with mean_cols");
        if (a.dir.n_zero_cols < 0 || a.dir.n_zero_cols > 1 || (a.dir.mean_cols && a.dir.n_zero_cols >= a.dir.n_cols))
            return fail(-11, "direction: n_zero_cols must be 0 or 1 and smaller than n_cols");
        if (a.dir.mean_cols && a.dir.n_cols > 1 && !a.dir.cdf) return fail(-11, "direction: cdf needed when n_cols > 1");
        if (!a.dir.mean_cols) a.dir.n_cols = 0;
    }
    a.acc.thin = 1;
    if (accum) {
        a.acc = *accum;
        if (a.acc.thin < 1) a.acc.thin = 1;
        if (a.acc.pooled_s1 || a.acc.pooled_s2) return fail(-12, "klhr_slice_run: pooled in-kernel moments are not supported");
        if (a.acc.chain_s2 && !a.acc.chain_s1) return fail(-12, "chain_s2 needs chain_s1");
    }
    if (trace) a.tr = *trace;
    if (n_chains == 0 || n_steps == 0) return 0;
    if (!theta_dev) return fail(-1, "theta must not be NULL");
    a.sp = *slice; a.tol = slice->tol;
    a.theta = theta_dev; a.B = n_chains;
    a.chain_offset = chain_offset; a.draw_offset = draw_offset; a.n_steps = n_steps; a.seed = seed;
    return cuda_fail(launchers(a.mp).slice(&a, dtype, false, stream), "klhr_slice_run");
}

int klhr_slice_replay(const klhr_model_t* model, const klhr_slice_t* slice, int dtype, void* theta_dev,
                      const void* rho_dev, const void* e_dev, const void* u0_dev, const void* shrink_u_dev,
                      const klhr_trace_t* trace, int64_t n_chains, void* stream) {
    SliceArgs a;
    std::memset(&a, 0, sizeof(a));
    if (int e = check_model(model, a.mp)) return e;
    if (int e = check_slice(slice)) return e;
    if (dtype != KLHR_F64 && dtype != KLHR_F32) return fail(-9, "dtype must be KLHR_F64 or KLHR_F32");
    if (n_chains < 0) return fail(-10, "n_chains must be non-negative");
    if (n_chains == 0) return 0;
    if (!theta_dev || !rho_dev || !e_dev || !u0_dev || !shrink_u_dev)
        return fail(-1, "theta, rho, e, u0, shrink_u must not be NULL");
    a.sp = *slice; a.tol = slice->tol;
    a.theta = theta_dev; a.B = n_chains;
    a.rho = rho_dev; a.e = e_dev; a.u0 = u0_dev; a.shrink_u = shrink_u_dev;
    a.n_steps = 1;
    a.acc.thin = 1;
    if (trace) a.tr = *trace;
    a.tr.slice_u = nullptr;                                       // input in this mode
    return cuda_fail(launchers(a.mp).slice(&a, dtype, true, stream), "klhr_slice_replay");
}

int klhr_kl_eval(const klhr_model_t* model, const klhr_fit_t* fit, int dtype, const void* theta_dev,
                 const void* rho_dev, const void* eta_dev, void* f_dev, void* grad_dev, void* hess_dev,
                 int64_t n_chains, void* stream) {
    KlArgs a;
    std::memset(&a, 0, sizeof(a));
    if (int e = check_model(model, a.mp)) return e;
    if (int e = check_fit(fit, a.fp)) return e;
    if (dtype != KLHR_F64 && dtype != KLHR_F32) return fail(-9, "dtype must be KLHR_F64 or KLHR_F32");
    if (n_chains < 0) return fail(-10, "n_chains must be non-negative");
    if (n_chains == 0) return 0;
    if (!theta_dev || !rho_dev || !eta_dev || !f_dev || !grad_dev)
        return fail(-1, "theta, rho, eta, f, grad must not be NULL");
    a.theta = theta_dev; a.rho = rho_dev; a.eta = eta_dev; a.f = f_dev; a.grad = grad_dev; a.hess = hess_dev;
    a.B = n_chains;
    return cuda_fail(launchers(a.mp).kl(&a, dtype, fit->family, stream), "klhr_kl_eval");
}

// ---- elementwise fp64 exp / log of the fit's inner loops (klhr_math.cuh), exposed for the accuracy tests
__global__ void math_kernel(int op, const double* __restrict__ x, double* __restrict__ y, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = op == 0 ? r_exp(x[i]) : r_log(x[i]);
}

int klhr_math_eval(int op, const double* x_dev, double* y_dev, int64_t n, void* stream) {
    if (op != 0 && op != 1) return fail(-16, "klhr_math_eval: op must be 0 (exp) or 1 (log)");
    if (n < 0) return fail(-10, "n must be non-negative");
    if (n == 0) return 0;
    if (!x_dev || !y_dev) return fail(-1, "x and y must not be NULL");
    math_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(op, x_dev, y_dev, n);
    return cuda_fail((int)cudaGetLastError(), "klhr_math_eval");
}

int klhr_launch_info(const klhr_model_t* model, const klhr_fit_t* fit, int dtype, int free_running, int accumulate,
                     int32_t* threads_per_cta, int32_t* smem_bytes, int32_t* regs) {
    StepArgs a;
    std::memset(&a, 0, sizeof(a));
    if (int e = check_model(model, a.mp)) return e;
    if (int e = check_fit(fit, a.fp)) return e;
    if (dtype != KLHR_F64 && dtype != KLHR_F32) return fail(-9, "dtype must be KLHR_F64 or KLHR_F32");
    a.acc.thin = 1;
    LaunchInfo li;
    const int e = dispatch_step(a, dtype, fit->family, !free_running, accumulate != 0, nullptr, &li, fit->flags);
    if (e) return cuda_fail(e, "klhr_launch_info") > 0 ? -30 : e;
    if (threads_per_cta) *threads_per_cta = li.threads;
    if (smem_bytes) *smem_bytes = li.smem;
    if (regs) *regs = li.regs;
    return li.ctas_per_sm;
}

// chain slices of the SYRK: 1024 consecutive chains each, whatever the batch size -- the canonical blocks of the
// bit-reproducible, sharding-invariant reduction (outer_reduce_kernel)
static void outer_slicing(int64_t n_chains, int32_t dim, int& tiles, long long& slices, long long& per) {
    tiles = (dim + 31) / 32;
    per = 1024;
    slices = (n_chains + per - 1) / per;
    if (slices < 1) slices = 1;
}

int64_t klhr_corr_pack_cholesky(const double* L_host, int32_t dim, double* out_host) {
    if (dim != 128 && dim != 256) {
        fail(-3, "klhr_corr_pack_cholesky: the tensor-core kernels take dim = 128 or 256");
        return -3;
    }
    const int T = dim / 8;
    if (out_host) {
        if (!L_host) {
            fail(-1, "klhr_corr_pack_cholesky: L_host is NULL");
            return -1;
        }
        for (int nt = 0; nt < T; ++nt) {
            double* o = out_host + dk_pack_offset(nt, T);
            for (int p = nt; p < T; ++p)
                for (int lane = 0; lane < 32; ++lane) {
                    const int r8 = lane >> 2, k4 = lane & 3;
                    *o++ = L_host[(size_t)(8 * p + k4) * dim + 8 * nt + r8];
                    *o++ = L_host[(size_t)(8 * p + 4 + k4) * dim + 8 * nt + r8];
                }
        }
    }
    return (int64_t)dk_pack_doubles(dim);
}

int64_t klhr_outer_scratch_doubles(int64_t n_chains, int32_t dim) {
    if (n_chains <= 0 || dim <= 0) return 0;
    int tiles;
    long long slices, per;
    outer_slicing(n_chains, dim, tiles, slices, per);
    return (int64_t)slices * ((int64_t)dim * dim + dim);
}

int klhr_outer_accumulate(int dtype, const void* theta_dev, const void* shift_dev, double* outer_dev, double* s1_dev,
                          int64_t n_chains, int32_t dim, double* scratch_dev, int64_t scratch_doubles, void* stream) {
    if (dtype != KLHR_F64 && dtype != KLHR_F32) return fail(-9, "dtype must be KLHR_F64 or KLHR_F32");
    if (!theta_dev || !outer_dev) return fail(-1, "theta and outer must not be NULL");
    if (n_chains < 0 || dim <= 0) return fail(-10, "bad sizes");
    if (n_chains == 0) return 0;
    int tiles;
    long long slices, per;
    outer_slicing(n_chains, dim, tiles, slices, per);
    if (scratch_dev && scratch_doubles < (int64_t)slices * ((int64_t)dim * dim + dim))
        return fail(-15, "scratch too small: see klhr_outer_scratch_doubles");
    dim3 grid(tiles, tiles, (unsigned)slices);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == KLHR_F64)
        outer_kernel<double><<<grid, 256, 0, st>>>((const double*)theta_dev, (const double*)shift_dev, outer_dev,
                                                   s1_dev, n_chains, dim, (int)per, scratch_dev);
    else
        outer_kernel<float><<<grid, 256, 0, st>>>((const float*)theta_dev, (const float*)shift_dev, outer_dev,
                                                  s1_dev, n_chains, dim, (int)per, scratch_dev);
    return cuda_fail((int)cudaGetLastError(), "klhr_outer_accumulate");
}

int klhr_outer_reduce(double* scratch_dev, int64_t scratch_doubles, double* outer_dev, double* s1_dev,
                      int64_t n_chains, int32_t dim, void* stream) {
    if (!scratch_dev || !outer_dev) return fail(-1, "scratch and outer must not be NULL");
    if (n_chains <= 0 || dim <= 0) return fail(-10, "bad sizes");
    int tiles;
    long long slices, per;
    outer_slicing(n_chains, dim, tiles, slices, per);
    const size_t plane = (size_t)dim * dim + dim;
    if (scratch_doubles < (int64_t)(slices * (long long)plane)) return fail(-15, "scratch too small: see klhr_outer_scratch_doubles");
    outer_reduce_kernel<<<(unsigned)((plane + 255) / 256), 256, 0, (cudaStream_t)stream>>>(scratch_dev, outer_dev, s1_dev, dim,
                                                                                         (int)slices);
    return cuda_fail((int)cudaGetLastError(), "klhr_outer_reduce");
}

}  // extern "C"
