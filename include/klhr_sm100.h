/* libklhr_sm100.so -- C ABI of the B200-native KL Hit-and-Run step.
 *
 * This is the drop-in boundary for the reference's hot path.  The reference reaches native
 * code through BridgeStan's C ABI, once per log-density evaluation (reference
 * bsmodel.py:18,27 -> bridgestan ctypes -> bs_log_density[_gradient]); here one call
 * advances EVERY chain by whole draws.  Each entry point names the reference interface it
 * replaces.  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - every pointer inside the descriptor structs and every `*_dev` argument is a DEVICE
 *     pointer (torch `tensor.data_ptr()`); the library never allocates persistent state;
 *   - `dtype` selects the arithmetic type of all real buffers: KLHR_F64 or KLHR_F32;
 *   - calls are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default);
 *   - return value: 0 ok, <0 invalid argument (see klhr_last_error), >0 a cudaError_t;
 *   - no exceptions cross the ABI; the last-error string is thread-local.
 */
#ifndef KLHR_SM100_H_
#define KLHR_SM100_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KLHR_ABI_VERSION 4

enum { KLHR_F64 = 0, KLHR_F32 = 1 };
enum { KLHR_FAMILY_GAUSS = 0, KLHR_FAMILY_SINH = 1 };

/* Stan programs of the reference with a hand-written device implementation
 * (reference stan/<name>.stan; SURVEY.md section 8a rows M1-M7). */
enum {
    KLHR_MODEL_NORMAL = 0,      /* stan/normal.stan       */
    KLHR_MODEL_ILL_NORMAL = 1,  /* stan/ill-normal.stan   data0 = inv_s2[D]                       */
    KLHR_MODEL_FUNNEL = 2,      /* stan/funnel.stan       i0 = D (number of alpha); dim = D + 1   */
    KLHR_MODEL_CORR_NORMAL = 3, /* stan/corr-normal.stan  data0 = dense precision P[D*D]; data1 (optional, fp64) =
                                   the lower Cholesky factor of P packed by klhr_corr_pack_cholesky: enables
                                   the triangular tensor-core kernels for D = 128 / 256                    */
    KLHR_MODEL_AR1 = 4,         /* stan/ar1.stan          s0 = alpha, s1 = 1/beta^2               */
    KLHR_MODEL_ARK = 5,         /* stan/arK.stan          i0 = K, i1 = T-K, data0 = [G|c|yy]      */
    KLHR_MODEL_ROSENBROCK = 6,  /* stan/rosenbrock.stan   i0 = D; dim = 2 D                       */
    KLHR_MODEL_EARNINGS = 7,    /* stan/earnings.stan     data0 = [N, Se, Sh, See, Seh, Shh]; dim = 4 */
    KLHR_MODEL_EIGHT_SCHOOLS_NC = 8, /* posteriordb eight_schools_noncentered  i0 = J, data0 = [y_1..J | w_1..J],
                                        w = 1/sigma^2; dim = J + 2, order [theta_trans, mu, log tau] */
    KLHR_MODEL_EIGHT_SCHOOLS_C = 9,  /* posteriordb eight_schools_centered     i0 = J, data0 = [y_1..J | w_1..J],
                                        w = 1/sigma^2; dim = J + 2, order [mu, log tau, theta]       */
    KLHR_MODEL_LOGISTIC_REGRESSION = 10, /* logistic regression  i0 = N >= 0, i1 = K >= 1, data0 = [X (N x (K+1),
                                            row-major, first column 1) | y_1..N in {0, 1}]; dim = K + 1, order [alpha, beta] */
    KLHR_MODEL_COUNT = 11
};

/* Target density descriptor (replaces a bridgestan.StanModel handle, bsmodel.py:10-13). */
typedef struct klhr_model {
    int32_t id;          /* KLHR_MODEL_*                               */
    int32_t dim;         /* number of unconstrained parameters         */
    int32_t i0, i1;      /* model integers, see enum                   */
    double s0, s1;       /* model scalars, see enum                    */
    const void* data0;   /* device buffer, see enum: `dtype` reals, except the sufficient statistics
                            of arK and earnings which are ALWAYS fp64   */
    const void* data1;   /* second device buffer, see enum (NULL if unused) */
} klhr_model_t;

#define KLHR_MAX_NODES 32
/* klhr_fit_t.flags: run the general octet-per-chain kernel even where the faster thread-per-chain
 * kernels (tile kernel: diagonal-Gaussian targets with the Gaussian family; chain kernel: every
 * other case whose rho tile fits in shared memory) apply -- the parity tests cover both paths */
#define KLHR_FIT_FORCE_OCTET 1
/* run the tile kernel (theta streamed through L2, octet-cooperative sweep) where the lane kernel (thread per
 * chain, theta resident in shared memory) would be chosen -- the parity tests cover both */
#define KLHR_FIT_FORCE_TILE 4
/* sinh family with the tail-weight parameter frozen at d = 1: the 3-parameter variant of reference
 * sub_klhr_sinh.py (SUBKLHRSINH); eta is still reported as (m, log s, 0, e) */
#define KLHR_FIT_FIX_D 2

/* Line-fit configuration: the reference's constructor arguments that reach the fit
 * (klhr.py:16-49 / klhr_sinh.py:15-47) plus the fixed iteration budget that replaces
 * scipy.optimize.minimize (klhr.py:127-139). */
typedef struct klhr_fit {
    int32_t family;              /* KLHR_FAMILY_*                                          */
    int32_t n_nodes;             /* N, Gauss-Hermite nodes (<= KLHR_MAX_NODES)            */
    int32_t n1, n2, nb;          /* stage-1 iterations, stage-2 Newton steps, halvings    */
    int32_t flags;               /* KLHR_FIT_* bits                                        */
    int32_t kmax;                /* cap on stage-2 KL evaluations per fit (<= 0: 1 + n2*nb) */
    int32_t overrelax_K;         /* 0: z' = T(z) proposal (klhr.py:180); K > 0: over-relaxed proposal with
                                    K trials (klhr.py:160-173, klhr_sinh.py:215-228), K <= 50  */
    double initscale;            /* klhr.py:24                                            */
    double tol;                  /* klhr.py:28 / klhr_sinh.py:26                          */
    double scale_clip;           /* klhr.py:30 / klhr_sinh.py:28                          */
    double gtol1, gtol2;         /* convergence thresholds of the two stages: |l'|/sqrt(-l'') of the 1-D mode
                                    search (1e-4: it only supplies the start of stage 2) and the inf-norm of the
                                    scaled KL gradient (1e-10)                                              */
    double step_cap, c1, basin;  /* Newton step cap, Armijo constant, full-step basin     */
    double grad_clip;            /* sinh family: elementwise clip of the model gradient inside KL -- the reference's
                                    KLHRSINH clips at its scale_clip (klhr_sinh.py:158-161), SUBKLHRSINH at its
                                    grad_clip (sub_klhr_sinh.py:152-154); applied for dim <= 16; 0 = no clip    */
    double x[KLHR_MAX_NODES];    /* nodes  hermgauss(N).x * sqrt(2)   (klhr.py:46-48)      */
    double w[KLHR_MAX_NODES];    /* weights hermgauss(N).w / sqrt(pi) (klhr.py:49)         */
} klhr_fit_t;

/* Direction law of the step (KLHR._random_direction, klhr.py:143-153):
 * rho = x / ||x + tol||, x ~ N(mean_j, diag(sd^2)), column j drawn with cumulative
 * probabilities cdf[0..n_cols-1] (eigen_method_one) or n_cols == 1 (method two: the host
 * pre-combines the eigenvectors).  A NULL `mean_cols` means a zero mean. */
typedef struct klhr_direction {
    const void* mean_cols;       /* [n_cols - n_zero_cols][D] reals or NULL                */
    const void* sd;              /* [D] reals, sqrt(_cov); NULL = ones                     */
    const void* cdf;             /* [n_cols] reals, last entry 1; NULL when n_cols <= 1    */
    int32_t n_cols;              /* number of candidate mean columns                       */
    int32_t n_zero_cols;         /* trailing columns that are identically zero and NOT stored
                                    in mean_cols: the "isotropic" extra column of
                                    eigen_method_one (klhr.py:64-66) -> 1, else 0           */
} klhr_direction_t;

/* Per-draw trace buffers, all optional (NULL = not written).  Layout [step][chain][..]. */
typedef struct klhr_trace {
    void* eta;        /* [S][B][2|4]  fitted line parameters (KLHR.fit return value)      */
    void* zp;         /* [S][B]       proposal along the line                              */
    void* r;          /* [S][B]       log MH ratio (klhr.py:183-186)                       */
    int32_t* accept;  /* [S][B]                                                            */
    int32_t* evals;   /* [S][B]       line evaluations (grad_evals increment)              */
    void* rho;        /* [S][B][D]    direction used                                       */
    void* z_init;     /* [S][B]       variates used (free-running mode only)               */
    void* z_prop;     /* [S][B]                                                            */
    void* u;          /* [S][B]                                                            */
    void* init4;      /* [S][B][4]    sinh family only (entries 2,3 used)                  */
    int32_t* or_r;    /* [S][B]       over-relaxation: binomial count r (klhr.py:165)            */
    void* or_v;       /* [S][B]       over-relaxation: beta variate v (klhr.py:168,171; 1 if unused).
                                      Outputs of klhr_run; INPUTS of klhr_step_replay when
                                      overrelax_K > 0                                            */
    void* slice_u;    /* [S][B][cap]  slice sampler: uniforms behind the shrinkage proposals, NaN-padded
                                      (klhr_slice_t.cap columns; output of klhr_slice_run)               */
    int32_t* slice_n; /* [S][B]       slice sampler: shrinkage proposals consumed (cap + 1: ran out)     */
} klhr_trace_t;

/* Slice sampling along a random direction (reference Slice.__init__, slice.py:14-39; only m = inf, the
 * configuration the reference can run: its finite-m branch raises NameError, slice.py:108,124). */
typedef struct klhr_slice {
    double w;         /* slice.py:18  width of the stepping-out interval (> 0)                 */
    double lower;     /* slice.py:20  bounds of the line coordinate (-inf / +inf = none)       */
    double upper;     /* slice.py:21                                                           */
    double tol;       /* slice.py:28  rho = x / ||x + tol||                                    */
    int32_t cap;      /* columns of trace.slice_u / of shrink_u in replay mode (>= 1)          */
    int32_t reserved;
} klhr_slice_t;

/* Accumulators of a free-running launch, all optional. */
typedef struct klhr_accum {
    const void* shift;           /* [D] reals subtracted before accumulation (or NULL)     */
    double* pooled_s1;           /* [D]  += sum over chains and draws of (theta - shift)   */
    double* pooled_s2;           /* [D]  += sum of (theta - shift)^2                       */
    double* chain_s1;            /* [B][D] += per-chain sum of (theta - shift)             */
    double* chain_s2;            /* [B][D] += per-chain sum of squares                     */
    long long* accept_count;     /* [B]  += accepted draws (acceptance_probability)        */
    unsigned long long* evals_total; /* [1] += line evaluations (grad_evals)               */
    void* draws;                 /* [S/thin][B][D] thinned draws (MCMCBase.sample rows)    */
    int32_t thin;                /* write every `thin`-th draw (>= 1)                      */
    int32_t skip_accum_last;     /* 1: the last draw of the launch is a window closure and
                                    is not accumulated (klhr.py:202-221)                   */
    int64_t thin_offset;         /* draws already taken towards `draws` by earlier launches:
                                    draw g = thin_offset + step + 1 is stored in row g/thin - 1
                                    when g % thin == 0, so a sample() may span launches    */
} klhr_accum_t;

int klhr_abi_version(void);

/* Copies the calling thread's last error message (NUL-terminated) into buf. */
size_t klhr_last_error(char* buf, size_t len);

/* Batched BSModel.log_density / log_density_gradient (bsmodel.py:15-30):
 * theta [B][D] -> lp [B], grad [B][D] (grad may be NULL).  Non-finite => lp = -inf,
 * grad = 0, never an error. */
int klhr_model_eval(const klhr_model_t* model, int dtype, const void* theta_dev, void* lp_dev,
                    void* grad_dev, int64_t n_chains, void* stream);

/* One KLHR.draw() / KLHRSINH.draw() for every chain with HOST-INJECTED variates
 * (replay mode): theta [B][D] is advanced in place using rho [B][D], z_init [B],
 * init4 [B][4] (sinh; may be NULL for gauss), z_prop [B], u [B].
 * Replaces klhr.py:196-201 (direction excluded) for B chains at once. */
int klhr_step_replay(const klhr_model_t* model, const klhr_fit_t* fit, int dtype, void* theta_dev,
                     const void* rho_dev, const void* z_init_dev, const void* init4_dev,
                     const void* z_prop_dev, const void* u_dev, const klhr_trace_t* trace,
                     int64_t n_chains, void* stream);

/* n_steps full draws for every chain with the in-kernel Philox4x32-10 streams
 * (free-running mode).  The variates of chain c at draw t depend only on
 * (seed, chain_offset + c, draw_offset + t), so results do not depend on how chains are
 * sharded over GPUs or how draws are split over launches.
 * Replaces the loop MCMCBase.sample (mcmc.py:31-37) -> KLHR.draw (klhr.py:196-223). */
int klhr_run(const klhr_model_t* model, const klhr_fit_t* fit, const klhr_direction_t* dir, int dtype,
             void* theta_dev, int64_t n_chains, int64_t chain_offset, int64_t draw_offset,
             int32_t n_steps, uint64_t seed, const klhr_accum_t* accum, const klhr_trace_t* trace,
             void* stream);

/* Random-walk Metropolis (reference mh.py:7-37, the comparison sampler of experiment_accuracy.py:69) on
 * the same engine: n_steps draws theta' = theta + stepsize N(0, I) per chain with the chain's Philox
 * stream.  accum: accept_count, draws/thin, chain_s1/chain_s2 (+shift) are honoured; pooled_s1/pooled_s2
 * are refused; trace: rho receives xi, plus r, accept, u. */
int klhr_mh_run(const klhr_model_t* model, int dtype, void* theta_dev, double stepsize, int64_t n_chains,
                int64_t chain_offset, int64_t draw_offset, int32_t n_steps, uint64_t seed,
                const klhr_accum_t* accum, const klhr_trace_t* trace, void* stream);

/* Slice sampling along KLHR's adapted directions (reference Slice.draw, slice.py:84-158; an algorithm of
 * experiment_accuracy.py:56-64) for n_steps draws per chain with the chain's Philox stream.  accum:
 * accept_count (+= n_steps: every draw moves), evals_total, draws/thin, chain_s1/chain_s2 (+shift) are
 * honoured; trace: zp receives the accepted line coordinate x1, z_init the exponential e, u the interval
 * uniform, plus evals, rho, slice_u, slice_n. */
int klhr_slice_run(const klhr_model_t* model, const klhr_slice_t* slice, const klhr_direction_t* dir, int dtype,
                   void* theta_dev, int64_t n_chains, int64_t chain_offset, int64_t draw_offset, int32_t n_steps,
                   uint64_t seed, const klhr_accum_t* accum, const klhr_trace_t* trace, void* stream);

/* One Slice._uni_slice (slice.py:84-146) for every chain with HOST-INJECTED direction and variates:
 * rho [B][D], e [B] standard exponentials, u0 [B] uniforms behind rng.uniform(0, w), shrink_u [B][cap]
 * uniforms behind the shrinkage proposals rng.uniform(L, R) (NaN = none left: the chain stays put and
 * reports slice_n = cap + 1).  theta is advanced in place. */
int klhr_slice_replay(const klhr_model_t* model, const klhr_slice_t* slice, int dtype, void* theta_dev,
                      const void* rho_dev, const void* e_dev, const void* u0_dev, const void* shrink_u_dev,
                      const klhr_trace_t* trace, int64_t n_chains, void* stream);

/* The reference's KL(eta, rho) (klhr.py:106-120 / klhr_sinh.py:163-176; the function its self-tests check
 * against a numerical Jacobian, klhr.py:249-259, klhr_sinh.py:339-349) for every chain: theta [B][D], rho
 * [B][D], eta [B][2|4] -> f [B], grad [B][2|4] in the reference's coordinates (m, log s[, log d, e]) and,
 * if hess is not NULL, the Hessian [B][n][n] the Newton iteration uses (l'' of the target, second derivatives
 * of the transport).  With KLHR_FIT_FIX_D the d row and column are those of the frozen parameter (0 / 1). */
int klhr_kl_eval(const klhr_model_t* model, const klhr_fit_t* fit, int dtype, const void* theta_dev,
                 const void* rho_dev, const void* eta_dev, void* f_dev, void* grad_dev, void* hess_dev,
                 int64_t n_chains, void* stream);

/* Test hook: y[i] = exp(x[i]) (op 0) or log(x[i]) (op 1) with the fp64 routines the fit kernels use
 * (csrc/klhr_math.cuh), so their accuracy can be checked against the host math library. */
int klhr_math_eval(int op, const double* x_dev, double* y_dev, int64_t n, void* stream);

/* Pooled second-moment accumulation for the adaptation PCA (replaces the per-sample CCIPCA
 * update onlinepca.py:13-26 with raw sums): outer[D][D] += sum_c (theta_c - shift)(theta_c - shift)^T,
 * s1[D] += sum_c (theta_c - shift).  fp64 accumulators regardless of dtype.
 *   scratch_dev == NULL  the chain slices are combined straight into outer / s1 with fp64 atomics;
 *   scratch_dev != NULL  (klhr_outer_scratch_doubles doubles, zeroed by the caller before the first call of a
 *                        window) every slice of 1024 consecutive chains ADDS into its own plane of the scratch
 *                        buffer and outer / s1 are not touched; klhr_outer_reduce folds the planes at the window
 *                        closure.  Sums are then bit-reproducible and do not depend on how the chains are
 *                        sharded over ranks (aligned power-of-two shards). */
int klhr_outer_accumulate(int dtype, const void* theta_dev, const void* shift_dev, double* outer_dev,
                          double* s1_dev, int64_t n_chains, int32_t dim, double* scratch_dev,
                          int64_t scratch_doubles, void* stream);

/* Doubles of scratch for n_chains x dim: one (dim*dim + dim) plane per slice of 1024 chains. */
int64_t klhr_outer_scratch_doubles(int64_t n_chains, int32_t dim);

/* outer[D][D] += tree-sum of the scratch planes' matrices, s1[D] += tree-sum of their first-moment rows (s1 may be
 * NULL), with the canonical pairwise tree over the slice index; the planes are zeroed for the next window. */
int klhr_outer_reduce(double* scratch_dev, int64_t scratch_doubles, double* outer_dev, double* s1_dev,
                      int64_t n_chains, int32_t dim, void* stream);

/* Occupancy query used by bench.py: threads per CTA and dynamic shared bytes the step
 * kernel would be launched with for this problem; returns resident CTAs per SM (<=0 error). */
int klhr_launch_info(const klhr_model_t* model, const klhr_fit_t* fit, int dtype, int free_running,
                     int accumulate, int32_t* threads_per_cta, int32_t* smem_bytes, int32_t* regs);

/* Host helper for klhr_model_t.data1 of KLHR_MODEL_CORR_NORMAL: packs the lower Cholesky factor L (host, row-major
 * [dim][dim], P = L L') into the order the tensor-core kernels consume it -- for column tile nt = 0 .. dim/8 - 1, for
 * k-pair p = nt .. dim/8 - 1, for lane = 0 .. 31 (r8 = lane / 4, k4 = lane % 4): L[8 p + k4][8 nt + r8] and
 * L[8 p + 4 + k4][8 nt + r8] (the zero part of the triangle is not stored).  Returns the number of doubles of the packed
 * stream (out_host may be NULL to query it), or < 0 unless dim is 128 or 256.  The caller copies the stream to the device. */
int64_t klhr_corr_pack_cholesky(const double* L_host, int32_t dim, double* out_host);

/* Test hook: out[i][0..3] = Philox4x32-10(counter = in[i][0..3], key = in[i][4..5]) with the generator the step
 * kernels use (csrc/klhr_common.cuh), for the Random123 known-answer vectors (tests/test_gpu_philox.py). */
int klhr_philox_eval(const uint32_t* ctr_key_dev, uint32_t* out_dev, int64_t n, void* stream);

/* Peak probes for the roofline denominators (BASELINE.md section 3: the FP64 / FP32 vector peaks are not in
 * MEASURED_PEAKS.json and must be measured with an FMA micro-kernel on the box).  Launches `ctas` CTAs of 256
 * threads running `iters` trips of micro-kernel `kind` (0 fp64 FMA, 1 Philox4x32-10 + fp32 Box-Muller normals --
 * the direction stream of the step --, 2 fp32 FMA, 3 cvt.f64.f32, 4 MUFU, 5 mul.wide.u32, 6 integer-pipe
 * fp32->fp64 promotion, 7 fp64 DMMA m8n8k4) asynchronously on `stream`; the caller times it.  Returns the number of operations the
 * launch issues (thread-level: one FMA = one operation = 2 flop), or < 0 on a bad argument. */
int64_t klhr_peak_probe(int kind, int64_t iters, int ctas, double* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KLHR_SM100_H_ */
