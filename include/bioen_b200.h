/* bioen_b200.h -- C ABI of libbioen_b200.so, the B200 (sm_100a) implementation of BioEn's optimisation
 * hot path.  Plain C: pointers and sizes only, no CUDA or torch types.
 *
 * Part 1 is the drop-in boundary: the exact symbols (names, argument order, struct layouts, error
 * convention) that the reference's Cython layer binds from its OpenMP C kernels, so that
 * bioen/optimize/ext/c_bioen.pyx (extern blocks at lines 10-129) links against this library unchanged.
 * All pointers in part 1 are HOST pointers owned by the caller, exactly as in the reference; the library
 * uploads what it needs, runs on the GPU, and writes results back before returning.
 *
 * Part 2 is the handle API the host-side Python mirror (bioen_b200/optimize) actually uses: yTilde is
 * uploaded once per problem and stays resident in HBM across evaluations, minimiser iterations and a whole
 * theta series.
 *
 * Citations are paths relative to the reference repository root (bio-phys/BioEn v0.1.3).
 */
#ifndef BIOEN_B200_H
#define BIOEN_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------
 * Part 1 -- reference-compatible symbols
 * ------------------------------------------------------------------------------------------------ */

/* bioen/optimize/ext/c_bioen_common.h:44-60 (passed BY VALUE to the _opt_* drivers) */
typedef struct params_t {
    double *forces;
    double *w0;
    double *g;
    double *G;
    double *yTilde;   /* m x n, row-major, C-contiguous float64 */
    double *YTilde;   /* m */
    double *w;        /* n, scratch */
    double *result;   /* n (logw) or m (forces): minimiser end point */
    double theta;
    double *yTildeT;  /* accepted and ignored: the GPU needs no transposed copy */
    int caching;      /* accepted and ignored */
    double *tmp_n;    /* scratch, may be NULL here */
    double *tmp_m;    /* scratch, may be NULL here */
    int m;
    int n;
} params_t;

/* c_bioen_common.h:62-67 */
typedef struct gsl_config_params {
    double step_size;
    double tol;
    int max_iterations;
    int algorithm;    /* 0 conjugate_fr, 1 conjugate_pr, 2 vector_bfgs2, 3 vector_bfgs, 4 steepest_descent */
} gsl_config_params;

/* c_bioen_common.h:69-79 */
typedef struct lbfgs_config_params {
    int linesearch;   /* 0 More-Thuente, 1 Armijo, 2 Wolfe (BioEn default), 3 strong Wolfe */
    int max_iterations;
    double delta;
    double epsilon;
    double ftol;
    double gtol;
    double wolfe;
    int past;
    int max_linesearch;
} lbfgs_config_params;

/* c_bioen_common.h:89-92 */
typedef struct visual_params {
    size_t debug;
    size_t verbose;
} visual_params;

/* replaces c_bioen_kernels_logw.c:55-94 -- w = softmax(g); returns s = sum_j exp(g_j).
 * (The device computes a max-stabilised log-sum-exp; s is reconstructed and overflows to +inf exactly when the
 * reference's un-stabilised sum does.) */
double _get_weights(const double *g, double *w, size_t n);

/* replaces c_bioen_kernels_logw.c:131-147 -- log-weights objective.  `w` and `weights_sum` are recomputed on
 * the device from g (every reference call site passes w = softmax(g)); `gradient`, `caching`, `yTildeT`,
 * `tmp_n`, `tmp_m` are unused as in the reference. */
double _bioen_log_posterior_logw(const double *g, const double *G, const double *yTilde, const double *YTilde,
                                 const double *w, const double *gradient, double theta, int caching,
                                 const double *yTildeT, double *tmp_n, double *tmp_m, int m, int n,
                                 double weights_sum);

/* replaces c_bioen_kernels_logw.c:151-268 -- log-weights gradient, written to gradient[n] */
void _grad_bioen_log_posterior_logw(const double *g, const double *G, const double *yTilde, const double *YTilde,
                                    const double *w, double *gradient, double theta, int caching,
                                    const double *yTildeT, double *tmp_n, double *tmp_m, int m, int n,
                                    double weights_sum);

/* replaces c_bioen_kernels_logw.c:367-509 (GSL multimin driver) and 581-669 (liblbfgs driver).
 * Return fmin; *error receives the GSL status / liblbfgs return code; func_params.result receives x. */
double _opt_bfgs_logw(params_t func_params, gsl_config_params config, visual_params visual, int *error);
double _opt_lbfgs_logw(params_t func_params, lbfgs_config_params config, visual_params visual, int *error);

/* replaces c_bioen_kernels_forces.c:111-224 -- w ~ w0 * exp(+ yTilde^T forces), normalised */
void _get_weights_from_forces(const double *w0, const double *yTilde, const double *forces, double *w,
                              int caching, const double *yTildeT, double *tmp_n, size_t m, size_t n);

/* replaces c_bioen_kernels_forces.c:227-277.  NOTE: like the reference this takes the WEIGHTS `w`, not the
 * forces; the device recomputes nothing here: KL and chi^2 are evaluated for the given w. */
double _bioen_log_posterior_forces(const double *w0, const double *yTilde, const double *YTilde, const double *w,
                                   const double *result, double theta, int caching, const double *yTildeT,
                                   double *tmp_n, double *tmp_m, int m, int n);

/* replaces c_bioen_kernels_forces.c:280-340 -- gradient w.r.t. the forces for the given weights w */
void _grad_bioen_log_posterior_forces(const double *w0, const double *yTilde, const double *YTilde,
                                      const double *w, double *gradient, double theta, int caching,
                                      const double *yTildeT, double *tmp_n, double *tmp_m, int m, int n);

/* replace c_bioen_kernels_forces.c:431-570 and 574-662 */
double _opt_bfgs_forces(params_t func_params, gsl_config_params config, visual_params visual, int *error);
double _opt_lbfgs_forces(params_t func_params, lbfgs_config_params config, visual_params visual, int *error);

/* c_bioen_common.c:32-61.  Both minimiser families are built in (no external GSL / liblbfgs needed): 1, 1.
 * The "fast OpenMP" flag is stored and returned but has no effect: device reductions are always fixed-order
 * (the reproducible mode).  _omp_set_num_threads is a no-op. */
int _library_gsl(void);
int _library_lbfgs(void);
void _omp_set_num_threads(int n);
void _set_fast_openmp_flag(int flag);
int _get_fast_openmp_flag(void);

/* c_bioen_error.c:14-115 -- message texts for GSL status codes and liblbfgs return codes */
const char *bioen_gsl_error(int gsl_errno);
const char *lbfgs_strerror(int error);

/* ------------------------------------------------------------------------------------------------
 * Part 2 -- handle API (yTilde resident in HBM)
 * All functions returning int return 0 on success, non-zero on failure (text: bioen_b200_last_error()).
 * ------------------------------------------------------------------------------------------------ */
typedef struct bioen_b200_ctx bioen_b200_ctx;

enum { BIOEN_B200_LOGW = 0, BIOEN_B200_FORCES = 1 };

const char *bioen_b200_last_error(void);
/* 1 if any entry point (part 1 included: those cannot return a status) failed on this thread since the last
 * call of this function; the flag is cleared by reading it */
int bioen_b200_error_pending(void);
int bioen_b200_device_count(void);

/* (m x n) = shape of the LOCAL block of yTilde (all of it on one GPU; this rank's columns when sharded) */
bioen_b200_ctx *bioen_b200_create(int m, int n, int device);
void bioen_b200_destroy(bioen_b200_ctx *ctx);

/* copy yTilde from host memory (row stride ld doubles) into HBM, or adopt a matrix already on the device
 * (even row stride, 16-byte aligned base; the caller keeps ownership) */
int bioen_b200_upload_ytilde(bioen_b200_ctx *ctx, const double *yTilde_host, size_t ld);
int bioen_b200_adopt_ytilde(bioen_b200_ctx *ctx, double *yTilde_dev, size_t ld);
/* chunked upload: copy rows [row0, row0+nrows) of yTilde from host memory (row stride ld doubles).  The device
 * matrix is allocated on the first call; a matrix larger than host memory can be streamed from disk block by block.
 * Call before bioen_b200_set_logw / bioen_b200_set_forces. */
int bioen_b200_upload_rows(bioen_b200_ctx *ctx, int row0, int nrows, const double *rows_host, size_t ld);
/* page-locked host memory: matrices and vectors that live in it are uploaded by plain asynchronous copies at PCIe
 * speed (bioen_b200_upload_ytilde detects it); NULL on failure */
void *bioen_b200_host_alloc(size_t bytes);
void bioen_b200_host_free(void *p);
/* allocate a zeroed device matrix for bioen_b200_generate_ytilde */
int bioen_b200_alloc_ytilde(bioen_b200_ctx *ctx);
/* copy the block [row0, row0+nrows) x [col0, col0+ncols) of the resident matrix to out_host (row-major, dense) */
int bioen_b200_download_ytilde(bioen_b200_ctx *ctx, int row0, int nrows, long long col0, long long ncols,
                               double *out_host);

/* per-method constant data: reference log-weights G[n] or reference weights w0[n], YTilde[m], theta */
int bioen_b200_set_logw(bioen_b200_ctx *ctx, const double *G_host, const double *YTilde_host, double theta);
int bioen_b200_set_forces(bioen_b200_ctx *ctx, const double *w0_host, const double *YTilde_host, double theta);
int bioen_b200_set_theta(bioen_b200_ctx *ctx, double theta);
/* tuning switches.  BIOEN_B200_OPT_FUSED_FORCES (default 1; call before bioen_b200_set_forces): keep a
 * structure-major copy of yTilde and evaluate the forces method in two fused passes instead of four.
 * BIOEN_B200_OPT_P2P (default 1; after bioen_b200_comm_init, on all ranks together): carry the per-evaluation
 * exchanges with the library's peer-memory kernel over NVLink instead of NCCL.
 * BIOEN_B200_OPT_LAZY_GRADIENT (default 1): the minimisers run the gradient half of an evaluation only when the
 * algorithm reads it (backtracking trials that fail the sufficient-decrease test skip it; GSL's f-then-df on one
 * point does not repeat the objective half).  Results are bit-identical either way; 0 exists for that comparison.
 * BIOEN_B200_OPT_FUSED_EXCHANGE (default 1; all ranks together): sharded log-weights evaluations and L-BFGS dot
 * products exchange from INSIDE the kernels that produce the values (no exchange launches; the log-sum-exp pair travels
 * with the row sums: one exchange per objective half).  0 restores the three separate exchanges per evaluation.
 * BIOEN_B200_OPT_PERSISTENT (default -1 = by size; 0 off; 1 on): run an evaluation as ONE persistent cooperative
 * kernel (grid barriers between its phases, yTilde kept in L2 when it fits) instead of 6-11 kernel launches; auto
 * selects it for matrices up to 0.6 GB per GPU.
 * BIOEN_B200_OPT_LBFGS_GRAM (default 0): the L-BFGS direction update runs in
 * coefficient space -- 2 kernels and 1 exchange per iteration instead of 14 and 13.  Algebraically the two-loop
 * recursion of liblbfgs, but it rounds differently, so trajectories differ from the default path in the last bits.
 * BIOEN_B200_OPT_FP32_STORAGE (default 0; set to 1 AFTER the matrix is uploaded / generated): replace the resident fp64
 * matrix by an fp32 copy.  Halves the bytes every pass streams (the roofline of an evaluation); products and sums stay
 * fp64, but the matrix entries carry fp32 rounding (relative 6e-8), so results are NOT within the 1e-11 parity bar
 * (measured: objective ~1e-8, gradient ~1e-7 relative; tests/test_gpu_fp32_storage.py).  Never the default.  The fused
 * forces kernels, the theta scan, downloads and row-affine transforms need the fp64 matrix and are unavailable.
 * BIOEN_B200_OPT_SLICE (default -1 = on when eligible; 0 off): problems small enough for
 * the CTAs to hold their columns of yTilde in shared memory (up to ~30 MB in all, e.g. every fixture of the
 * reference's test-suite and the ala5 example) run an evaluation as ONE cooperative kernel with ONE grid barrier: the
 * matrix is read once per launch and every sweep runs out of shared memory (csrc/slice_eval.cuh).  Takes precedence
 * over the persistent kernel and the fused forces kernels; BIOEN_B200_OPT_PERSISTENT = 0 disables it as well.
 * BIOEN_B200_OPT_LBFGS_SMALL (default 1): minimisations over at most 1024
 * variables (the forces method; log-weights with few structures) run the L-BFGS update -- the new (s, y) pair and the
 * two-loop recursion -- as ONE single-CTA kernel instead of 15 launches; same arithmetic, bit-identical up to 256
 * variables.
 * BIOEN_B200_OPT_LBFGS_SPECULATIVE (default 1): the first trial of a line
 * search is enqueued behind the update without fetching the initial slope first (it arrives with the trial's scalars):
 * one host round trip per iteration instead of two.  Results are identical.
 * BIOEN_B200_OPT_STRUCTURE_MAJOR_ONLY (default 0; set to 1 before the matrix is uploaded / generated, or afterwards: the
 * resident matrix is then transposed once and released): the context holds ONLY the structure-major copy that the
 * fused two-pass forces kernels read -- half the device memory of the default forces set-up (which keeps both
 * layouts), e.g. 8 GB instead of 16 GB at N = 1e6 x M = 1e3, and 100 GB per GPU instead of 200 GB for N = 1e7 x M = 5e3
 * on 4 GPUs.  Uploads are transposed chunk by chunk through a 256 MB staging buffer, the generator writes the
 * structure-major layout directly.  Available: forces evaluations and minimisers (256 <= M <= ~5500), weights,
 * averages, downloads; the log-weights method, the theta scan, row-affine transforms and the given-weights entry
 * points need the row-major matrix and fail with a message.
 * BIOEN_B200_OPT_FETCH_ZEROCOPY (default 1): the 512-byte scalar file of an
 * evaluation reaches the host through stores of a one-warp kernel into page-locked memory + a sequence number the host
 * spins on, instead of a copy-engine transfer and an event.  Same values; a few microseconds less per evaluation.
 * Options 1, 3, 4, 5, 6, 8, 9, 10 and 12 belong to the context; bioen_b200_create starts every one at its default
 * (bioen_b200_query what = 10 reports which differ from it). */
enum { BIOEN_B200_OPT_FUSED_FORCES = 1, BIOEN_B200_OPT_P2P = 2, BIOEN_B200_OPT_LAZY_GRADIENT = 3,
       BIOEN_B200_OPT_FUSED_EXCHANGE = 4, BIOEN_B200_OPT_PERSISTENT = 5, BIOEN_B200_OPT_LBFGS_GRAM = 6,
       BIOEN_B200_OPT_FP32_STORAGE = 7, BIOEN_B200_OPT_SLICE = 8, BIOEN_B200_OPT_LBFGS_SMALL = 9,
       BIOEN_B200_OPT_LBFGS_SPECULATIVE = 10, BIOEN_B200_OPT_STRUCTURE_MAJOR_ONLY = 11,
       BIOEN_B200_OPT_FETCH_ZEROCOPY = 12 };
int bioen_b200_set_option(bioen_b200_ctx *ctx, int option, int value);

/* one evaluation with host vectors.  grad_host may be NULL (objective only: one pass over yTilde instead of
 * two for logw, two instead of four for forces). */
int bioen_b200_eval(bioen_b200_ctx *ctx, int method, const double *x_host, double *f, double *grad_host);
/* gradient at the point of the LAST objective-only bioen_b200_eval of `method` (SciPy-style callers ask f(x) and
 * then fprime(x)): only the gradient half runs, bit-identical to a full evaluation.  Returns 2 and does nothing
 * when no such evaluation is pending (any other call on the context in between voids it). */
int bioen_b200_grad_continue(bioen_b200_ctx *ctx, int method, double *grad_host);
/* weights for log-weights g[n] / forces f[m]; w_host[n]; *sum (may be NULL) = sum_j exp(g_j) for logw */
int bioen_b200_weights(bioen_b200_ctx *ctx, int method, const double *x_host, double *w_host, double *sum);
/* avg[m] = yTilde . w for host w[n] (post-processing with the resident matrix) */
int bioen_b200_average(bioen_b200_ctx *ctx, const double *w_host, double *avg_host);
/* in-place row-affine transform of the resident matrix: yTilde_ij <- scale[i] * yTilde_ij + offset[i] (host vectors of m
 * entries).  Commits refitted nuisance parameters -- DEER modulation depth: (1 - m + m s_ij) / err_i, scattering scale:
 * c s_ij / err_i, both affine in the rows -- to the matrix in HBM instead of rebuilding and re-uploading it
 * (the reference rebuilds it on the host: bioen/analyze/observables/observables.py:110-143, 191-216).  One read and
 * one write pass over the matrix.  A structure-major copy made for the forces method is rebuilt.  Not available for
 * adopted matrices (caller-owned). */
int bioen_b200_affine_rows(bioen_b200_ctx *ctx, const double *scale_host, const double *offset_host);
/* objective / gradient of the forces method for GIVEN weights w[n] (reference semantics, part 1) */
int bioen_b200_forces_from_weights(bioen_b200_ctx *ctx, const double *w_host, double *f, double *grad_host);

/* minimisers; x0_host/x_host have n (logw) or m (forces) entries and may alias.  The function result is the
 * minimiser's own status (liblbfgs return code / GSL status, see part 1); *fmin the final objective;
 * info[0] = iterations.  GSL: info[1] = gradient evaluations, info[2] = f-only probes, info[3] = how many of info[1]
 * ran one half of the evaluation only (gradient of the point just probed; rejected steepest-descent steps).  L-BFGS: info[1] = callback
 * evaluations as liblbfgs counts them, info[2] = how many of those were line-search trials that failed the
 * sufficient-decrease test, for which the gradient pass over yTilde was skipped (liblbfgs never reads it).
 * A CUDA failure returns -2000 and sets bioen_b200_last_error(). */
int bioen_b200_opt_lbfgs(bioen_b200_ctx *ctx, int method, const double *x0_host, double *x_host,
                         lbfgs_config_params config, visual_params visual, double *fmin, int info[4]);
int bioen_b200_opt_gsl(bioen_b200_ctx *ctx, int method, const double *x0_host, double *x_host,
                       gsl_config_params config, visual_params visual, double *fmin, int info[4]);

/* theta scan (L-curve): K <= 32 problems of one method that differ only in theta (and start point) minimised
 * together by K lockstep L-BFGS machines; every pass streams yTilde once for all K (fp64 tensor-core skinny GEMMs:
 * two per evaluation for BIOEN_B200_LOGW, four for BIOEN_B200_FORCES).  Requires bioen_b200_set_logw /
 * bioen_b200_set_forces (their theta is ignored).  x0_host / x_host: [K][n] row-major, n = N (logw) or M (forces);
 * fmin[K]; codes[K] (liblbfgs return codes); info[2K] = {iterations, evaluations} per problem; stats[4] = {lockstep rounds, GEMM
 * launches, seconds, 0}.  The reference's counterpart is the Python loop over theta in
 * bioen/analyze/procedure.py:62-83. */
int bioen_b200_theta_scan(bioen_b200_ctx *ctx, int method, int K, const double *thetas, const double *x0_host,
                          double *x_host, lbfgs_config_params config, visual_params visual, double *fmin, int *codes, int *info,
                          double *stats);

/* batched replicates: K <= 32 problems of one method that share the resident yTilde and differ in theta, start
 * point and, per problem, in any of the arrays below (row-major host arrays; NULL = every problem uses the vector the
 * context holds).  The bootstrap (resampled observables, structures or experimental noise) and cross-validation over
 * observables are batches of this kind; they run on the theta scan's lockstep engine.
 *   YTilde      [K][M]  observed data of each problem (noise replicates); finite
 *   row_weights [K][M]  observable weights c_i >= 0, finite: chi^2 = 1/2 sum_i c_i r_i^2 (resampled or held-out rows)
 *   w0          [K][N]  reference weights >= 0, finite, positive sum (resampled structures); BIOEN_B200_FORCES only:
 *                       the log-weights parametrisation cannot represent a structure of weight zero
 *   row_scale   [K][M]  a_i, finite (zeros allowed); NULL = all ones
 *   row_offset  [K][M]  b_i, finite; NULL = all zeros.  Problem k is the one of the matrix a_i yTilde_ij + b_i
 *                       (row-affine nuisance parameters: DEER modulation depth, scattering scale factor) while the
 *                       resident yTilde is neither read twice nor changed.  Its averages are a_i avg_i + b_i; the avg
 *                       outputs below stay yTilde . w of the RESIDENT matrix.
 * Invalid arrays, and sharded contexts, are refused before anything runs.  Fields may be added at the end of the
 * struct: zero-initialise it (e.g. `bioen_b200_batch b = {0};`) so that fields a caller does not know are NULL. */
typedef struct bioen_b200_batch {
    int K;
    const double *thetas;        /* [K] */
    const double *YTilde;
    const double *row_weights;
    const double *w0;
    const double *row_scale;
    const double *row_offset;
} bioen_b200_batch;

/* lockstep L-BFGS of the batch: x0_host / x_host, fmin, codes, info, stats as for bioen_b200_theta_scan (which is this
 * call with every array NULL).  Then one objective evaluation at the returned points gives, per problem,
 * avg[K][M] = yTilde . w(x_k) of the resident matrix, chi2[K] (with the row weights and the row-affine transform)
 * and kl[K] (the relative entropy, without theta); each
 * may be NULL.  All three are NaN when the L-BFGS parameters are refused. */
int bioen_b200_batch_minimize(bioen_b200_ctx *ctx, int method, const bioen_b200_batch *batch, const double *x0_host,
                              double *x_host, lbfgs_config_params config, visual_params visual, double *fmin,
                              int *codes, int *info, double *stats, double *avg, double *chi2, double *kl);
/* one batched evaluation at x_host[K][n]: f[K], grad_host[K][n] (NULL: objective half only), avg[K][M], chi2[K],
 * kl[K] (each may be NULL) */
int bioen_b200_batch_eval(bioen_b200_ctx *ctx, int method, const bioen_b200_batch *batch, const double *x_host,
                          double *f, double *grad_host, double *avg, double *chi2, double *kl);

/* bench.py: time `steps` batched f+g evaluations of K problems (CUDA events); *gemm_ms = mean duration of one
 * skinny-GEMM launch.  bioen_b200_time_batch_evals: the same for a batch with per-problem arrays.  bioen_b200_dmma_peak: fp64 tensor-core peak of the device, measured with a
 * register-resident mma.sync.m8n8k4.f64 loop (the roofline denominator of the GEMMs). */
int bioen_b200_time_scan_evals(bioen_b200_ctx *ctx, int method, int K, const double *thetas, const double *x0_host,
                               int warmup, int steps, float *ms, float *gemm_ms, long long *launches);
int bioen_b200_time_batch_evals(bioen_b200_ctx *ctx, int method, const bioen_b200_batch *batch, const double *x0_host,
                                int warmup, int steps, float *ms, float *gemm_ms, long long *launches);
int bioen_b200_dmma_peak(int device, double *tflops);
/* mean GB/s of `reps` launches of a plain read-only stream (16-byte loads, nothing written) over the resident
 * yTilde: what a read-only pass can reach on this device, next to the copy figure of MEASURED_PEAKS.json */
int bioen_b200_read_stream_peak(bioen_b200_ctx *ctx, int reps, double *gbs);

/* host-only test hook (no GPU needed): runs the liblbfgs line search selected by config (More-Thuente or one of
 * the three backtracking variants, lbfgs.c:645-1001) on the 1-D function phi(stp) -> (f, df/dstp).  Returns the
 * liblbfgs verdict (> 0: number of trials on success, < 0: error code). */
int bioen_b200_selftest_linesearch(lbfgs_config_params config, double finit, double dginit, double stp0,
                                   void (*phi)(double stp, double *f, double *dg), double *stp_out, double *f_out,
                                   int *ntrials);

/* host-only test hook: quadratic / cubic interpolation of GSL's Fletcher line minimisation (linear_minimize.c) */
double bioen_b200_selftest_interpolate(double a, double fa, double fpa, double b, double fb, double fpb, double xmin,
                                       double xmax, int order);

/* host-only test hooks: the tile sequence CTA `cta` of a matrix pass walks (pass_mode 0 row pass, 1 column pass;
 * arrays of max_tiles entries: tile coordinates, partial-sum slot, 1 where the CTA's part of a run ends; returns the
 * number of tiles), and the number of slots the readers of the partial sums expect for a run */
long long bioen_b200_selftest_tilewalk(int pass_mode, int nRT, int nCB, int grid, long long chunk, int interleave,
                                       int cta, long long max_tiles, int *rt, int *cb, long long *slot, int *closes);
int bioen_b200_selftest_num_slots(long long run, long long L, long long chunk);
/* host-only test hook: the launch geometry of the shared-memory slice kernel (csrc/slice_eval.cuh, slice_plan) for an
 * m x n problem on a device with `sms` SMs and `max_dyn_smem` bytes of dynamic shared memory per CTA.  Returns 1 when
 * the problem is eligible; out = {columns per CTA, row stride of the slice, record stride of the tables, CTAs,
 * log2 threads along the columns (column sums), log2 lanes per row (row sums), log2 lanes per row (table sums),
 * dynamic shared memory in bytes}. */
int bioen_b200_selftest_slice_plan(int m, int n, int sms, long long max_dyn_smem, long long out[8]);
/* host-only test hook: the schedule of the two-loop recursion over the `bound` newest pairs of an m-slot ring whose
 * newest pair is in slot end - 1 (1 <= m <= 16, 1 <= bound <= m, 0 <= end < m).  Writes 2*bound + 1 steps of 11 ints,
 * {init, u_kind, u_slot, v_kind, v_slot, c_num, c_den, csign, c2_num, scale, out}, to steps and returns their number
 * (-1: arguments out of range).  One step is d <- (init ? -g : d) + coef * u ; d *= sc[16] / sc[17] when scale ;
 * sc[out] = v . d, where coef = csign * sc[c_num] / sc[c_den] (- sc[c2_num] / sc[c_den] when c2_num >= 0), kinds are
 * 0 none, 1 s_slot, 2 y_slot, 3 g, and sc is the 64-double scalar file (ys ring at 24, raw s.d ring at 40). */
int bioen_b200_selftest_twoloop_schedule(int end, int bound, int m, int *steps);
/* device test hook: ONE L-BFGS direction update (new pair s = x - xp, y = g - gp into ring slot end_old, then the
 * two-loop recursion over `bound` pairs, lbfgs.c:543-598) from a given state, on engine 0 (multi-kernel), 1 (single-CTA
 * kernel, unsharded, n <= 1024), 2 (coefficient space with the resident Gram matrix, filled first from S and Y, its
 * diagonal s_t . y_t from ys_ring; reachable states only: bound < 6 needs end_old = bound - 1) or 3
 * (the batched planes of the theta scan; unsharded contexts), through the same host code as the minimisers.  n = N
 * (BIOEN_B200_LOGW; this rank's columns when sharded) or M (BIOEN_B200_FORCES); m = 6; K problems (1 for engines 0-2,
 * 1..32 for engine 3; engine 3 needs bioen_b200_set_logw / _set_forces first).  Row-major host arrays:
 *   in      end_old[K] in 0..5, bound[K] in 1..6 (0: inactive problem, engine 3), x[K][n], g[K][n], ys_ring[K][m]
 *   in/out  xp[K][n], gp[K][n], S[K][m][n], Y[K][m][n], d[K][n], scalars[K][64] (the scalar file; its ys ring is
 *           replaced by ys_ring on input)
 * An inactive problem's arrays come back as they went in. */
int bioen_b200_selftest_lbfgs_update(bioen_b200_ctx *ctx, int engine, int method, int K, const int *end_old,
                                     const int *bound, const double *x, const double *g, double *xp, double *gp,
                                     double *S, double *Y, const double *ys_ring, double *d, double *scalars);

/* multi-GPU: one process per GPU, N sharded.  Rank 0 creates the id, the host layer broadcasts it. */
int bioen_b200_nccl_unique_id(char id[128]);
int bioen_b200_comm_init(bioen_b200_ctx *ctx, const char id[128], int rank, int nranks, long long n_total);
/* the same for a group of contexts inside ONE process (one host thread per rank, every rank calls this with the same
 * `group` >= 0; the same or different devices): no NCCL, no IPC -- the ranks find each other through a process-wide
 * table and exchange over peer memory only.  This is how the sharded path runs on a single-GPU box (tests), and a
 * single-process multi-GPU program can use it as well.  Messages above the inbox size (theta scan) are not supported. */
int bioen_b200_comm_init_local(bioen_b200_ctx *ctx, int group, int rank, int nranks, long long n_total);
/* how the per-evaluation exchanges travel: 0 single rank, 1 NCCL, 2 peer-memory kernel (CUDA IPC + NVLink) */
int bioen_b200_comm_mode(bioen_b200_ctx *ctx);

/* device-pointer entry points (inputs already resident in HBM; used by bench.py and torch carriers).
 * Everything is enqueued on the context's stream; bioen_b200_fetch waits for it. */
int bioen_b200_set_logw_dev(bioen_b200_ctx *ctx, const double *G_dev, const double *YTilde_host, double theta);
int bioen_b200_set_forces_dev(bioen_b200_ctx *ctx, const double *w0_dev, const double *YTilde_host, double theta);
int bioen_b200_eval_dev(bioen_b200_ctx *ctx, int method, double *x_dev, double *grad_dev);
int bioen_b200_fetch(bioen_b200_ctx *ctx, double *f, double *gnorm2);
int bioen_b200_opt_lbfgs_dev(bioen_b200_ctx *ctx, int method, double *x_dev, lbfgs_config_params config,
                             visual_params visual, double *fmin, int info[4]);
/* time `steps` evaluations (after `warmup` untimed ones) with CUDA events on the context's stream.
 * Successive steps evaluate at x + k*eps*dir so no step repeats the previous one.  Returns total ms in *ms,
 * the mean duration of one yTilde pass kernel in *pass_ms, and the number of kernels launched inside the
 * timed region in *launches. */
int bioen_b200_time_evals(bioen_b200_ctx *ctx, int method, double *x_dev, double *grad_dev, int warmup, int steps,
                          float *ms, float *pass_ms, long long *launches);
/* generate a synthetic "generic data" yTilde block on the device (counter-based RNG, reproducible per
 * (seed, row, global column)); see bench.py */
int bioen_b200_generate_ytilde(bioen_b200_ctx *ctx, unsigned long long seed, long long col_offset,
                               const double *ytrue_over_sigma_host, double inv_sigma);
long long bioen_b200_kernels_launched(bioen_b200_ctx *ctx);
/* facts about how the context evaluates (bench.py, tests): what = 0: 1 if the forces method runs on the fused
 * two-pass kernels; 1 / 2: exchanges between the ranks per log-weights / forces f+g evaluation (0 on one GPU);
 * 3: 1 if evaluations run as ONE persistent cooperative kernel with yTilde held in L2 (small problems);
 * 4: bytes per element of the resident matrix (8, or 4 with BIOEN_B200_OPT_FP32_STORAGE); 5: one-launch evaluations
 * (persistent or slice kernel) so far; 6: of those, launches of the shared-memory slice kernel; 7: 1 if evaluations
 * run on the slice kernel now; 8: bytes of device memory held by the context's copies of yTilde (row-major +
 * structure-major + fp32); 9: 1 in structure-major-only mode; 10: bitmask with bit (1 << option) set for each of the
 * options 1, 3, 4, 5, 6, 8, 9, 10 and 12 whose value differs from its default.  Returns -1 for an unknown `what`. */
long long bioen_b200_query(bioen_b200_ctx *ctx, int what);
/* copy `count` doubles of a device buffer the context holds (tests): what = 0 the scalar file (64), 1 weights, 2
 * averages, 3 / 4 the forces method's per-structure vectors, 5 the L-BFGS store of the last minimisation,
 * [g | xp | gp | d | s_0..s_5 | y_0..y_5] with each vector's n rounded up to 16 */
int bioen_b200_debug_read(bioen_b200_ctx *ctx, int what, double *out_host, size_t count);
/* the context's cudaStream_t (for callers that enqueue their own work around the device entry points) */
void *bioen_b200_stream(bioen_b200_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* BIOEN_B200_H */
