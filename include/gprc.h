/*
 * gprc.h -- C ABI of libgprc, the B200 (sm_100a) implementation of the Gaussian-process hot path of the R
 * package `gprc` (MoHawastaken/Gaussian-Process-Regression).
 *
 * The reference has no FFI layer (pure R, SURVEY.md section 8b); these entry points are what a `.Call` shim
 * (src/gprc_shim.c) binds so that R/GPRclass.R, R/GPCclass.R and R/fit.R keep their signatures.  Every function
 * cites the reference lines it replaces.  Conventions:
 *   - all matrices are column-major FP64 (R's layout); X is d x n with leading dimension d (points contiguous,
 *     reference R/GPRclass.R:132,137);
 *   - plain pointers and sizes only; the caller owns every host buffer, the library owns device memory behind the
 *     opaque handles;
 *   - return value: 0 = ok, < 0 = CUDA/argument error (text in gprc_last_error()); numerical failure is reported
 *     LAPACK-style through `info` (> 0: 1-based index of the first non-positive pivot), never by a non-zero
 *     return, so the host can run the reference's retry policy (R/GPRclass.R:141-149);
 *   - functions ending in `_dev` take DEVICE pointers for the bulk arrays (bench "value" leg: inputs already in
 *     HBM); all others take HOST pointers and include the copies.
 *   - no CPU fallback exists: without a CUDA device gprc_ctx_create fails.
 */
#ifndef GPRC_H
#define GPRC_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gprc_ctx gprc_ctx; /* one device, one stream, workspaces, phase timers          */
typedef struct gprc_gpr gprc_gpr; /* device: X, L (lower), L^-1 (lazy), alpha; host: logp      */
typedef struct gprc_gpc gprc_gpc; /* device: X, K, f_hat, sqrt(W), L(B); host: objective trace */

/* The six built-in kernels of R/GPRclass.R:381-403 plus "precomputed" for arbitrary R closures. */
typedef enum {
  GPRC_CONSTANT = 0,   /* k = c                                   R/GPRclass.R:382 */
  GPRC_LINEAR = 1,     /* k = sum_d sigma_d x_d y_d               R/GPRclass.R:386 */
  GPRC_POLYNOMIAL = 2, /* k = (x.y + sigma)^p                     R/GPRclass.R:390 */
  GPRC_SQREXP = 3,     /* k = exp(-|x-y|^2 / (2 l^2))             R/GPRclass.R:394 */
  GPRC_GAMMAEXP = 4,   /* k = exp(-(|x-y| / l)^gamma)             R/GPRclass.R:398 */
  GPRC_RATQUAD = 5,    /* k = (1 + |x-y|^2 / (2 alpha l^2))^-alpha R/GPRclass.R:402 */
  GPRC_PRECOMPUTED = 6
} gprc_kernel_id;

/* Parameters are NAMED, never positional (the reference mixes orders, SURVEY.md A.6). */
typedef struct {
  int id; /* gprc_kernel_id */
  double c, sigma, p, l, gamma, alpha;
  const double* sigma_vec; /* HOST pointer; linear kernel with one sigma per dimension (R/GPRclass.R:298), or NULL */
  int sigma_len;           /* 0 => scalar `sigma` is recycled (fit.R:17) */
} gprc_kernel;

/* flags for gprc_ctx_set_option */
enum {
  GPRC_OPT_GRAM_DMMA = 1, /* kernel-matrix build on the FP64 tensor cores (TMA-fed 64 x 64 tiles, X^T Y by DMMA, norm
                             expansion for distances; eligible: sqrexp / rationalquadratic / polynomial / linear, d a
                             multiple of 4 in 4..32).  0: never (direct differences exactly as R/GPRclass.R:394 writes
                             them); 1 (default): where it measured faster (dot-product kernels, d >= 12); 2: wherever
                             eligible */
  GPRC_OPT_PREDICT_PATH = 2, /* variance pass v = L^-1 K_star: 0 auto (default), 1 invert L once and multiply
                               (one launch per chunk; best for repeated / small predicts), 2 blocked substitution with
                               two launches per block row (no n^3/3 inversion), 3 the same substitution as one
                               persistent kernel with per-tile progress counters (chosen automatically for >= 18 944
                               test points when no inverse exists yet), 4 the substitution with its O(n^2 m) products
                               on the INT8 tensor cores (tcgen05, Ozaki digit splitting; FP64 diagonal solves) */
  GPRC_OPT_OZAKI_DIGITS = 3, /* 8-bit digits per operand entry on path 4: 6, 7 (default; 54 bits below the row /
                               column maximum) or 8 */
  GPRC_OPT_INT8_AUTO = 4, /* 1 (default): the automatic choice takes path 4 where it takes the substitution today
                            (>= 18 944 test points, no inverse at hand) if n >= 4096; 0: FP64 paths only */
  GPRC_OPT_INT8_TEST_SHRINK = 6, /* tests only: lower the per-test-point exponents of path 4 by this many bits so that
                            v leaves its fixed-point range: the overflow flag must fire and the chunk be redone in FP64 */
  GPRC_OPT_CHOL_TILES = 8, /* Cholesky (R/GPRclass.R:142): matrices of at most this many 128-blocks (n <= 128 * value) are
                        factored by ONE persistent kernel (tile tasks, per-row progress counters) instead of three
                        dependent launches per block column; default 128 (n <= 16 384), 0 = never */
  GPRC_OPT_TRSV = 7, /* alpha = L^-T L^-1 y (R/GPRclass.R:152): 1 (default) both sweeps as one dataflow kernel (a CTA per
                        row block; consumers poll the published entries); 0 two cooperative sweeps with a grid-wide
                        barrier per block step (round 1) */
  GPRC_OPT_INT8_TILE = 5 /* kernel of path 4 (all give the same digits; 1 and 64 are bit-identical):
                            2 (default) stacked digit planes on clusters of two CTAs: one tcgen05.mma multiplies a digit
                              plane of L with up to four planes of V (N up to 256), two block rows of L share every V digit
                              tile through TMA multicast, one small FP64 step inside each pair of block rows;
                            1 stacked digit planes, one block row per launch;
                            64 one MMA per digit pair (round 1: bound by the tensor core's shared-memory operand port);
                            128 128 x 128 tiles with the orders in two passes (round 1) */

};

/* what to fetch with gprc_gpr_get / gprc_gpc_get */
enum {
  GPRC_GET_L = 0,     /* n x n, lower, explicit zeros above the diagonal (R: t(chol(.)))   */
  GPRC_GET_ALPHA = 1, /* n                                                                  */
  GPRC_GET_LINV = 2,  /* n x n lower, L^-1 (forces the inversion)                           */
  GPRC_GET_FHAT = 3,  /* n    (GPC)                                                         */
  GPRC_GET_SQRTW = 4  /* n    (GPC)                                                         */
};

/* gradient formulas for gprc_logml_grad */
enum {
  GPRC_GRAD_AS_CODED = 0, /* fit.R:128-138 literally: noise-free K, 0.5*sum(diag(aa'-K^-1) %*% dK)  (A.5) */
  GPRC_GRAD_TEXTBOOK = 1  /* 0.5 tr((aa' - Ky^-1) dK) with Ky = K + noise I (vignettes/gpr.Rmd:137)      */
};

/* phase timers (milliseconds, CUDA events on the library's stream; accumulated since gprc_ctx_reset_timers) */
enum {
  GPRC_T_BUILD_K = 0,   /* covariance_matrix(X, X, k) + noise       */
  GPRC_T_CHOL = 1,      /* blocked Cholesky                         */
  GPRC_T_SOLVE = 2,     /* alpha (two triangular solves) + logp     */
  GPRC_T_TRTRI = 3,     /* L^-1                                     */
  GPRC_T_BUILD_KS = 4,  /* K_star tiles + mean                      */
  GPRC_T_VAR = 5,       /* v = L^-1 K_star with fused column norms  */
  GPRC_T_NEWTON = 6,    /* GPC Newton loop                          */
  GPRC_T_PREDICT = 7,   /* whole predict call (K_star build + variance pass + finalize) as one span */
  GPRC_T_COUNT = 8
};

/* ---- context ------------------------------------------------------------------------------------------- */
int gprc_ctx_create(gprc_ctx** out, int device);
void gprc_ctx_free(gprc_ctx* ctx);
int gprc_ctx_set_option(gprc_ctx* ctx, int option, int value);
int gprc_ctx_sync(gprc_ctx* ctx);
/* Long predicts poll `fn(user)` between chunks of test points (every few hundred ms at n = 50k); a non-zero return
 * abandons the call with status -8 ("interrupted") after the queued work has drained.  The R shim installs a callback
 * that asks R for a pending user interrupt without long-jumping (R_ToplevelExec around R_CheckUserInterrupt), SURVEY.md 8b.
 * fn = NULL removes it. */
typedef int (*gprc_interrupt_fn)(void* user);
int gprc_ctx_set_interrupt(gprc_ctx* ctx, gprc_interrupt_fn fn, void* user);
void gprc_ctx_reset_timers(gprc_ctx* ctx);
int gprc_ctx_get_timers(gprc_ctx* ctx, double* ms /* GPRC_T_COUNT */, long* kernel_launches);
/* user event pair on the library's stream: device-side timing of an arbitrary region (bench.py) */
int gprc_ctx_mark(gprc_ctx* ctx, int slot /* 0..7 */);
int gprc_ctx_elapsed_ms(gprc_ctx* ctx, int slot_start, int slot_stop, double* ms);
/* variance-pass path (1..4, see GPRC_OPT_PREDICT_PATH) the most recent predict on this context resolved to; 0 = none yet */
/* Device memory freed by the library is kept in a per-context caching allocator (an optimiser calls gprc_logml hundreds
   of times); this hands the parked blocks back to the driver.  *bytes (nullable) = bytes released. */
int gprc_ctx_trim(gprc_ctx* ctx, unsigned long long* bytes);
int gprc_ctx_last_predict_path(gprc_ctx* ctx);
/* chunks of test points that predict was cut into (each chunk reads the factor once: bench.py's algorithmic bytes) */
long gprc_ctx_last_predict_chunks(gprc_ctx* ctx);
const char* gprc_last_error(void);
int gprc_version(void);

/* ---- device memory helpers (bench / tests; the R shim never needs them) ---------------------------------- */
int gprc_dev_malloc(gprc_ctx* ctx, void** dptr, unsigned long long bytes);
int gprc_dev_free(gprc_ctx* ctx, void* dptr);
int gprc_dev_h2d(gprc_ctx* ctx, void* dptr, const void* host, unsigned long long bytes);
int gprc_dev_d2h(gprc_ctx* ctx, void* host, const void* dptr, unsigned long long bytes);
int gprc_host_register(void* host, unsigned long long bytes);   /* pin an existing host buffer */
int gprc_host_unregister(void* host);

/* ---- (1) kernel-matrix build ----------------------------------------------------------------------------- */
/* covariance_matrix(A, B, k), R/GPRclass.R:355-357.  out is nA x nB column-major (host). */
int gprc_cov_matrix(gprc_ctx* ctx, const gprc_kernel* k, const double* A, int d, long nA, const double* B, long nB,
                    double* out);
/* k(A, B) applied column-wise to two d x n matrices: the `.matrix` contract, R/GPRclass.R:378-403. out: n (host). */
int gprc_cov_pointwise(gprc_ctx* ctx, const gprc_kernel* k, const double* A, const double* B, int d, long n,
                       double* out);

/* ---- (2)+(3) GPR: K build, Cholesky of K + noise I, alpha, logp -- GPR$initialize, R/GPRclass.R:138-153 ----- */
/* One attempt with the given noise; *info > 0 means chol() would have thrown: the host re-calls with the next
 * noise of the schedule R/GPRclass.R:141-148.  On info > 0 no model is created (*out = NULL). */
int gprc_gpr_fit(gprc_ctx* ctx, const gprc_kernel* k, const double* X, int d, long n, const double* y, double noise,
                 gprc_gpr** out, double* logp, long* info);
int gprc_gpr_fit_dev(gprc_ctx* ctx, const gprc_kernel* k, const double* dX, int d, long n, const double* dy,
                     double noise, gprc_gpr** out, double* logp, long* info);
/* k is an arbitrary closure evaluated by the host: K (n x n, no noise added yet) comes in precomputed. */
int gprc_gpr_fit_precomputed(gprc_ctx* ctx, const double* K, long n, const double* y, double noise, gprc_gpr** out,
                             double* logp, long* info);
/* Append k training points (Xnew: d x k, points contiguous; ynew: k) to a fitted model, in place.  Afterwards the
 * model is what gprc_gpr_fit gives for cbind(X, Xnew), c(y, ynew) with the model's noise (the possibly bumped one),
 * up to rounding.  *logp receives the new log marginal likelihood.  info > 0: the enlarged K + noise I is not positive
 * definite (1-based row); the model is left exactly as it was.  Built-in kernels only: a closure-kernel
 * (precomputed) model returns an argument error. */
int gprc_gpr_append(gprc_gpr* g, const double* Xnew, long k, const double* ynew, double* logp, long* info);
/* GPR$predict(X_star, pointwise_var = TRUE), R/GPRclass.R:155-165: mean (m), var (m). */
int gprc_gpr_predict(gprc_gpr* g, const double* Xs, long m, double* mean, double* var);
int gprc_gpr_predict_dev(gprc_gpr* g, const double* dXs, long m, double* dmean, double* dvar);
/* precomputed K_star (n x m) and kss = k(X_star, X_star) (m) for closure kernels */
int gprc_gpr_predict_precomputed(gprc_gpr* g, const double* Ks, const double* kss, long m, double* mean, double* var);
/* Test grids on the device (SURVEY.md 8f-4): the points combine_all(lapply(1:d, function(k) seq(lo_k, hi_k, length.out =
 * per_dim))) of R/simulation.R:101-102, 338-349 -- d x per_dim^d, points contiguous, first dimension slowest.
 * limits: d x 2 (lo, hi per dimension, row-major pairs).  gprc_grid_points copies the grid to the host (tests,
 * plotting); gprc_gpr_predict_grid predicts on it without the grid ever existing on the host. */
int gprc_grid_points(gprc_ctx* ctx, const double* limits, int d, int per_dim, double* out);
int gprc_gpr_predict_grid(gprc_gpr* g, const double* limits, int per_dim, double* mean, double* var);

/* GPR$predict(X_star, pointwise_var = FALSE), R/GPRclass.R:167-168: mean (m), cov (m x m). */
int gprc_gpr_predict_cov(gprc_gpr* g, const double* Xs, long m, double* mean, double* cov);
int gprc_gpr_get(gprc_gpr* g, int what, double* host);
long gprc_gpr_n(const gprc_gpr* g);
/* nrow(X) of the model (0 for a closure-kernel model): the shim checks nrow(X_star) against it before any buffer of
   d x m doubles is read (the reference fails with "non-conformable arrays" in covariance_matrix, R/GPRclass.R:356) */
int gprc_gpr_dim(const gprc_gpr* g);
void gprc_gpr_free(gprc_gpr* g);

/* ---- fit(): log marginal likelihood and gradient -- dens / dens_deriv, R/fit.R:117-139 -------------------- */
/* logp as fit.R:121-123.  min_leading_logdet = min_i log det((K + noise I)[1:i,1:i]) = min prefix sum of
 * 2 log L_ii, so the host can apply the literal fit.R:119 rule (det underflow, SURVEY.md A.4) or the
 * Cholesky-success rule.  info > 0: not positive definite. */
int gprc_logml(gprc_ctx* ctx, const gprc_kernel* k, const double* X, int d, long n, const double* y, double noise,
               double* logp, double* min_leading_logdet, long* info);
/* nparam gradient entries in the order of the reference's `v` (the optimiser's parameter vector, fit.R:118):
 * sqrexp (l); gammaexp (l, gamma); rationalquadratic (l, alpha); polynomial (sigma, p). */
int gprc_logml_grad(gprc_ctx* ctx, const gprc_kernel* k, const double* X, int d, long n, const double* y,
                    double noise, int formula, double* grad, int nparam, long* info);
/* nspec independent evaluations (multi-start / grid), the unit that shards across GPUs (SURVEY.md 8e). */
int gprc_logml_batch(gprc_ctx* ctx, const gprc_kernel* specs, int nspec, const double* X, int d, long n,
                     const double* y, double noise, double* logp, double* min_leading_logdet, long* info);

/* ---- fit(): the optimiser inside the library (SURVEY.md 8f-3) -- R/fit.R:47-69, 143-160 --------------------- */
/* Objective / gradient callbacks: return 0 and the value(s), or non-zero when the evaluation fails (the reference's
 * objective throws: stopifnot, chol, solve).  `par` has `npar` entries. */
typedef int (*gprc_objective_fn)(const double* par, int npar, void* user, double* value);
typedef int (*gprc_gradient_fn)(const double* par, int npar, void* user, double* grad);
/* R's Brent_fmin (src/appl/fmin.c: optimize(), optim(method = "Brent")): minimiser of fn on [lower, upper].
 * Returns 1 if fn failed (no R counterpart: the error would propagate), else 0. */
int gprc_optim_brent(gprc_objective_fn fn, void* user, double lower, double upper, double tol, double* xmin);
/* R's vmmin (src/appl/optim.c: optim(method = "BFGS")); par: start -> minimiser.  counts = {fn, gr} evaluations;
 * fail = 1 when maxit was reached.  Returns 1 if the start value is not finite or a callback failed. */
int gprc_optim_vmmin(gprc_objective_fn fn, gprc_gradient_fn gr, void* user, double* par, int npar, int maxit,
                     double abstol, double reltol, double* value, int* counts, int* fail);
/* optim_until_error(start, f, method, ...) with control = list(fnscale = -1) (R/fit.R:47-69,149-150,158): MAXIMISES
 * fn; a failing objective scores -10000; a failing gradient ends the search and the best recorded evaluation wins.
 * method: 0 = Brent on [lower, upper] (npar = 1), 1 = BFGS from `start` (gr required). */
int gprc_optim_until_error(gprc_objective_fn fn, gprc_gradient_fn gr, void* user, const double* start, int npar,
                           int method, double lower, double upper, double* par, double* value);
/* One pass of fit()'s loop body (R/fit.R:113-162) for the covariance family `kernel_id`, entirely inside the library:
 * X (d x n) and y are uploaded once and every dens / dens_deriv evaluation of the trajectory runs on the device
 * (the trajectory is the one fit.py's host optimiser produces through gprc_logml / gprc_logml_grad).
 * minors_rule: 0 = literal R/fit.R:119 (det underflow, SURVEY.md A.4), 1 = Cholesky succeeds.  par (2), npar, value =
 * the family's optimum (polynomial: (sigma, degree) over degrees 1..10, R/fit.R:145-156).  evaluations (nullable, 2) =
 * {objective, gradient} device evaluations. */
int gprc_fit_family(gprc_ctx* ctx, int kernel_id, const double* X, int d, long n, const double* y, double noise,
                    int minors_rule, double* par, int* npar, double* value, long* evaluations);

/* ---- (4) GPC: Laplace-approximation Newton loop -- GPC$initialize, R/GPCclass.R:73-103 ------------------ */
/* guard != 0 applies the reference's divergence rule R/GPCclass.R:90 literally (SURVEY.md A.2); when it fires
 * the return value is 0, *status = 1 and no model is created.  objective_trace receives min(iters, trace_cap)
 * values.  sum_diagL / sum_log_diagL are over the final factor of B = I + W^1/2 K W^1/2 (A.3).
 * status: 0 converged, 1 guard fired ("Apparently does not converge."), 2 not positive definite. */
int gprc_gpc_fit(gprc_ctx* ctx, const gprc_kernel* k, const double* X, int d, long n, const double* y, double eps,
                 int guard, int max_iter, gprc_gpc** out, int* iters, double* objective_trace, int trace_cap,
                 double* sum_diagL, double* sum_log_diagL, int* status);
int gprc_gpc_fit_precomputed(gprc_ctx* ctx, const double* K, long n, const double* y, double eps, int guard,
                             int max_iter, gprc_gpc** out, int* iters, double* objective_trace, int trace_cap,
                             double* sum_diagL, double* sum_log_diagL, int* status);
/* fs_bar and Vfs of GPC$predict_class, R/GPCclass.R:110-115 (the quadrature of :116-117 stays on the host). */
int gprc_gpc_predict_latent(gprc_gpc* g, const double* Xs, long m, double* fs_bar, double* Vfs);
int gprc_gpc_predict_latent_precomputed(gprc_gpc* g, const double* Ks, const double* kss, long m, double* fs_bar,
                                        double* Vfs);
/* GPC$predict_class complete, R/GPCclass.R:108-118: latent mean/variance and, per test point, the reference's
 * integrate(sigmoid(z) * dnorm(z, fs_bar, sd = Vfs), -Inf, Inf) evaluated on the device by a statement-by-statement
 * port of QUADPACK dqagi (the routine behind R's integrate(); same tolerances .Machine$double.eps^0.25, 100
 * subdivisions, same silent ~0 on peaks narrower than its sampling grid).  ier[i] (nullable) is QUADPACK's error
 * code per point (R stops when it is > 0); -1 flags a non-finite integrand (Vfs <= 0 or NaN). */
int gprc_gpc_predict_class(gprc_gpc* g, const double* Xs, long m, double* prob, int* ier);
/* the quadrature alone: out[i] = integral of sigmoid(z) N(z | mean[i], sd[i]) dz  (host arrays, computed on the GPU) */
int gprc_logistic_gaussian(gprc_ctx* ctx, const double* mean, const double* sd, long m, double* out, int* ier);
int gprc_gpc_get(gprc_gpc* g, int what, double* host);
long gprc_gpc_n(const gprc_gpc* g);
int gprc_gpc_dim(const gprc_gpc* g); /* as gprc_gpr_dim */
void gprc_gpc_free(gprc_gpc* g);

/* ---- posterior sampling helper (SURVEY.md 8f-2) ------------------------------------------------------------- */
/* multivariate_normal(n, mean, covariance), R/GPRclass.R:360-370: out (m x ns) = mean + t(chol(covariance)) %*% Z with
 * Z (m x ns) standard normals drawn by the caller (R's rnorm stream stays R's).  info > 0: chol() failed and nothing is
 * written -- the host then runs the reference's eigen fallback (R/GPRclass.R:363-368). */
int gprc_mvn_sample(gprc_ctx* ctx, const double* mean, const double* cov, long m, const double* Z, long ns, double* out,
                    long* info);

/* ---- multi-GPU: Cholesky + solve for n beyond one GPU (SURVEY.md 8e, BASELINE config 5) ------------------------ */
/* One process per GPU.  K + noise I is distributed by outer panels of 512 columns (panel p on rank p mod world) and
 * factored right-looking with panel broadcasts over NCCL (bound at run time with dlopen).  Replaces, collectively,
 * the same reference lines as gprc_gpr_fit (R/GPRclass.R:138-153) when K does not fit one device. */
typedef struct gprc_dist gprc_dist;
/* rank 0 creates the 128-byte NCCL unique id; the caller ships it to the other ranks (torch.distributed, MPI, ...) */
int gprc_dist_unique_id(char* id128, const char* nccl_path /* nullable: libnccl.so.2 */);
int gprc_dist_create(gprc_ctx* ctx, const char* id128, int rank, int world, const char* nccl_path, gprc_dist** out);
void gprc_dist_free(gprc_dist* d);
/* Per-panel timeline of the distributed factorisation (evidence for the layout choice, SURVEY.md 8e row 4): when switched
   on, the next gprc_dist_gpr_fit* records CUDA events around, per 512-column panel p, [0,1] the look-ahead update +
   factorisation on its owner, [2,3] its ncclBroadcast, [4,5] the trailing update with it; gprc_dist_get_timeline returns
   npan x 6 milliseconds since the start of the factorisation on this rank (NaN where this rank recorded nothing). */
int gprc_dist_set_timeline(gprc_dist* D, int on);
int gprc_dist_get_timeline(gprc_dist* D, double* ms, int cap_panels, int* npan);
/* Collective.  X (d x n), y: HOST, identical on every rank.  alpha (n, host, nullable) and logp are returned on every
 * rank.  phase_ms (nullable, 4): build, factor, solve, total -- CUDA events on this rank's stream. */
int gprc_dist_gpr_fit(gprc_dist* d, const gprc_kernel* k, const double* X, int dim, long n, const double* y,
                      double noise, double* logp, double* alpha, long* info, double* phase_ms);

/* Same collective factorisation, but every rank also assembles the complete factor from the panels it receives anyway
 * and gets an ordinary model handle: train on N GPUs, then gprc_gpr_predict on each rank's shard of test points. */
int gprc_dist_gpr_fit_replicated(gprc_dist* d, const gprc_kernel* k, const double* X, int dim, long n, const double* y,
                                 double noise, gprc_gpr** out, double* logp, long* info, double* phase_ms);

/* ---- raw device primitives (tests, roofline microbenchmarks) ---------------------------------------------- */
/* In-place blocked Cholesky of the lower triangle of the n x n column-major device matrix dA (ld >= n, both
 * multiples of 128).  dinv: device workspace (n/128) * 128*128 doubles receiving the inverted diagonal blocks. */
int gprc_dev_potrf(gprc_ctx* ctx, double* dA, long n, long ld, double* dinv, long* info);
/* C (M x N) = beta*C + alpha * A (M x K, col-major) * op(B); transb = 1: B is N x K col-major (C += A B^T),
 * transb = 0: B is K x N col-major.  M, N multiples of 128, K multiple of 16. */
int gprc_dev_dgemm(gprc_ctx* ctx, int transb, long M, long N, long K, double alpha, const double* dA, long lda,
                   const double* dB, long ldb, double beta, double* dC, long ldc);
/* Measured INT8 tensor-pipe rate -- the roofline denominator of predict path 4 (bench.py `roofline.peak`): a pure stream
   of 128 x 256 x 32 tcgen05.mma kind::i8 on every SM for about `seconds` (milliseconds: burst; seconds: under the power
   cap).  tops = 1e-12 x INT8 operations per second (2 per multiply-add); clk_per_mma from CTA 0's clock counter (math
   floor: 128).  No reference counterpart (measurement only). */
int gprc_dev_int8_rate(gprc_ctx* ctx, double seconds, double* tops, double* clk_per_mma);
/* W = L^-1 for a lower-triangular n x n device matrix whose diagonal blocks' inverses are in dinv. dscratch: n x n. */
int gprc_dev_trtri(gprc_ctx* ctx, const double* dL, long n, long ld, const double* dinv, double* dW,
                   double* dscratch);

#ifdef __cplusplus
}
#endif
#endif /* GPRC_H */
