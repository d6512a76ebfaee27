/*
 * hbegp.h — C ABI of libhbegp.so: the B200-native Gaussian-process surrogate hot path of hbetune.
 *
 * The reference (latk/hbetune.rs) has no FFI or plugin ABI; its seam is a pair of Rust traits
 * (src/core/surrogate_model.rs:6-65).  This header is the boundary a Rust `impl Estimator<A>` /
 * `impl SurrogateModel<A>` binds to (INTEGRATION.md shows the `extern "C"` block).  Each entry
 * point names the reference code it replaces.
 *
 * Conventions
 *  - All pointers are HOST pointers unless the name ends in `_device`; arrays are row-major and
 *    caller-owned.  `void*` data arrays hold f64 (HBEGP_F64) or f32 (HBEGP_F32, `--use-32`,
 *    src/bin/hbetune/main.rs:240-244) elements; hyper-parameters are always f64
 *    (src/gpr/matern_kernel.rs:12-15).
 *  - theta layout everywhere: [ln noise, ln c, ln l_1 .. ln l_d], p = d + 2 (src/gpr/fit.rs:140-144).
 *  - Every function returns an int status: 0 ok, < 0 error (never aborts the process).  Per-evaluation
 *    "kernel matrix not positive definite" (src/gpr/lml.rs:47-50) is reported in a status array as
 *    HBEGP_NOT_PD, not as an error.
 *  - A context is bound to one GPU and is used from one thread at a time (the reference's model calls
 *    all happen on the minimizer's thread, src/gpr/fit.rs:92 uses a RefCell).
 *  - There is no CPU fallback: without a CUDA device every compute entry point fails with HBEGP_ERR_CUDA.
 */
#ifndef HBEGP_H
#define HBEGP_H

#ifdef __cplusplus
extern "C" {
#endif

#define HBEGP_F64 0
#define HBEGP_F32 1

#define HBEGP_OK 0
#define HBEGP_NOT_PD 1            /* per-evaluation status: Cholesky failed (lml.rs:47-50) */
#define HBEGP_ERR_INVALID (-1)    /* bad argument / call order */
#define HBEGP_ERR_CUDA (-2)       /* CUDA runtime failure (incl. no device) */
#define HBEGP_ERR_NOMEM (-3)      /* device memory exhausted */
#define HBEGP_ERR_UNSUPPORTED (-4)/* e.g. nu other than 0.5 / 1.5 / 2.5 / +INFINITY (NaN and -INFINITY included) */
#define HBEGP_ERR_NO_CAPTURE (-5) /* fit: no evaluation succeeded (fit.rs:161 unwrap panic) */

typedef struct hbegp_ctx hbegp_ctx;
typedef struct hbegp_model hbegp_model;

/* ---- library ---------------------------------------------------------------------------------- */
const char* hbegp_version(void);
/* Last error message of this thread (valid until the next failing call on the thread). */
const char* hbegp_last_error(void);

/* ---- context ---------------------------------------------------------------------------------- */
/* `stream` is a cudaStream_t (NULL: the library creates its own); all work of the context is ordered
 * after / before work on that stream, so CUDA events recorded on it bracket the library's kernels. */
int hbegp_ctx_create(int device, int dtype, void* stream, hbegp_ctx** out);
int hbegp_ctx_destroy(hbegp_ctx* ctx);
/* Caps the device memory the context may use for batched evaluation workspaces (0: default 70% of free). */
int hbegp_ctx_set_workspace_limit(hbegp_ctx* ctx, unsigned long long bytes);
/* Retained-model policy.  The reference's minimizer keeps the model of EVERY generation (all_models,
 * src/core/minimize.rs:331, :407) although only the newest one is asked anything; an n x n factor per generation would
 * exhaust the device (50 generations at n = 4096: 6.7 GB; two models at n = 16384 fill a GPU).  Only the `max_resident`
 * most recently created / used models of a context keep their factor on the device (default 4; <= 0: all).  An older
 * model stays valid and cheap (X^T / l, alpha and the parameters remain: O(n d)); its next variance prediction
 * refactorises (one n^3 / 3 evaluation) and makes it resident again. */
int hbegp_ctx_set_resident_models(hbegp_ctx* ctx, int max_resident);
int hbegp_ctx_model_stats(hbegp_ctx* ctx, int* live, int* resident, long long* evictions, long long* rebuilds);
/* Number of kernels this context has launched so far (bench.py reports it as gpu_launches). */
long long hbegp_ctx_launch_count(hbegp_ctx* ctx);

/* Training data of the current fit: X (n x d), y (n).  Replaces the x_train / y_train arguments of
 * LmlWithGradient::of (src/gpr/lml.rs:16-27) and FittedKernel::new (src/gpr/fit.rs:18-31).
 * Limit of this implementation (the reference has none beyond host memory): n <= 46000 (one n x n factor and its inverse
 * per evaluation must fit one GPU) -> HBEGP_ERR_INVALID.  The feature count is not limited in practice (<= 65536): the
 * kernels stage features in chunks of 64. */
int hbegp_set_data(hbegp_ctx* ctx, long n, int d, const void* x, const void* y);
int hbegp_set_data_device(hbegp_ctx* ctx, long n, int d, const void* x_device, const void* y_device);

/* ---- LML + gradient, batched over thetas ------------------------------------------------------- */
/* Every `nu` argument selects the correlation M of the kernel c M + noise I: nu = 0.5, 1.5, 2.5 the Matern orders of
 * src/gpr/matern_kernel.rs:65-80 (of r = sqrt(s)), nu = +INFINITY the squared exponential (RBF; sklearn's RBF, which
 * sklearn's Matern(nu=inf) also is) M = exp(-0.5 s), the product by 0.5 exact and no square root taken.  In both,
 * s = sum_k (x_ik / l_k - x_jk / l_k)^2 (division first, features summed left to right), and K_ii = c + noise.  The
 * RBF's theta gradient is dK/d ln c = c M and dK/d ln l_k = c M (x_ik - x_jk)^2 / l_k^2 (sklearn's anisotropic RBF).  A
 * model keeps its nu through extend, rebuild, replicas, predictions, gradients and the acquisition searches.
 *
 * B evaluations of src/gpr/lml.rs:29-79 for Product<ConstantKernel, Matern(nu)> + noise, one per theta
 * row.  `lo`/`hi` (natural units, length p, may be NULL) clamp exp(theta[1..]) like with_clamped_theta
 * (src/gpr/fit.rs:95; noise is not clamped).  Outputs: lml[B]; grad[B*p] (may be NULL: value only);
 * status[B] in {HBEGP_OK, HBEGP_NOT_PD}; on NOT_PD lml = -inf and grad = 0 (fit.rs:103-113 returns +inf
 * for -lml with a zero gradient). */
int hbegp_lml_grad_batch(hbegp_ctx* ctx, double nu, int B, const double* theta, const double* lo,
                         const double* hi, double* lml, double* grad, int* status);

/* ---- restart loop ------------------------------------------------------------------------------ */
typedef struct hbegp_run_result {
    double best_lml;      /* largest LML seen at ANY evaluation of this run (fit.rs:115-125)        */
    long long best_eval;  /* index (0-based, within the run) of the first evaluation that reached it */
    long long n_evals;    /* evaluations this run performed (<= maxeval)                            */
    double final_f;       /* optimiser's final objective value (= -lml), gradmin.rs:56-59           */
    int status;           /* HBEGP_OK, or HBEGP_NOT_PD if no evaluation of the run succeeded        */
    int reserved;
} hbegp_run_result;

/* Runs `n_runs` independent bounded L-BFGS optimisations of -LML (src/util/gradmin.rs:35-60: box bounds,
 * maxeval evaluations) from the given start points, all runs advancing in lockstep so that each
 * optimiser step is ONE batched GPU evaluation.  This is the shardable unit of the restart loop
 * (src/util/gradmin.rs:19-30): rank r of G passes the runs it owns.  bounds_lo/bounds_hi: natural
 * units, length p (theta bounds are their logs, fit.rs:140 / kernel.bounds()).
 * Outputs per run: results[n_runs], best_theta[n_runs*p] (the theta of the best evaluation). */
int hbegp_fit_runs(hbegp_ctx* ctx, double nu, int n_runs, const double* starts, const double* bounds_lo,
                   const double* bounds_hi, int maxeval, hbegp_run_result* results, double* best_theta);

/* The same loop across `world` processes (one per GPU, each with its own context holding the same data): every rank
 * passes identical arguments plus its rank.  Each round the live runs are dealt out round-robin, every rank
 * evaluates its share and `allreduce` (called once per round on every rank) must sum `count` doubles element-wise
 * over all ranks in place -- e.g. ncclAllReduce / torch.distributed.all_reduce(SUM).  All ranks return the records of
 * ALL runs, bit-identical to the single-process loop (each value is summed with zeros only).  The work stays
 * balanced while runs finish at different times (a static split of the runs leaves GPUs idle in the tail).
 * With allreduce = NULL the exchange runs inside the library on the communicator of hbegp_comm_init (ncclAllReduce on
 * the device-resident round record).  If the exchange fails on one rank that rank returns an error while its peers are
 * still inside the collective: the caller must tear the job down (NCCL's own failure mode; there is no recovery). */
typedef int (*hbegp_allreduce_fn)(void* user, double* values, long count); /* 0 on success */
int hbegp_fit_runs_sharded(hbegp_ctx* ctx, double nu, int n_runs, const double* starts, const double* bounds_lo,
                           const double* bounds_hi, int maxeval, int rank, int world, hbegp_allreduce_fn allreduce,
                           void* allreduce_user, hbegp_run_result* results, double* best_theta);

/* ---- exchange between GPUs inside the library: NCCL over NVLink on device buffers ----------------------------
 * Multi-process mode (one process and one context per GPU; the launcher only has to hand every rank the same 128-byte
 * id, e.g. over MPI / torch.distributed / a file): rank 0 calls hbegp_comm_unique_id, every rank hbegp_comm_init.
 * Afterwards hbegp_fit_runs_sharded may be called with allreduce = NULL (the per-round record is packed on the device
 * and summed with ncclAllReduce), and the two calls below shard a batched evaluation / a prediction with one
 * ncclAllGather of the device-resident results and one device-to-host copy.  libnccl.so.2 is loaded at run time (the
 * copy already in the process if there is one, else $HBEGP_NCCL_LIB, else the system library). */
#define HBEGP_COMM_ID_BYTES 128
int hbegp_comm_unique_id(void* id_out /* HBEGP_COMM_ID_BYTES */);
int hbegp_comm_init(hbegp_ctx* ctx, int world, int rank, const void* id);
/* Any output may be NULL.  collective_ms / n_collectives: device time (CUDA events around the NCCL calls) and count of
 * the collectives this context has issued so far. */
int hbegp_comm_info(hbegp_ctx* ctx, int* rank, int* world, int* nccl_version, double* collective_ms, long long* n_collectives);
/* hbegp_lml_grad_batch over the ranks of the communicator: every rank passes the same B thetas and receives all B
 * results; rank r evaluates thetas r, r + world, ...  (src/util/gradmin.rs:19-30: the restarts are independent). */
int hbegp_lml_grad_batch_sharded(hbegp_ctx* ctx, double nu, int B, const double* theta, const double* lo, const double* hi,
                                 double* lml, double* grad, int* status);
/* hbegp_predict over the ranks of the model's context: every rank passes the same m candidate rows and receives all m
 * means / variances; rank r predicts the r-th contiguous block of ceil(m / world) rows.  (The list of
 * hbegp_predict_warn_values is not exchanged, only the count.) */
int hbegp_predict_sharded(hbegp_model* model, long m, const void* xs, void* mean, void* var, long* n_below_warn);

/* Single-process mode -- what a drop-in for the reference needs, which is one process (src/bin/hbetune/main.rs:255-355):
 * one handle over n_gpus devices (devices = NULL: 0 .. n_gpus - 1).  Thetas of a batch / live runs of a fit round are
 * dealt round-robin to the GPUs and evaluated concurrently; candidate rows go out in contiguous blocks; training data
 * and the fitted model are replicated with ncclBroadcast.  Results are bit-identical to one GPU. */
typedef struct hbegp_multi hbegp_multi;
typedef struct hbegp_multi_model hbegp_multi_model;
int hbegp_multi_create(int n_gpus, const int* devices, int dtype, hbegp_multi** out);
int hbegp_multi_destroy(hbegp_multi* multi);
int hbegp_multi_n_gpus(const hbegp_multi* multi);
hbegp_ctx* hbegp_multi_ctx(hbegp_multi* multi, int i); /* the context of GPU i (owned by the handle) */
int hbegp_multi_set_data(hbegp_multi* multi, long n, int d, const void* x, const void* y);
int hbegp_multi_lml_grad_batch(hbegp_multi* multi, double nu, int B, const double* theta, const double* lo, const double* hi,
                               double* lml, double* grad, int* status);
int hbegp_multi_fit_runs(hbegp_multi* multi, double nu, int n_runs, const double* starts, const double* bounds_lo,
                         const double* bounds_hi, int maxeval, hbegp_run_result* results, double* best_theta);
/* One evaluation on GPU 0 (as hbegp_model_create), then the model travels to the other GPUs over NVLink. */
int hbegp_multi_model_create(hbegp_multi* multi, double nu, const double* theta, const double* lo, const double* hi,
                             hbegp_multi_model** out, double* lml, void* alpha_out, void* kinv_out);
int hbegp_multi_model_destroy(hbegp_multi_model* model);
hbegp_model* hbegp_multi_model_replica(hbegp_multi_model* model, int i); /* GPU i's replica (owned by the multi model) */
int hbegp_multi_predict(hbegp_multi_model* model, long m, const void* xs, void* mean, void* var, long* n_below_warn);

/* The loop over a caller-supplied batched objective instead of the GPU (the restart loop of gradmin.rs:7-33 for any
 * function): objective(user, B, p, theta[B*p], lml[B], grad[B*p], status[B]) returns 0 on success; status[b] != 0
 * marks a failed evaluation (treated like a non-PD matrix, fit.rs:103-113).  rank / world / allreduce as above
 * (0, 1, NULL for one process). */
typedef int (*hbegp_batch_objective_fn)(void* user, int batch, int p, const double* theta, double* lml, double* grad,
                                        int* status);
int hbegp_fit_runs_with(hbegp_batch_objective_fn objective, void* objective_user, int p, int n_runs, const double* starts,
                        const double* bounds_lo, const double* bounds_hi, int maxeval, int rank, int world,
                        hbegp_allreduce_fn allreduce, void* allreduce_user, hbegp_run_result* results, double* best_theta);

/* ---- batched objective for a caller-owned optimiser ------------------------------------------------------
 * The route that keeps the reference's optimiser -- NLopt L-BFGS, one instance per restart, src/util/gradmin.rs:35-60 --
 * in the loop while still evaluating all restarts in one batched GPU call per step.  The host starts one thread per
 * run (start points drawn up front in reference order, gradmin.rs:21-24); each thread runs its optimiser, whose
 * objective closure (fit.rs:93-134) calls hbegp_batcher_eval.  The call blocks until every run that is still live
 * has submitted a theta; the last arrival evaluates the round with one hbegp_lml_grad_batch (rows ordered by run
 * index) and wakes the others.  A thread whose optimiser has returned calls hbegp_batcher_leave so that the
 * remaining runs stop waiting for it.  Results per evaluation are those of hbegp_lml_grad_batch (bit-identical whatever
 * the batch composition), so each run's trajectory is exactly the one its optimiser would take alone.  The batcher
 * records the capture rule of fit.rs:115-125 per run (hbegp_batcher_results), to be resolved across runs with
 * hbegp_pick_best_run.  One thread per run; the context must not be used by anyone else meanwhile. */
typedef struct hbegp_batcher hbegp_batcher;
int hbegp_batcher_create(hbegp_ctx* ctx, double nu, int n_runs, const double* bounds_lo, const double* bounds_hi,
                         hbegp_batcher** out);
/* status (may be NULL): HBEGP_OK or HBEGP_NOT_PD (then *lml = -inf and grad = 0, fit.rs:103-113). */
int hbegp_batcher_eval(hbegp_batcher* batcher, int run, const double* theta, double* lml, double* grad, int* status);
int hbegp_batcher_leave(hbegp_batcher* batcher, int run, double final_f);
/* results[n_runs], best_theta[n_runs * p] as for hbegp_fit_runs; n_rounds = batched GPU evaluations issued. */
int hbegp_batcher_results(hbegp_batcher* batcher, hbegp_run_result* results, double* best_theta, long long* n_rounds);
int hbegp_batcher_destroy(hbegp_batcher* batcher);

/* Deterministic winner pick over runs in reference order (fit.rs:116-117: strict `>`, so the earliest
 * (run, evaluation) wins ties).  Returns the winning run index or -1 if none succeeded. */
int hbegp_pick_best_run(int n_runs, const hbegp_run_result* results);

/* ---- fitted model ------------------------------------------------------------------------------ */
/* One evaluation at `theta` and the prediction pre-computations of src/gpr/fit.rs:155-175 (also the whole
 * of FittedKernel::extend, fit.rs:33-68).  The model keeps X, alpha and the inverse Cholesky factor on
 * the device.  Optional host outputs: lml, alpha_out[n], kinv_out[n*n] (full symmetric K^-1, the
 * reference's `k_inv`).  Returns HBEGP_NOT_PD (and no model) if the kernel matrix is not invertible
 * (the reference panics there, fit.rs:55). */
int hbegp_model_create(hbegp_ctx* ctx, double nu, const double* theta, const double* lo, const double* hi,
                       hbegp_model** out, double* lml, void* alpha_out, void* kinv_out);
/* FittedKernel::extend (src/gpr/fit.rs:33-68) from a prior model: the prior's kernel and noise (as evaluated)
 * on the context's CURRENT data (hbegp_set_data), one evaluation, no optimisation.  Outputs as for
 * hbegp_model_create.  When the prior's training rows are an unchanged prefix of the new data -- the one
 * in-tree call site appends the validation samples to the evaluation history, minimize.rs:629-644 -- only the
 * added rows are factorised (an O(n^2 k) block append, checked on the device; the result is the same model up to
 * rounding); otherwise this is the full evaluation.  *appended (may be NULL) reports which: 1 append, 0 full.
  * The append keeps the first floor(n_prior / 128) * 128 rows of the prior factor (at least 128), so that appended blocks stay aligned with
 * the 128-wide GEMM tiles.  The prior stays valid and must belong to `ctx`. */
int hbegp_model_extend(hbegp_ctx* ctx, hbegp_model* prior, hbegp_model** out, double* lml, void* alpha_out,
                       void* kinv_out, int* appended);
int hbegp_model_destroy(hbegp_model* model);
long hbegp_model_n(const hbegp_model* model);
int hbegp_model_dim(const hbegp_model* model);

/* src/gpr/predict.rs:7-52: mean[m] = k* alpha; if var != NULL: var[m] = c + 1e-5 - k* K^-1 k*^T, values
 * below 0 clamped to 0; *n_below_warn (may be NULL) counts values < -sqrt(1e-5) BEFORE clamping, i.e. the
 * entries the reference lists in its stderr warning (predict.rs:39-46). */
int hbegp_predict(hbegp_model* model, long m, const void* xs, void* mean, void* var, long* n_below_warn);
/* The values the reference lists in its warning ("Variances below 0 were predicted and will be corrected: ...",
 * src/gpr/predict.rs:39-46): the pre-clamp variances < -sqrt(1e-5) of the LAST hbegp_predict / hbegp_predict_mean_ei /
 * hbegp_predict_confidence_bound call on this model, in row order, with their row indices (rows_out may be NULL).
 * Returns how many were written (<= cap; the library keeps at most 4096 per call, n_below_warn has the full count). */
int hbegp_predict_warn_values(const hbegp_model* model, int cap, double* values_out, long* rows_out);
/* Same with device-resident candidates and outputs (asynchronous on the context's stream). */
int hbegp_predict_device(hbegp_model* model, long m, const void* xs_device, void* mean_device,
                         void* var_device, long* n_below_warn_device);

/* ---- batched acquisition epilogues on the device (SURVEY section 8 "next" rows f1 / f2) ------------- */
/* Forward declaration of the y-normalisation record defined below. */
struct hbegp_ynorm;
/* predict_mean_ei_a (src/core/gpr.rs:179-212) for m candidates in one call: mean_out[m] = de-normalised mean,
 * ei_out[m] = expected improvement (acquisition.rs:141-171, evaluated in f64) against fmin given in NATURAL
 * units (it is projected into normalised space in A first, gpr.rs:192-196).  best_index (may be NULL) receives
 * find_best_candidate_by_ei's argmax (acquisition.rs:177-202: the LAST maximum wins).  Any output may be NULL.
 * ei_out[i] is NaN exactly where hbegp_expected_improvement is: where the mean, sqrt(variance) or the projected fmin
 * is NaN or infinite (the log projection of fmin <= expected, say), whatever the variance.  NaN rows never win, so
 * best_index is -1 when every row is NaN; a caller should check it before using it. */
int hbegp_predict_mean_ei(hbegp_model* model, const struct hbegp_ynorm* yn, long m, const void* xs, double fmin,
                          void* mean_out, void* ei_out, long* best_index, long* n_below_warn);
/* predict_confidence_bound (src/core/gpr.rs:94-112) for m points: out[m] = location_from(mean + sqrt(var) * cb);
 * best_index (may be NULL) = find_best_individual_by_confidence_bound's argmin (minimize.rs:680-714: strict `<`,
 * the FIRST minimum wins). */
int hbegp_predict_confidence_bound(hbegp_model* model, const struct hbegp_ynorm* yn, long m, const void* xs,
                                   double cb, void* out, long* best_index, long* n_below_warn);

/* ---- gradients in the candidate ----------------------------------------------------------------------
 * x is in the caller's units, as the row-major candidates of hbegp_predict.  With x~_k = x_k / l_k, X~_jk = X_jk / l_k
 * and s_j = sum_k (x~_k - X~_jk)^2, d k*_j / d x_k = -c dk_factor(s_j) (x~_k - X~_jk) / l_k, dk_factor = -2 dM/ds, so
 *   dmean = sum_j alpha_j grad k*_j,   dvar = -2 sum_j v_j grad k*_j,  v = K^-1 k*  (normalised units).
 * Definitions where the functions are not smooth:
 *   - a term with s_j = 0 (the candidate on a training point) contributes 0, for every nu (for nu = 1/2 the
 *     derivative does not exist there; the reference's non-finite -> 0 rule gives 0; for the other orders and the
 *     RBF, whose dk_factor = M, 0 is the derivative);
 *   - where the variance is clamped to 0 (its pre-clamp value is < 0, or exactly 0), dvar = 0;
 *   - d sqrt(var) = dvar / (2 sqrt(var)) where sqrt(var) > 0, else 0;
 *   - EI (f64, normalised units): -Phi(z) dmean + phi(z) d sqrt(var); in the std-zero branch -dmean where
 *     mean < fmin and 0 otherwise; NaN in every component where EI is NaN;
 *   - de-normalisation: amplitude * dy (linear projection), amplitude * exp(y * amplitude) * dy (logarithmic), with
 *     y = mean for the mean and y = mean + cb sqrt(var) (dy = dmean + cb d sqrt(var)) for the confidence bound.
 * The values returned equal those of hbegp_predict / _mean_ei / _confidence_bound bit for bit, the calls count as the
 * last prediction for hbegp_predict_warn_values, and an evicted model is rebuilt first.  A candidate's gradients do not
 * depend on the other rows predicted with it, among m > 64 rows; the m <= 64 path agrees with it to rounding. */
/* Gradients of hbegp_predict's outputs: dmean[m*d] (required) and dvar[m*d] (may be NULL), row-major, in the data
 * type; mean[m] (required) and var[m] (may be NULL) as hbegp_predict. */
int hbegp_predict_grad(hbegp_model* model, long m, const void* xs, void* mean, void* var, void* dmean, void* dvar,
                       long* n_below_warn);
/* hbegp_predict_mean_ei plus dmean_out[m*d] (de-normalised mean) and dei_out[m*d] (EI, normalised units).  Any output
 * may be NULL. */
int hbegp_predict_mean_ei_grad(hbegp_model* model, const struct hbegp_ynorm* yn, long m, const void* xs, double fmin,
                               void* mean_out, void* ei_out, void* dmean_out, void* dei_out, long* n_below_warn);
/* hbegp_predict_confidence_bound plus dout[m*d].  Either output may be NULL. */
int hbegp_predict_confidence_bound_grad(hbegp_model* model, const struct hbegp_ynorm* yn, long m, const void* xs,
                                        double cb, void* out, void* dout, long* n_below_warn);

/* ---- acquisition search on the device ------------------------------------------------------------
 * S independent bounded L-BFGS searches over the box lo <= x <= hi (lo, hi: f64, length d), one per start point
 * (starts[S*d], data type), advancing in lockstep: hbegp_acquire_ei maximises EI, hbegp_acquire_confidence_bound
 * minimises the de-normalised bound.  An alternative to the reference's BOBYQA searches (SearchingAcquisition::acquire,
 * suggest_optimum), not a restatement of them: NLopt is not available, so the chosen points are not hbetune's.
 *  - The optimiser is BoundedLbfgs (the fit's optimiser, memory 10) with the tolerances hbegp_lbfgs_set_tolerances has
 *    set at call time.  Its objective is -EI with gradient -dei (EI) or the bound with its gradient: the values and
 *    gradients of hbegp_predict_mean_ei_grad / hbegp_predict_confidence_bound_grad, widened to f64.  A non-finite
 *    value is a failed trial, as a non-PD matrix is in the fit; a start whose first value is not finite ends at once
 *    (the log projection with fmin <= expected, a mean that is not finite).
 *  - Every round evaluates all S rows, in start order; a finished start's row keeps its last trial point and its result
 *    is ignored.  The batch therefore has the same shape, and takes the same prediction path, in every round: a start's
 *    bits do not depend on when the others finish.  Each start's steps equal BoundedLbfgs of lbfgs.h bit for bit.
 *    Starts outside the box are clamped.  f32 models: the optimiser works in f64; the point evaluated is the f64 trial
 *    rounded to float.
 *  - Each start keeps the best point it evaluated (the first finite value, then only a strictly better one):
 *    x_out[S*d] holds it as evaluated, in the data type (the clamped start if there is none), and results[S] its record.
 *    mean_out[S] (EI only, may be NULL) holds the de-normalised mean there (NaN if there is none).
 *  - best_index: the last maximum of the EI (find_best_candidate_by_ei, max_by) or the first minimum of the bound
 *    (minimize.rs:680-714), among the starts with status HBEGP_OK; -1 if there is none.  n_rounds: rounds in which at least
 *    one start was live.
 *  - n_starts = 0 is a no-op.  maxeval = 0 evaluates nothing: x_out = the clamped starts, every status HBEGP_NOT_PD,
 *    best_index -1, n_rounds 0.  HBEGP_ERR_INVALID: a NULL required pointer (all but mean_out), n_starts < 0,
 *    maxeval < 0, a non-finite start or bound, lo > hi.
 *  - All rounds run on the device: a round is predict -> acquisition epilogue -> gradients -> one optimiser step per
 *    start, and the host looks at the count of live starts only every few rounds (a CUDA graph of those rounds).  The
 *    starts go up and the results come back once per call.
 *  - An evicted model is rebuilt first.  The search is not a prediction for hbegp_predict_warn_values: the list of the
 *    last prediction call stays as it was.  One GPU (on a multi model, pass a replica). */
typedef struct hbegp_acq_result {
    double best_value;   /* EI: largest EI seen (normalised units, as ei_out of hbegp_predict_mean_ei);
                            bound: smallest bound seen (de-normalised, as out of hbegp_predict_confidence_bound); NaN if none */
    long long best_eval; /* 0-based evaluation of this start that first reached it; -1 if no value was finite */
    long long n_evals;   /* evaluations this start performed (<= maxeval) */
    int status;          /* HBEGP_OK, or HBEGP_NOT_PD if no evaluation of this start had a finite value */
    int reserved;
} hbegp_acq_result;
int hbegp_acquire_ei(hbegp_model* model, const struct hbegp_ynorm* yn, double fmin, long n_starts, const void* starts,
                     const double* lo, const double* hi, int maxeval, void* x_out, void* mean_out, hbegp_acq_result* results,
                     long* best_index, long long* n_rounds);
int hbegp_acquire_confidence_bound(hbegp_model* model, const struct hbegp_ynorm* yn, double cb, long n_starts,
                                   const void* starts, const double* lo, const double* hi, int maxeval, void* x_out,
                                   hbegp_acq_result* results, long* best_index, long long* n_rounds);

/* ---- host-side pieces of the reference interface (no GPU needed) -------------------------------- */
/* Bounded L-BFGS used by hbegp_fit_runs, exposed with a callback objective
 * (objective(x, grad_out, user) -> f), mirroring minimize_by_gradient (src/util/gradmin.rs:35-60).
 * x[n] is updated in place; returns the number of evaluations (>= 0) or an error. */
typedef double (*hbegp_objective_fn)(const double* x, double* grad_out, void* user);
int hbegp_minimize_by_gradient(hbegp_objective_fn objective, void* user, int n, double* x,
                               const double* lo, const double* hi, int maxeval, double* f_out);

/* Stopping tolerances of the bounded L-BFGS for every run started afterwards (process-wide).  Defaults ftol = 1e-11
 * (two consecutive accepted steps with a relative decrease below it end a run) and gtol = 1e-8 (largest free gradient
 * component); a value <= 0 switches that rule off, leaving maxeval as the only stop like the reference's NLopt
 * configuration (src/util/gradmin.rs:52-54). */
int hbegp_lbfgs_set_tolerances(double ftol, double gtol);

/* Xoshiro256** restart-start sampler: src/core/random.rs + src/util/gradmin.rs:21-24.  `state[4]` is the
 * generator state (updated).  hbegp_rng_seed = RNG::new_with_seed, hbegp_rng_fork = fork_random_state,
 * hbegp_rng_uniform = rng.uniform(lo..=hi). */
void hbegp_rng_seed(unsigned long long seed, unsigned long long state[4]);
void hbegp_rng_fork(unsigned long long state[4], unsigned long long child[4]);
double hbegp_rng_uniform(unsigned long long state[4], double lo, double hi);

/* ---- adapter pieces around src/gpr (host-side, no GPU) --------------------------------------------- */
#define HBEGP_PROJ_LINEAR 0
#define HBEGP_PROJ_LOG 1
/* YNormalize (src/core/ynormalize.rs:7-12): amplitude / expected hold values of the data type `dtype`. */
typedef struct hbegp_ynorm {
    double amplitude;
    double expected;
    int projection;
    int dtype;
} hbegp_ynorm;
/* YNormalize::new_project_into_normalized (ynormalize.rs:162-195); known_optimum may be NULL. */
int hbegp_ynorm_fit(int dtype, int projection, long n, const void* y, const double* known_optimum,
                    void* y_normalized_out, hbegp_ynorm* out);
/* op 0: project_into_normalized(a)            (ynormalize.rs:197-210)
 * op 1: project_location_from_normalized(a)   (:215-225)
 * op 2: project_mean_from_normalized(a = mean, b = variance)   (:227-247)
 * op 3: project_std_from_normalized(a = mean, b = variance)    (:249-267)
 * op 4: project_cv_from_normalized(a = mean, b = variance)     (:269-288) */
int hbegp_ynorm_apply(const hbegp_ynorm* yn, int op, long n, const void* a, const void* b, void* out);
/* estimate_amplitude (src/core/gpr.rs:429-450): out = {start, lo, hi}; bounds (2 values) may be NULL. */
int hbegp_estimate_amplitude(int dtype, long n, const void* y, const double* bounds, double out[3]);
/* expected_improvement (src/core/acquisition.rs:141-171), f64; NaN where the reference would panic. */
double hbegp_expected_improvement(double mean, double std, double fmin);
/* The per-row loop of predict_mean_ei_a (src/core/gpr.rs:198-208): ei[i] = EI(mean[i], sqrt(var[i]), fmin). */
int hbegp_expected_improvement_a(int dtype, long m, const void* mean, const void* var, double fmin, void* ei_out);
/* statrs Normal::inverse_cdf as used for the quartiles of predict_statistics (src/core/gpr.rs:140-166). */
double hbegp_normal_inverse_cdf(double p, double mean, double std);

/* ---- trait Kernel, standalone (src/gpr/kernel.rs:8-43) -------------------------------------------- */
/* For Product<ConstantKernel, Matern(nu)> with theta = [ln c, ln l_1 .. ln l_d] (kernel.theta(), product_kernel.rs:80-85;
 * no noise term, no clamping).  A plain Matern kernel (the reference's golden vectors matern_kernel.rs:189-253) is the
 * case ln c = 0.  The context supplies device, data type and stream; its training data is not touched.
 *   hbegp_kernel_matrix:      Kernel::kernel(x1 (n1 x d), x2 (n2 x d)) -> k_out (n1 x n2)   (kernel.rs:10-14), computed by the
 *                             production cross-kernel code (the k* tiles of predict);
 *   hbegp_kernel_theta_grad:  Kernel::theta_grad(x (n x d)) -> k_out (n x n), grad_out (n x n x (d + 1)), slice 0 =
 *                             d/d ln c, slices 1..d = d/d ln l_k (kernel.rs:16-21, product_kernel.rs:40-70); either may be NULL;
 *   hbegp_kernel_diag:        Kernel::diag(x) -> diag_out (n) = c (kernel.rs:23-24); host-only. */
int hbegp_kernel_matrix(hbegp_ctx* ctx, double nu, int d, const double* theta, long n1, const void* x1, long n2,
                        const void* x2, void* k_out);
int hbegp_kernel_theta_grad(hbegp_ctx* ctx, double nu, int d, const double* theta, long n, const void* x, void* k_out,
                            void* grad_out);
int hbegp_kernel_diag(int dtype, int d, const double* theta, long n, void* diag_out);

/* ---- debugging / parity aids -------------------------------------------------------------------- */
/* Copies out intermediates of ONE evaluation at theta (any pointer may be NULL): k[n*n] lower triangle of
 * K + noise I (upper = 0), w[n*n] = L^-1 (the inverse Cholesky factor; L itself is consumed by the fused
 * factor-and-invert recursion), kinv[n*n] full symmetric. */
int hbegp_debug_factor(hbegp_ctx* ctx, double nu, const double* theta, void* k, void* w, void* kinv,
                       int* status);

/* Overwrites the context's batched evaluation workspaces with NaN bit patterns (test aid: results must not depend on
 * what a previous evaluation or allocation left behind). */
int hbegp_debug_poison(hbegp_ctx* ctx);

/* Times (CUDA events on the context's stream, average of `reps` after one warm-up) a truncated batched
 * evaluation of B thetas: phase 0 = kernel-matrix assembly, 1 = + factor/inverse recursion, 2 = + alpha and
 * K^-1 = W^T W, 3 = the whole LML + gradient evaluation, 5 = only the K^-1 = W^T W product launches (on the W
 * the previous evaluation left).  Used by bench.py for the per-kernel rooflines. */
int hbegp_bench_phase(hbegp_ctx* ctx, double nu, int B, const double* theta, int phase, int reps, float* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* HBEGP_H */
