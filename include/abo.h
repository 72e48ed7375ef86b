/* abo.h — C ABI of libabo_cuda.so: the B200-native GP-surrogate + acquisition hot path of
 * AbstractBayesOpt.jl (reference paths below are relative to the reference repository).
 *
 * There is no FFI in the reference (it is pure Julia on AbstractGPs/KernelFunctions); these
 * entry points are what new `AbstractSurrogate` / `AbstractAcquisition` subtypes bind with
 * `ccall` so that `BOStruct` / `optimize` (src/bayesian_opt.jl:364-449) run unchanged.
 * See INTEGRATION.md for the Julia-side stubs.
 *
 * Conventions
 *  - every function returns an abo_status (0 = OK); all floating data is double;
 *  - host matrices are "point-major": X[i*d + k] is coordinate k of point i — the memory of a
 *    Julia d x n column-major Matrix{Float64} (reduce(hcat, xs)) or a NumPy (n, d) C array;
 *  - GradientGP observations / multi-output results are OUT-MAJOR, idx = out*n + i, exactly
 *    prep_output (src/surrogates/GradientGP.jl:919-922);
 *  - indices returned to the caller are 0-based int64 (the Julia shim adds 1);
 *  - pointers named d_* are DEVICE pointers (on the context's device), everything else is
 *    host memory owned by the caller; the library never keeps a host pointer after return;
 *  - calls are synchronous: results are in the caller's buffers when the function returns.
 *  - no CPU fallback: every entry point fails with ABO_ERR_CUDA when no device is usable.
 */
#ifndef ABO_H
#define ABO_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct abo_ctx abo_ctx;   /* one CUDA device + stream + workspace (+ optional NCCL rank) */
typedef struct abo_gp abo_gp;     /* a conditioned surrogate resident in HBM */

typedef enum {
    ABO_OK = 0,
    ABO_ERR_INVALID = 1,       /* bad argument (ArgumentError) */
    ABO_ERR_DIM = 2,           /* DimensionMismatch (test/test_bayesian_opt.jl:788-817) */
    ABO_ERR_NOT_POSDEF = 3,    /* LinearAlgebra.PosDefException(info) (src/bayesian_opt.jl:126-141) */
    ABO_ERR_CUDA = 4,          /* CUDA runtime failure / no device */
    ABO_ERR_NOT_FITTED = 5,    /* posterior queried before update() */
    ABO_ERR_NCCL = 6,
    ABO_ERR_ALLOC = 7
} abo_status;

/* base kernels: KernelFunctions SqExponentialKernel / Matern52Kernel / Matern72Kernel and the
 * in-repo ApproxMatern / ADMatern kernels (src/surrogates/GradientGP.jl:52-101,133-249,278-327,356-474) */
typedef enum {
    ABO_KERNEL_SE = 0, ABO_KERNEL_MATERN52 = 1, ABO_KERNEL_MATERN72 = 2,
    ABO_KERNEL_APPROX_MATERN52 = 3, ABO_KERNEL_APPROX_MATERN72 = 4,
    ABO_KERNEL_AD_MATERN52 = 5, ABO_KERNEL_AD_MATERN72 = 6
} abo_kernel;

/* acquisition functions (src/acquisition_functions/{ExpectedImprovement,ProbabilityImprovement,
 * UpperConfidenceBound,gradNormUCB}.jl).  params: EI/PI = {xi, best_y}; UCB / GradientNormUCB = {beta}. */
typedef enum { ABO_ACQ_EI = 0, ABO_ACQ_PI = 1, ABO_ACQ_UCB = 2, ABO_ACQ_GRADNORM_UCB = 3 /* abo_acq_eval_multi only */ } abo_acq;

int32_t abo_version(void);
const char* abo_last_error(void);          /* thread-local message of the last failure */

/* ---- context ------------------------------------------------------------------------- */
int32_t abo_ctx_create(int32_t device, abo_ctx** out);
/* Handles of this context that are still alive are orphaned: their device memory is released and only
 * abo_gp_destroy remains valid on them (finalizers of GC'd bindings run in arbitrary order). */
int32_t abo_ctx_destroy(abo_ctx* ctx);
/* release everything the context caches between calls: pooled posterior buffer sets (up to 3 sets / 24 GB kept
 * for the BO loop's per-iteration re-fit), grow-only workspaces, pinned staging memory */
int32_t abo_ctx_trim(abo_ctx* ctx);
int32_t abo_ctx_device(const abo_ctx* ctx, int32_t* device);
/* cudaStream_t the context launches on (for callers that time with events on that stream) */
int32_t abo_ctx_stream(const abo_ctx* ctx, void** stream);
/* number of kernels this context has launched so far (bench.py "gpu_launches") */
int32_t abo_ctx_launch_count(const abo_ctx* ctx, int64_t* count);

/* per-kernel device timing of the candidate sweep (CUDA events on the context's stream around
 * every launch; bench.py's roofline leg).  enable != 0 resets and starts collecting; read
 * returns accumulated milliseconds and launch counts for {K* tile builder, DMMA triangular
 * product + sum-of-squares, acquisition epilogue}. */
int32_t abo_ctx_profile(abo_ctx* ctx, int32_t enable);
int32_t abo_ctx_profile_read(abo_ctx* ctx, double ms[3], int64_t launches[3]);

/* inspection: SM-clock timestamps of the phases of the last diagonal-block factorisation kernel
 * (load, factor, store L, inverse level 0, inverse levels, store) — tools/potrf_probe.py */
int32_t abo_debug_potf2_clocks(abo_ctx* ctx, int64_t out[16]);

/* ---- surrogate: struct StandardGP / GradientGP (src/surrogates/StandardGP.jl:11-16,
 *      GradientGP.jl:17-22).  p = 1 (StandardGP) or d + 1 (GradientGP). --------------------- */
int32_t abo_gp_create(abo_ctx* ctx, int32_t kernel_id, int32_t d, int32_t p, abo_gp** out);
int32_t abo_gp_destroy(abo_gp* gp);
/* inv_lengthscale is the stored ScaleTransform s = 1/l (surrogates_utils.jl:28-47), scale is the
 * ScaledKernel sigma^2, noise_var the observation noise, mean_c[p] the constant prior mean per
 * output (NULL = ZeroMean).  Invalidates any posterior held by the handle. */
int32_t abo_gp_set_params(abo_gp* gp, double inv_lengthscale, double scale, double noise_var,
                          const double* mean_c);
/* ARD: one inverse length scale PER DIMENSION, s_k = 1/l_k (KernelFunctions ARDTransform in place of ScaleTransform).  The
 * reference lists it as a TODO (src/bayesian_opt.jl:193-194); every entry point below (fit, append, posteriors incl. the
 * derivative blocks of a GradientGP, acquisitions and their gradients, multi-GPU sync) honours it.  d <= 32. */
int32_t abo_gp_set_params_ard(abo_gp* gp, const double* inv_lengthscales /* d */, double scale, double noise_var,
                              const double* mean_c);
/* update(model, xs, ys) (StandardGP.jl:79-83, GradientGP.jl:659-668): K + noise*I, Cholesky,
 * alpha.  *info = 0, or the 1-based failing pivot in the caller's out-major ordering is NOT
 * guaranteed — only info > 0 is (status ABO_ERR_NOT_POSDEF); the handle is then un-fitted. */
int32_t abo_gp_fit(abo_gp* gp, const double* X, const double* y, int64_t n, int64_t* info);
/* O(n^2) append of one observation (x[d], y[p]): one row for a StandardGP, the block of p = d+1 rows
 * for a GradientGP; transactional: on ABO_ERR_NOT_POSDEF the handle still holds the previous
 * posterior.  (The reference re-fits: bayesian_opt.jl:125.) */
int32_t abo_gp_append(abo_gp* gp, const double* x, const double* y, int64_t* info);
/* Base.copy(::StandardGP) (StandardGP.jl:26, surrogates_utils.jl:12-14).  Value semantics of a deep
 * copy at O(1) cost: the clone shares the device buffers (reference counted) and whichever handle
 * is written next (abo_gp_fit, abo_gp_append, the receiving side of abo_gp_sync) first takes a
 * private set — copy-on-write.  The BO loop's per-iteration snapshot (bayesian_opt.jl:116) is free. */
int32_t abo_gp_clone(const abo_gp* gp, abo_gp** out);
int32_t abo_gp_n(const abo_gp* gp, int64_t* n);
/* read back alpha (N = n*p, out-major) — PosteriorGP.data.α */
int32_t abo_gp_alpha(const abo_gp* gp, double* alpha);

/* read back the Cholesky factor (which = 0: lower L with K + noise*I = L L^T — the transpose of
 * PosteriorGP.data.C.U) or its inverse (which = 1) as a dense N x N row-major matrix in the
 * library's internal POINT-major ordering idx = i*p + out.  Inspection / tests only. */
int32_t abo_gp_factor(const abo_gp* gp, int32_t which, double* out);

/* posterior_mean / posterior_var (StandardGP.jl:361-379, GradientGP.jl:985-1003) when
 * outputs == 1; posterior_grad_mean / posterior_grad_var (GradientGP.jl:936-955) when
 * outputs == p (results out-major, length m*p).  mean / var may each be NULL. */
int32_t abo_gp_posterior(abo_gp* gp, const double* Xc, int64_t m, int32_t outputs,
                         double* mean, double* var);

/* full posterior covariance over all (point, output) pairs of a SMALL query set, out-major,
 * (m*outputs)^2 doubles row-major: cov(model.gpx(x)) / posterior_grad_cov (GradientGP.jl:968-971).
 * outputs == 1 or p; m*outputs <= 8192. */
int32_t abo_gp_posterior_cov(abo_gp* gp, const double* Xc, int64_t m, int32_t outputs, double* cov);

/* Joint samples of the latent value f over a candidate set: f_s = mu + chol(Sigma + tau I) z_s, where
 * Sigma = K(Xc,Xc) - K(Xc,X) (K + noise I)^-1 K(X,Xc) (+ 1e-18 I, as abo_gp_posterior_cov). This is AbstractGPs
 * rand(rng, posterior(fx)(Xc), S). Value output only, also for a GradientGP. Units are the model's own, the same as
 * abo_gp_posterior's mean.
 * samples: S x m, sample-major (row s = draw s). In Julia this is the m x S matrix rand returns. Nullable.
 * argmin_idx / argmin_val: per draw, the minimising candidate. Ties go to the first index. A NaN in a draw yields that
 * draw's first NaN, as Julia's findmin does. Both are nullable. The S argmins are a q = S Thompson batch, drawn with
 * replacement.
 * z_s[i] is a standard normal that depends only on (seed, s, i): Philox4x64-10 with key (seed, s), counter (i/4 + 1, 0, 0, 0)
 * -- NumPy's np.random.Philox(key=[seed, s]).random_raw() words 4j..4j+3 -- turned into four normals by two Box-Muller
 * pairs. So a call with S draws repeats, bit for bit, the S' < S draws of a call with S', and the argmins do not depend on
 * whether samples is NULL.
 * jitter > 0 is relative to the kernel scale: tau_k = jitter * sigma^2 * 10^k for k = 0..6, and the first tau whose
 * Cholesky succeeds is used and returned in *jitter_used (nullable). ABO_ERR_NOT_POSDEF after k = 6.
 * 1 <= m <= 16384, 1 <= S <= 4096; m <= 0 or S <= 0 is a no-op. The posterior held by gp is only read.
 * Device workspace: about 8 (2 m^2 + 2 m n p + 2 m S) bytes, 8 GB at m = 16384, n p = 8192, S = 4096 (abo_ctx_trim
 * releases it). */
int32_t abo_gp_posterior_sample(abo_gp* gp, const double* Xc, int64_t m, int64_t S, uint64_t seed, double jitter,
                                double* samples, int64_t* argmin_idx, double* argmin_val, double* jitter_used);

/* fused acquisition sweep: scores = acq(surrogate, Xc) (ExpectedImprovement.jl:40-45 etc.) and
 * sortperm(scores; rev=true)[1:k] (acq_utils.jl:50-52): stable, descending, NaN first.
 * scores (m) may be NULL — then only the k selected (index, value) pairs leave the device (the
 * selection is an exact radix select on the GPU; below 65 536 candidates the host picks them from
 * the read-back scores); k may be 0 (top_idx/top_val then unused).  Host candidate sets above
 * 262 144 points are staged, evaluated and read back in overlapped pieces. */
int32_t abo_acq_eval(abo_gp* gp, int32_t acq_id, const double* params, const double* Xc, int64_t m,
                     double* scores, int64_t k, int64_t* top_idx, double* top_val);
/* same, candidates already resident in HBM (d_Xc: m*d doubles, point-major); d_scores (device,
 * m doubles) may be NULL.  top_idx/top_val are host buffers. */
int32_t abo_acq_eval_dev(abo_gp* gp, int32_t acq_id, const double* params, const double* d_Xc,
                         int64_t m, double* d_scores, int64_t k, int64_t* top_idx, double* top_val);

/* EnsembleAcquisition (src/acquisition_functions/EnsembleAcq.jl:53-55): scores = sum_q weights[q] * acq_q(surrogate, Xc) with
 * members acq_ids[q] in {ABO_ACQ_EI, ABO_ACQ_PI, ABO_ACQ_UCB, ABO_ACQ_GRADNORM_UCB}; params is nmem x 2 (row q = the member's
 * {xi, best_y} or {beta, unused}); weights are used as given (the reference normalises them in the constructor).  ONE
 * posterior pass serves all members.  GradientNormUCB (gradNormUCB.jl:43-51, needs a GradientGP): per candidate the
 * posterior gradient mean m and the d x d posterior gradient covariance S are formed on the device —
 * -(m.m + tr S) + beta sqrt(max(4 m^T S m + 2 |S|_F^2, 1e-12)) — a single member with weight 1 is the plain acquisition.
 * scores / top-k as abo_acq_eval. */
int32_t abo_acq_eval_multi(abo_gp* gp, int32_t nmem, const int32_t* acq_ids, const double* weights, const double* params,
                           const double* Xc, int64_t m, double* scores, int64_t k, int64_t* top_idx, double* top_val);

/* acquisition value AND its gradient with respect to the query point for a batch of m points
 * (batched local refinement of optimize_acquisition, acq_utils.jl:55-71: the reference differentiates
 * single-point evaluations by finite differences; here mu, sigma^2 and their analytic gradients
 * come from one pass).  scores: m; grad: m x d point-major; mean / var (m) may be NULL.  d <= 32. */
int32_t abo_acq_eval_grad(abo_gp* gp, int32_t acq_id, const double* params, const double* Xc, int64_t m,
                          double* scores, double* grad, double* mean, double* var);

/* nlml(model, [log l, log sig2], xs, ys) and its gradient for R parameter vectors at once
 * (StandardGP.jl:99-149, GradientGP.jl:684-738, driven by bayesian_opt.jl:259-300).
 * logparams: R x 2 (row r = {log l, log sig2}); nlml: R; grad: R x 2 (may be NULL);
 * info: R (0 or failing pivot; a failed restart has nlml = +Inf, like the skipped restarts of
 * bayesian_opt.jl:296-299).  Uses gp's kernel id, noise and prior mean; does not touch its
 * posterior. */
int32_t abo_nlml_batch(abo_gp* gp, const double* X, const double* y, int64_t n,
                       const double* logparams, int64_t R, double* nlml, double* grad, int32_t* info);

/* the same for ARD parameter vectors {log l_1 .. log l_d, log sig2}: logparams R x (d+1), grad R x (d+1) (the extension of the
 * nlml parameter vector the reference plans at bayesian_opt.jl:193-194); StandardGP (p = 1), d <= 32. */
int32_t abo_nlml_batch_ard(abo_gp* gp, const double* X, const double* y, int64_t n,
                           const double* logparams, int64_t R, double* nlml, double* grad, int32_t* info);

/* monte_carlo_fill_distance (src/BO_utils.jl:140-159): max over the m sample points S (m x d) of the
 * distance to the nearest of the n training points X (n x d); the caller draws the samples. */
int32_t abo_fill_distance(abo_ctx* ctx, const double* X, int64_t n, int32_t d, const double* S, int64_t m,
                          double* h_fill);

/* get_mean_std + std_y of standardize_problem (src/BO_utils.jl:44-64; StandardGP.jl:164-204, GradientGP.jl:756-783) on the
 * device.  y: n*p observations, out-major; choice 0 "mean_scale", 1 "scale_only" (mu = 0), 2 "mean_only" (sd = 1).
 * mu[p], sd[p]: the empirical mean of the VALUE output (0 for gradient outputs) and its corrected sample standard deviation
 * (the same for every output); y_std[n*p] = (y - mu) / sd[0]; *best (nullable) = minimum of the standardised value output,
 * the incumbent update(acq, ys, model) needs (ExpectedImprovement.jl:81-83). */
int32_t abo_standardize(abo_ctx* ctx, const double* y, int64_t n, int32_t p, int32_t choice, double* mu, double* sd,
                        double* y_std, double* best);

/* ---- standalone factorisation entry (Cholesky TFLOP/s metric; A is n x n row-major, lower
 *      triangle referenced, overwritten by L on device; d_A device pointer, ld >= n) ---------- */
int32_t abo_potrf_dev(abo_ctx* ctx, double* d_A, int64_t n, int64_t ld, int64_t* info);

/* ---- multi-GPU (one process per GPU; NCCL over NVLink) -------------------------------- */
int32_t abo_nccl_unique_id(uint8_t id[128]);
int32_t abo_ctx_init_rank(abo_ctx* ctx, int32_t rank, int32_t nranks, const uint8_t id[128]);
/* rank / number of ranks of the context's NCCL communicator (0 / 1 when abo_ctx_init_rank was never called):
 * callers use it to decide whether the abo_*allgather* entry points span the job */
int32_t abo_ctx_ranks(const abo_ctx* ctx, int32_t* rank, int32_t* nranks);
/* broadcast the posterior (X, the lower tiles of L and L^-1, alpha, hyper-parameters) from `root` to every
 * rank.  COLLECTIVE, including its outcome: the root's state travels in the header and every rank's
 * validation / allocation status is all-gathered before any bulk transfer, so all ranks return the same
 * status (an un-fitted root, a handle created with another (d, p), an allocation failure) and none is left
 * blocked inside a collective. */
int32_t abo_gp_sync(abo_gp* gp, int32_t root);
/* all-gather every rank's (value, global index) top-k lists and merge them with the
 * (value desc, index asc, NaN first) order; in/out arrays have length k (count valid entries) */
int32_t abo_topk_allgather(abo_ctx* ctx, int64_t k, int64_t count, int64_t* top_idx, double* top_val,
                           int64_t* out_count);

/* all-gather `count` doubles per rank in rank order (recv: nranks * count); used for the results of
 * NLML restarts sharded R/G per rank (bayesian_opt.jl:264-300 runs them one after the other) */
int32_t abo_allgather_f64(abo_ctx* ctx, const double* send, int64_t count, double* recv);

#ifdef __cplusplus
}
#endif
#endif /* ABO_H */
