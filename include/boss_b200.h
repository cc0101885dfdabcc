/* boss_b200.h -- C ABI of libboss_b200.so, the B200 (sm_100a) backend for BOSS.jl's GP hot path.
 *
 * This is the drop-in boundary.  BOSS.jl (pure Julia) has no FFI of its own; the backend module
 * (julia/BossB200.jl, see INTEGRATION.md) adds more specific methods for the reference's documented
 * extension interfaces and `ccall`s the entry points below.  Each entry point cites the reference
 * function(s) it replaces (paths relative to the BOSS.jl v0.6.1 source tree).
 *
 * Conventions
 *   - All matrices are Float64, column-major with points as columns, exactly BOSS.jl's layout
 *     (src/types/data.jl:19-22): X is d x n  => point k is the d contiguous doubles at X + k*d.
 *   - Pointers are caller-owned HOST memory (pageable or pinned) valid for the duration of the call, except in
 *     the `_dev` variants where every array argument is a DEVICE pointer on the calling thread's device.  All
 *     library work runs on the library's own stream (boss_stream()).  The last argument `stream` of a `_dev`
 *     entry point is the CUDA stream on which the caller PRODUCED those device arrays (NULL = the legacy default
 *     stream, which is what torch and CUDA.jl use unless told otherwise): the library orders its stream after
 *     that stream before it reads them, and every entry point synchronises its own stream before it returns, so
 *     results are visible to any stream afterwards.
 *   - Raw hyper-parameters are passed exactly as the reference passes them to `finite_gp`
 *     (src/models/gaussian_process.jl:216-245): the library asserts >= 0 and adds MIN_PARAM_VALUE
 *     = 1e-8 itself.
 *   - Return value: 0 ok; > 0 a numerical condition that the reference reports by throwing and that
 *     its SafeFunction wrappers map to -Inf (BOSS_NOT_POSDEF, BOSS_NEG_VARIANCE); < 0 argument /
 *     CUDA errors with text in boss_last_error().  Nothing aborts, nothing throws across the ABI.
 *   - Devices.  boss_init(device): one process drives one GPU (the one-process-per-GPU layout of torchrun;
 *     candidates / samples are then sharded by the caller, boss.jl_b200/parallel.py).  boss_init_multi(n): ONE
 *     process drives GPUs 0..n-1 -- the layout a Julia caller has.  Fits are then replicated on every device
 *     (bit-identical: same deterministic kernels, same inputs), and the host-pointer scoring / log-likelihood /
 *     multi-start calls deal contiguous candidate blocks / sample ranges / starts to the devices (one host thread
 *     and one stream set per device) and reduce the (best value, index) pairs on the host in Julia's argmax
 *     order.  Results are bit-identical to the single-device call.  These are the reference's thread-parallel
 *     axes: src/acquisition_maximizers/grid.jl:58-62, sampling.jl:50-52, src/model_fitters/sampling.jl:40-49,
 *     src/utils/optim_multistart.jl:62.  boss_set_device(k) pins the calling thread to device k (for `_dev`
 *     calls and single-device use of a multi-device process); boss_set_device(-1) undoes it.
 *   - Thread-safe: entry points serialise on a per-device mutex (the reference may call from
 *     Threads.@threads tasks when parallel=true, src/utils/optim_multistart.jl:62).  boss_last_error() is
 *     per calling thread.  boss_shutdown() invalidates the handles that are still alive: later calls on them
 *     return BOSS_ERR_STATE, boss_gp_free() on them stays valid.
 *   - Limits that the reference does not have: x_dim <= 32, y_dim <= 16 (argument errors otherwise).
 */
#ifndef BOSS_B200_H
#define BOSS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BOSS_OK 0
#define BOSS_NOT_POSDEF 1      /* LinearAlgebra.PosDefException in cholesky()                     */
#define BOSS_NEG_VARIANCE 2    /* DomainError of _clip_var, src/models/gaussian_process.jl:186-194 */
#define BOSS_ERR_ARG (-1)
#define BOSS_ERR_CUDA (-2)
#define BOSS_ERR_STATE (-3)

/* kernel_id : KernelFunctions kernels the reference's GaussianProcess accepts on this path */
#define BOSS_KERNEL_SE 0        /* SqExponentialKernel                         */
#define BOSS_KERNEL_MATERN32 1  /* Matern32Kernel (examples/example.jl:88)     */
#define BOSS_KERNEL_MATERN52 2  /* Matern52Kernel (default, src/deprecated.jl:34) */

typedef struct boss_gp boss_gp; /* opaque: one fitted GP = one output slice x one hyper-parameter vector */

/* ---- runtime ---------------------------------------------------------------------------- */
int boss_init(int device);            /* select device, create streams + workspace; idempotent      */
int boss_init_multi(int n_gpus);      /* drive devices 0..n_gpus-1 from this process (see Devices above) */
int boss_set_device(int device);      /* pin the calling thread to one initialised device; -1 = unpin */
int boss_n_devices(void);             /* devices multi-device calls fan out to (1 after boss_init)  */
void boss_shutdown(void);
const char *boss_last_error(void);    /* of the calling thread; valid until its next library call   */
int boss_version(void);
int boss_device(void);                /* device of the calling thread's context, -1 before boss_init */
void *boss_stream(void);              /* the cudaStream_t library work on that device is ordered on (for event timing) */

/* ---- a1 + a2 : fit -----------------------------------------------------------------------
 * Replaces posterior_gp (src/models/gaussian_process.jl:199-211) -> finite_gp (:216-248) ->
 * AbstractGPs.posterior: builds K = a^2 kappa(|(x-x')/l|) + s^2 I, factors it (FP64 blocked
 * Cholesky), forms the triangular inverse and alpha = K^-1 (y - m(X)), and keeps them on the device
 * (the "factor cache": the reference refactors on every model_posterior call).
 *   X             d x n   training inputs
 *   y_minus_mean  n       Y[slice,:] - m(X)  (prior mean evaluated by the caller: nothing / const / closure)
 *   lengthscales  d       raw lambda[:,slice];  amplitude, noise_std raw alpha[slice], sigma[slice]
 *   discrete_mask d bytes or NULL  (DiscreteKernel, src/models/utils/kernels.jl:43-69: round, then scale)
 *   loglik_out    optional: log marginal likelihood of the same fit (gaussian_process.jl:269-280)
 * Returns BOSS_NOT_POSDEF (and *out = NULL) when the factorisation meets a non-positive pivot. */
int boss_gp_fit(const double *X, int d, int n, const double *y_minus_mean, const double *lengthscales,
                double amplitude, double noise_std, int kernel_id, const uint8_t *discrete_mask,
                boss_gp **out, double *loglik_out);
/* S posterior fits in one call (same X, per-fit hyper-parameters and targets): the batches of
 * model_posterior over BI samples x output slices (src/posterior.jl:15-19,38-41) -- TuringBI keeps tens to
 * hundreds of hyper-parameter samples and the reference refactors each one separately.  Arguments as
 * boss_gp_loglik_batch; out[s] receives a handle or NULL where K_s is not positive definite (return value
 * BOSS_NOT_POSDEF if any); loglik_out (S) optional. */
int boss_gp_fit_batch(const double *X, int d, int n, const double *Y_minus_mean, int64_t ldy,
                      const double *lengthscales, const double *amplitude, const double *noise_std, int kernel_id,
                      const uint8_t *discrete_mask, int64_t S, boss_gp **out, double *loglik_out);

/* Incremental factor cache: add ONE training point to a fitted GP with unchanged hyper-parameters in O(n^2)
 * (new row of L and of W = L^-1, alpha and the log-likelihood updated in place) instead of the O(n^3)
 * refactorisation the reference performs for every speculative point of SequentialBatchAM
 * (src/acquisition_maximizers/batch.jl:26-38 -> augment_dataset!, src/types/problem.jl:191-198) and for
 * every BO iteration (src/bo.jl:40-45).   x_new d coordinates; y_minus_mean_new = y - m(x_new).
 * Returns BOSS_NOT_POSDEF (handle unchanged) when the extended matrix is not positive definite. */
int boss_gp_append(boss_gp *gp, const double *x_new, double y_minus_mean_new, double *loglik_out);
void boss_gp_free(boss_gp *gp);
int boss_gp_n(const boss_gp *gp);
int boss_gp_d(const boss_gp *gp);

/* ---- a3 + a4 : predict --------------------------------------------------------------------
 * Replaces mean / var / mean_and_var(::GaussianProcessPosterior, x | X)
 * (src/models/gaussian_process.jl:143-178) incl. _clip_var (:186-194).
 *   Xs d x M candidates; prior_mean_s M values m(x*) or NULL (zero mean)
 *   mu, var  M each (either may be NULL); status M int32 or NULL: 0 ok, BOSS_NEG_VARIANCE where the
 *   reference would throw DomainError (var is then the raw unclipped value).
 * Returns 0, or BOSS_NEG_VARIANCE if any status is non-zero. */
int boss_gp_predict(const boss_gp *gp, const double *Xs, int64_t M, const double *prior_mean_s,
                    double *mu, double *var, int32_t *status);

/* Same with device pointers (Xs, prior mean and outputs already resident in HBM). */
int boss_gp_predict_dev(const boss_gp *gp, const double *Xs_dev, int64_t M, const double *prior_mean_s_dev,
                        double *mu_dev, double *var_dev, int32_t *status_dev, void *stream);

/* Posterior mean and variance with their x-gradients, for every posterior of a BI model in one call: what BOSS.jl
 * obtains by pushing ForwardDiff.Dual numbers through mean_and_var (gaussian_process.jl:169-178), e.g. to
 * differentiate an arbitrary NonlinFitness closure on the host (DESIGN.md 2.12).
 *   slices, y_dim, n_samples, Xs, prior_mean_s, prior_mean_grad_s  as boss_ei_value_grad (the prior mean and its
 *       gradient, y_dim x M and y_dim x d x M, are shared by the BI samples)
 *   P = n_samples * y_dim posteriors, q = s*y_dim + i;  outputs candidate-major, any of them may be NULL:
 *   mu, var, status  P x M at index m*P + q: bit for bit what boss_gp_predict gives for slices[q] (_clip_var included)
 *   dmu, dvar        P x d x M at index (m*d + j)*P + q;  at least one of the two must be given (else BOSS_ERR_ARG:
 *       boss_gp_predict gives mu and var alone)
 * Gradient conventions: dvar is 0 where the raw variance was < 0 (the clipped branch is a constant), discrete
 * (rounded) dims have zero derivative, dmu includes prior_mean_grad_s when given.  Limits as the gradient path:
 * x_dim <= 32, y_dim <= 16.  Returns 0, or BOSS_NEG_VARIANCE if any status is non-zero; M = 0 returns 0. */
int boss_gp_predict_grad(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                         const double *prior_mean_s, const double *prior_mean_grad_s, double *mu, double *var,
                         double *dmu, double *dvar, int32_t *status);

/* Replaces cov / mean_and_cov(::GaussianProcessPosterior, X) (gaussian_process.jl:163-167,180-184):
 * full M x M posterior covariance (column-major), diagonal clipped.  Intended for small M. */
int boss_gp_cov(const boss_gp *gp, const double *Xs, int64_t M, const double *prior_mean_s,
                double *mu, double *cov);

/* ---- a5 + a6 + a7 : acquisition scoring -----------------------------------------------------
 * Replaces the closure built by construct_safe_acquisition (src/acquisition.jl:21-25) ->
 * construct_acquisition(::ExpectedImprovement) (src/acquisitions/expected_improvement.jl:49-90) applied
 * to every column of Xs, and the argmax loops of GridAM / SamplingAM
 * (src/acquisition_maximizers/grid.jl:52-65, sampling.jl:37-48).
 *   slices        n_samples x y_dim handles, sample-major: slices[s*y_dim + i]  (posterior.jl:15-19,38-41)
 *   prior_mean_s  y_dim x M (column-major: y_dim contiguous per candidate) or NULL
 *   fit_coefs     y_dim LinFitness coefficients
 *   best          pointer to best-so-far fitness or NULL (= `nothing`, no feasible observation)
 *   y_max         y_dim constraints (+Inf = unconstrained, cdf == 1 exactly) or NULL (no constraints)
 *   lb, ub        d each or NULL: out-of-bounds candidates score 0. (make_safe, :58-65; inclusive)
 *   cons_mask     M bytes or NULL: 0 => cons(x) violated => score 0.
 *   acq           M scores or NULL;  grad d x M x-gradients or NULL
 *   best_val / best_idx  Julia argmax semantics: first maximal, NaN maximal (may be NULL)
 * Candidates whose variance fails _clip_var score -Inf (SafeFunction, src/utils/optim.jl:20-34). */
int boss_ei_score(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                  const double *prior_mean_s, const double *fit_coefs, const double *best,
                  const double *y_max, const double *lb, const double *ub, const uint8_t *cons_mask,
                  double *acq, double *grad, double *best_val, int64_t *best_idx);

/* Same, every array argument a device pointer (candidates already resident in HBM); ordered after `stream`
 * (see Conventions) and synchronised before return.  best_val / best_idx are HOST pointers. */
int boss_ei_score_dev(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs_dev,
                      int64_t M, const double *prior_mean_s_dev, const double *fit_coefs, const double *best,
                      const double *y_max, const double *lb, const double *ub, const uint8_t *cons_mask_dev,
                      double *acq_dev, double *grad_dev, double *best_val, int64_t *best_idx, void *stream);

/* The k best candidates of the same scores (SampleOptAM's starts, src/acquisition_maximizers/sample_opt.jl:41-52),
 * selected on the device: no M-sized output, no host sort.  Arguments as boss_ei_score; top_val / top_idx are HOST
 * arrays of k (also in the _dev variant, whose other array arguments are device pointers).
 *   k        1 <= k <= min(M, 8192), BOSS_ERR_ARG otherwise (BOSS.jl's order[1:multistart] throws for multistart > samples)
 *   order    the scores in descending order under Julia's isless: NaN largest (all NaNs rank equal), -0.0 below +0.0,
 *            ties to the lower index -- Julia's stable sortperm(vals; rev=true), truncated to k.  This is the order of
 *            best_val / best_idx too: top_val[0], top_idx[0] equal boss_ei_score's pair bit for bit.
 *   indices  0-based, into Xs; with boss_init_multi the result is bit-identical to the single-device call.
 * With `best` set and at least 64 Ki candidates the call scores exactly only candidates whose EI upper bound can still
 * reach the k best (DESIGN.md 2.10); the result is the same either way. */
int boss_ei_score_topk(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                       const double *prior_mean_s, const double *fit_coefs, const double *best, const double *y_max,
                       const double *lb, const double *ub, const uint8_t *cons_mask, int64_t k, double *top_val,
                       int64_t *top_idx);
int boss_ei_score_topk_dev(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs_dev, int64_t M,
                           const double *prior_mean_s_dev, const double *fit_coefs, const double *best,
                           const double *y_max, const double *lb, const double *ub, const uint8_t *cons_mask_dev,
                           int64_t k, double *top_val, int64_t *top_idx, void *stream);

/* Same scoring with the candidates GENERATED ON THE DEVICE -- the batch never exists in host memory
 * (16 Mi x 8 candidates = 1 GiB in BASELINE config C2).  Indices are global; a shard [first, first + M) of the
 * index range reproduces exactly the points of the unsharded call, so multi-GPU sharding is by index block.
 *   grid     GridAM's Iterators.product over per-dimension ranges, first dimension fastest
 *            (src/acquisition_maximizers/grid.jl:30-43): x_j = lo_j + step_j * ((m / prod_{i<j} count_i) mod count_j);
 *            M = -1 scores to the end of the grid
 *   uniform  SamplingAM with a uniform prior over the box (src/acquisition_maximizers/sampling.jl:59-75):
 *            x_j = lb_j + u(seed, m*d + j) (ub_j - lb_j), u a stateless splitmix64 counter hash in [0, 1)
 *   prior_mean_s / cons_mask / acq  optional HOST arrays indexed by (m - first);  best_x d coordinates of the winner */
int boss_ei_score_grid(const boss_gp *const *slices, int y_dim, int n_samples, int d, const double *grid_lo,
                       const double *grid_step, const int64_t *grid_count, int64_t first, int64_t M,
                       const double *prior_mean_s, const double *fit_coefs, const double *best, const double *y_max,
                       const double *lb, const double *ub, const uint8_t *cons_mask, double *acq, double *best_val,
                       int64_t *best_idx, double *best_x);
int boss_ei_score_uniform(const boss_gp *const *slices, int y_dim, int n_samples, int d, uint64_t seed, int64_t first,
                          int64_t M, const double *box_lb, const double *box_ub, const double *prior_mean_s,
                          const double *fit_coefs, const double *best, const double *y_max, const uint8_t *cons_mask,
                          double *acq, double *best_val, int64_t *best_idx, double *best_x);

/* Monte-Carlo expected improvement of a NonlinFitness on the device, for fitness functions from a small expression
 * set; replaces expected_improvement(::NonlinFitness, mean, var, eps, best) (src/acquisitions/expected_improvement.jl:104-111)
 * inside the same four construct_ei cases, guards and argmax as boss_ei_score:
 *   EI(x) = 1/K sum_k max(0, f(mu(x) + sqrt(var(x)) .* eps[:,k]) - best)
 *   fit_kind 1  f(y) = c0 + sum_i c_i y_i                          (affine)
 *            2  f(y) = c0 + sum_i c_i y_i + sum_i q_i (y_i - t_i)^2 (diagonal quadratic)
 *            3  f(y) = c0 + max_i (c_i y_i + t_i) over outputs with c_i != 0
 *            4  f(y) = c0 + min_i (c_i y_i + t_i) over outputs with c_i != 0
 *   fit_c / fit_q / fit_t  y_dim each (NULL = zeros);  eps  y_dim x n_eps column-major = the reference's
 *   sample_eps matrix (:119), n_eps <= 4096; with n_samples > 1 (BI) posterior s uses column s and n_eps == n_samples.
 * A fitness that is an arbitrary Julia closure cannot run on the device: boss_gp_predict returns mu, var and the
 * host finishes (INTEGRATION.md). */
int boss_mcei_score(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                    const double *prior_mean_s, int fit_kind, double fit_c0, const double *fit_c, const double *fit_q,
                    const double *fit_t, const double *eps, int n_eps, const double *best, const double *y_max,
                    const double *lb, const double *ub, const uint8_t *cons_mask, double *acq, double *best_val,
                    int64_t *best_idx);

/* The same Monte-Carlo EI for OptimizationAM and SampleOptAM (the reference pushes ForwardDiff.Dual numbers through
 * expected_improvement(::NonlinFitness, ...)).  fit_kind, fit_c0, fit_c, fit_q, fit_t, eps and n_eps as in
 * boss_mcei_score, with the same limits and error texts; every other argument as in the LinFitness twin.
 *   boss_mcei_value_grad           as boss_ei_value_grad: acq equals boss_mcei_score's acq bit for bit
 *   boss_mcei_maximize_multistart  as boss_ei_maximize_multistart; eps is uploaded once per solve and device
 *   boss_mcei_score_topk           as boss_ei_score_topk (same order and k range); never screened
 * The x-gradient (DESIGN.md 2.11): for posterior s with eps columns K_s, y_k = mu + sd .* eps_k, imp_k = f(y_k) - best,
 *   d EI_s / dx_j = sum_i A_i d mu_i/dx_j + B_i d sd_i/dx_j ,
 *   A_i = 1/|K_s| sum_{k: imp_k > 0} g_i(y_k) ,  B_i = 1/|K_s| sum_{k: imp_k > 0} g_i(y_k) eps_ik ,  g_i = df/dy_i:
 *   affine c_i;  quadratic c_i + 2 q_i (y_i - t_i);  max / min c_i* for the output i* the value took, 0 for the others.
 *   d sd_i = d var_i / (2 sd_i) when sd_i > 0 and the variance was not clipped, else 0.  PoF enters by the product rule,
 *   the result is averaged over s, and the guards of boss_ei_value_grad apply.  With best == NULL (PoF only) the
 *   gradient equals boss_ei_value_grad's bit for bit.
 * Conventions at the measure-zero kinks: the derivative of the branch the value took -- imp_k == 0 contributes 0
 * (the value takes imp > 0 ? imp : 0), a max / min tie goes to the first output.  A candidate whose value is NaN gets a
 * NaN gradient.  Whether ForwardDiff returns the same numbers at these points has not been checked.
 * Cost: |K_s| y_dim per candidate and posterior for A and B, then d y_dim for the gradient. */
int boss_mcei_value_grad(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                         const double *prior_mean_s, const double *prior_mean_grad_s, int fit_kind, double fit_c0,
                         const double *fit_c, const double *fit_q, const double *fit_t, const double *eps, int n_eps,
                         const double *best, const double *y_max, const double *lb, const double *ub,
                         const uint8_t *cons_mask, double *acq, double *grad);
int boss_mcei_maximize_multistart(const boss_gp *const *slices, int y_dim, int n_samples, const double *starts,
                                  int64_t M, int iters, int history, const double *prior_mean_affine, int fit_kind,
                                  double fit_c0, const double *fit_c, const double *fit_q, const double *fit_t,
                                  const double *eps, int n_eps, const double *best, const double *y_max,
                                  const double *lb, const double *ub, const uint8_t *discrete_mask, double *x_out,
                                  double *f_out, double *best_x, double *best_val, int64_t *best_idx, int *evals_out);
int boss_mcei_score_topk(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                         const double *prior_mean_s, int fit_kind, double fit_c0, const double *fit_c,
                         const double *fit_q, const double *fit_t, const double *eps, int n_eps, const double *best,
                         const double *y_max, const double *lb, const double *ub, const uint8_t *cons_mask, int64_t k,
                         double *top_val, int64_t *top_idx);

/* Value + analytic x-gradient of the same acquisition for a batch of points: what OptimizationAM's
 * multi-start solver needs per iteration over all starts (src/acquisition_maximizers/optimization.jl:89-118;
 * the reference obtains the gradient by pushing ForwardDiff.Dual numbers through the posterior).
 *   prior_mean_grad_s  y_dim x d x M (index (m*d + j)*y_dim + i) gradient of the host-evaluated prior mean, or NULL
 *   grad               d x M;  zero for out-of-domain / failed candidates; discrete (rounded) dims have zero derivative */
int boss_ei_value_grad(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs, int64_t M,
                       const double *prior_mean_s, const double *prior_mean_grad_s, const double *fit_coefs,
                       const double *best, const double *y_max, const double *lb, const double *ub,
                       const uint8_t *cons_mask, double *acq, double *grad);
int boss_ei_value_grad_dev(const boss_gp *const *slices, int y_dim, int n_samples, const double *Xs_dev, int64_t M,
                           const double *prior_mean_s_dev, const double *prior_mean_grad_s_dev,
                           const double *fit_coefs, const double *best, const double *y_max, const double *lb,
                           const double *ub, const uint8_t *cons_mask_dev, double *acq_dev, double *grad_dev,
                           void *stream);

/* Device-resident multi-start maximisation: OptimizationAM (src/acquisition_maximizers/optimization.jl:55-118)
 * with all `multistart` local solves advancing in lock-step as projected L-BFGS with Armijo backtracking; every
 * value + gradient evaluation of all starts is one batched pass on the device, the points never leave HBM
 * between iterations.  Ends with the reference's discrete rounding + re-evaluation (optimization.jl:116-117) and
 * the argmax over the starts (first maximal; failed starts = -Inf, optim_multistart.jl:28-42).
 *   starts d x M; lb / ub the box (required); discrete_mask d bytes or NULL
 *   prior_mean_affine  y_dim x (d + 1) or NULL: slice i has prior mean c_i + b_i . x with [c_i, b_i1..b_id] at
 *                      prior_mean_affine + i*(d+1) (constant means, linear parametric part of a Semiparametric model)
 *   x_out d x M final points, f_out M final values (either may be NULL); best_val == -Inf <=> all runs failed
 *   evals_out  evaluated points / M of the backtracking searches (a trial only re-evaluates the starts that have not
 *              accepted a step; once few starts are left the next step sizes of a search are evaluated speculatively
 *              in the same pass -- same trajectory, fewer passes -- and those extra points are not counted)
 * General prior-mean closures and `cons` constraints are host code and are not supported here: use
 * boss_ei_value_grad per iteration for those. */
int boss_ei_maximize_multistart(const boss_gp *const *slices, int y_dim, int n_samples, const double *starts, int64_t M,
                                int iters, int history, const double *prior_mean_affine, const double *fit_coefs,
                                const double *best,
                                const double *y_max, const double *lb, const double *ub, const uint8_t *discrete_mask,
                                double *x_out, double *f_out, double *best_x, double *best_val, int64_t *best_idx,
                                int *evals_out);

/* ---- a8 + a9 : batched log marginal likelihood ------------------------------------------------
 * Replaces data_loglike(::GaussianProcess) / gp_data_loglike_slice (gaussian_process.jl:250-280)
 * -> logpdf(::FiniteGP, y) evaluated for S hyper-parameter vectors at once: the batches built by
 * SamplingMAP (src/model_fitters/sampling.jl:59-78), OptimizationMAP multistart
 * (optimization.jl:116-119) and the TuringBI model (ext/TuringExt.jl:78-86), for ONE output slice.
 *   Y_minus_mean  n (ldy == 0: shared by all samples) or S x n with sample s at Y_minus_mean + s*ldy
 *                 (Semiparametric: the mean depends on theta_s)
 *   lengthscales  d x S (sample s = d contiguous doubles), amplitude S, noise_std S (raw values)
 *   loglik        S results; -Inf where K is not positive definite (safe_data_loglike)
 * Returns 0 or BOSS_NOT_POSDEF if any sample failed; BOSS_ERR_ARG for a negative or NaN hyper-parameter (the
 * reference's asserts).  The `_dev` variants cannot inspect device-resident hyper-parameters on the host: a
 * negative one yields NaN for that sample.  NaN in X or Y yields -Inf (LAPACK's potrf rejects a NaN pivot). */
int boss_gp_loglik_batch(const double *X, int d, int n, const double *Y_minus_mean, int64_t ldy,
                         const double *lengthscales, const double *amplitude, const double *noise_std,
                         int kernel_id, const uint8_t *discrete_mask, int64_t S, double *loglik);

int boss_gp_loglik_batch_dev(const double *X_dev, int d, int n, const double *Y_minus_mean_dev, int64_t ldy,
                             const double *lengthscales_dev, const double *amplitude_dev,
                             const double *noise_std_dev, int kernel_id, const uint8_t *discrete_mask,
                             int64_t S, double *loglik_dev, void *stream);

/* Same batch, plus the gradient of each log-likelihood w.r.t. the raw hyper-parameters, ordered like the
 * reference's vectorizer [vec(lambda); alpha; sigma] (src/models/gaussian_process.jl:300-328):
 *   d LML / d theta = 1/2 tr((alpha alpha^T - K^-1) dK/dtheta),  K^-1 = W^T W formed on the tensor cores.
 * Replaces the ForwardDiff.Dual sweep through logpdf(::FiniteGP) that OptimizationMAP's gradient algorithms
 * and NUTS (TuringBI) perform (src/model_fitters/optimization.jl:41,153; docs/src/example.md:155-163).
 *   grad  S x (d + 2), sample s at grad + s*(d+2); zeros where the sample is not positive definite. */
int boss_gp_loglik_grad_batch(const double *X, int d, int n, const double *Y_minus_mean, int64_t ldy,
                              const double *lengthscales, const double *amplitude, const double *noise_std,
                              int kernel_id, const uint8_t *discrete_mask, int64_t S, double *loglik, double *grad);
int boss_gp_loglik_grad_batch_dev(const double *X_dev, int d, int n, const double *Y_minus_mean_dev, int64_t ldy,
                                  const double *lengthscales_dev, const double *amplitude_dev,
                                  const double *noise_std_dev, int kernel_id, const uint8_t *discrete_mask,
                                  int64_t S, double *loglik_dev, double *grad_dev, void *stream);

/* Same batch and outputs, plus the gradient w.r.t. the parameters theta of a parametric prior mean m(x; theta) -- the
 * Semiparametric model's part of what ForwardDiff differentiates in OptimizationMAP / NUTS:
 *   d LML / d theta_c = alpha^T J[:, c],   alpha = K^-1 (y - m(X; theta)),   J = dm(X; theta)/dtheta   (DESIGN.md 2.13)
 * The caller differentiates m on the host (ForwardDiff.jacobian's n x k layout) and passes Y_minus_mean per sample.
 *   mean_jac   n x k column-major per sample (element (i, c) at i + c*n), sample s at mean_jac + s*ldj;
 *              ldj == 0: one Jacobian shared by all samples (a mean linear in theta)
 *   grad_mean  S x k, sample s at grad_mean + s*k: sum over the n rows of alpha_i J_ic; zeros where the sample is not
 *              positive definite
 * loglik and grad equal boss_gp_loglik_grad_batch's bit for bit, and a sample's grad_mean does not depend on the batch it
 * is evaluated in.  BOSS_ERR_ARG also for k < 1, a NULL grad / mean_jac / grad_mean, and 0 < ldj < k*n. */
int boss_gp_loglik_grad_batch_mean(const double *X, int d, int n, const double *Y_minus_mean, int64_t ldy,
                                   const double *mean_jac, int k, int64_t ldj,
                                   const double *lengthscales, const double *amplitude, const double *noise_std,
                                   int kernel_id, const uint8_t *discrete_mask, int64_t S,
                                   double *loglik, double *grad, double *grad_mean);
int boss_gp_loglik_grad_batch_mean_dev(const double *X_dev, int d, int n, const double *Y_minus_mean_dev, int64_t ldy,
                                       const double *mean_jac_dev, int k, int64_t ldj,
                                       const double *lengthscales_dev, const double *amplitude_dev,
                                       const double *noise_std_dev, int kernel_id, const uint8_t *discrete_mask,
                                       int64_t S, double *loglik_dev, double *grad_dev, double *grad_mean_dev,
                                       void *stream);

/* ---- instrumentation ---------------------------------------------------------------------
 * CUDA-event time (ms) of the dominant kernel class inside the last scoring / loglik call, and the
 * number of kernel launches the library has issued since boss_init (bench.py's gpu_launches). */
void boss_set_timing(int on);          /* bracket kernel classes with CUDA events (default off)              */
double boss_last_kernel_ms(int which); /* 0 = scoring TRMM, 1 = kernel-matrix / cross-covariance, 2 = Cholesky GEMMs, 3 = whole call */
int boss_last_kernel_count(int which); /* launches summed into boss_last_kernel_ms(which)                     */
int64_t boss_launch_count(void);

/* ---- debug / test hooks (used by tests/ only) ------------------------------------------------ */
int boss_dbg_gemm_nt(const double *A, const double *B, int M, int N, int K, double *C); /* C = A B^T, row-major dense */
/* device scalar functions of the kernel-matrix stages: which = 0 exp(-t), 1 sqrt(t), 2-4 kappa(d2) SE / Matern32 /
 * Matern52, 5-7 kappa'(r)/r of the same */
int boss_dbg_kernel_fn(int which, const double *t, int n, double *out);
int boss_dbg_factors(const boss_gp *gp, double *L, double *W, double *alpha);          /* dense row-major n x n, n   */
/* BOSS_DEBUG_REDZONE=1 (environment, read at the first allocation): every device allocation is exact-sized and
 * bracketed by 64 KB guard bands of 0xA5.  Returns the number of guard bytes overwritten so far on the calling
 * thread's device (0 = clean), -1 when the mode is off; *n_allocs = live allocations scanned.  The pool that builds
 * this library has compute-sanitizer closed (profiles/r02_compute_sanitizer_closed.txt); this is the bounds check
 * it recommends instead. */
int64_t boss_dbg_check_redzones(int64_t *n_allocs);
int64_t boss_dbg_redzone_selftest(void);   /* negative control: writes 2 guard bytes on purpose, returns how many the scan found */
/* argmax / top-k screening of the last scoring call on the current device: out[0] = 0 not screened, 1 screened, 2 fell back
 * to the full path after the first chunk; out[1] = candidates bounded; out[2] = candidates that survived the bound and
 * the re-seeded threshold (the pool scored exactly) */
int boss_dbg_screen_stats(int64_t *out);
/* the FP32 mean tier of the last screened call: out[0] = candidates in the ambiguous band (their means were recomputed in
 * FP64), out[1] = the pool as the chunks left it (definite keeps plus ambiguous candidates), before the FP64 refinement
 * and the re-seeded threshold */
int boss_dbg_screen_ambiguous(int64_t *out);
/* the FP32 tier's mean mu~ and error bound E, and the FP64 mean, of M candidates (d x M column-major) under gp
 * (K*^T alpha, no prior mean) */
int boss_dbg_screen_mean(const boss_gp *gp, const double *Xs, int64_t M, double *mu32, double *E, double *mu64);
/* the FP32 tier's kappa at d2 = (float)(r^2), kid 0 SE, 1 Matern32, 2 Matern52 */
int boss_dbg_kappa_f32(int kid, const double *r, int n, double *out);

#ifdef __cplusplus
}
#endif
#endif /* BOSS_B200_H */
