/* lfm_b200.h -- C-ABI of the B200-native latent-force-model (LFM) hot path.
 *
 * Drop-in boundary for wejpurvis/DIS_project's GP latent force model.  The reference has no FFI
 * of its own: its "operator API" is four Python call shapes (SURVEY.md 8b).  Every entry point
 * below names the reference call site (file:line under the reference repo) whose numerics it
 * replaces; INTEGRATION.md shows the reference-side binding (jax.ffi / ctypes).
 *
 * Conventions
 *   - all arithmetic is IEEE fp64 (the reference runs with jax_enable_x64, src/dataset.py:18);
 *   - every pointer is a DEVICE pointer unless the function name ends in _host;
 *   - calls are stream-ordered on `stream` (a cudaStream_t passed as void*), never synchronise,
 *     never allocate: scratch comes from the caller through the *_workspace_bytes queries;
 *   - inputs X / Xstar are the reference's (n,3) row-major arrays [time, gene_index, flag]
 *     (src/dataset.py:358-399, src/utils.py:268-287), gene index and flag stored as doubles;
 *   - theta is the CONSTRAINED hyper-parameter vector [true_d(G), true_s(G), true_b(G), l,
 *     obs_stddev] (src/model.py:64-121), P = 3G+2 doubles; theta_unc is the same vector in the
 *     unconstrained space of the tfp bijectors (softplus on all but l, Sigmoid(0.5,3.5) on l);
 *   - return value: LFM_OK or a negative lfm_status.  Numerical failure (Sigma not positive
 *     definite) is reported asynchronously through the device word `info` (0 = ok, k>0 = 1-based
 *     failing pivot), exactly like LAPACK; the outputs are then NaN, as in the reference
 *     (JAX's Cholesky returns NaN instead of raising).  One deviation: the dense factorisation also
 *     fails at a positive pivot below DBL_MIN (2^-1022), which LAPACK would factor (its reciprocal
 *     square root flushes subnormals to zero).
 */
#ifndef LFM_B200_H
#define LFM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* lfm_stream_t; /* cudaStream_t */

typedef enum lfm_status {
  LFM_OK = 0,
  LFM_ERR_INVALID = -1,     /* bad argument (null pointer, non-positive size, N % G != 0 ...) */
  LFM_ERR_CUDA = -2,        /* a CUDA runtime call failed; cudaGetLastError has the detail      */
  LFM_ERR_UNSUPPORTED = -3, /* size outside what the kernels support (e.g. batched N > 128)     */
  LFM_ERR_WORKSPACE = -4,   /* workspace too small                                             */
  LFM_ERR_NO_DEVICE = -5,   /* no sm_100 device: there is NO CPU fallback                       */
  LFM_ERR_COMM = -6         /* NCCL is not loadable on this host, or an NCCL call failed          */
} lfm_status;

#define LFM_ABI_VERSION 2

int lfm_abi_version(void);
const char* lfm_status_string(int status);
/* LFM_OK iff the current CUDA device exists and is compute capability 10.x. */
int lfm_device_check(void);

/* ---- (a) covariance blocks ------------------------------------------------------------------ */

/* ExactLFM.cross_covariance(kernel, x, y) with ExactLFM.kernel (src/model.py:372-394, 152-195):
 * flag-switched blend of k_xx (:197-235), k_xf (:237-282) and k_ff (:284-312).  out is N x M
 * row-major with leading dimension ld_out >= M. */
int lfm_cross_covariance(lfm_stream_t stream, int64_t N, int64_t M, const double* X, const double* Y,
                         int G, const double* theta, double* out, int64_t ld_out);

/* ExactLFM.gram(kernel, x) (src/model.py:396-414) == cross_covariance(x, x), full N x N. */
int lfm_gram(lfm_stream_t stream, int64_t N, const double* X, int G, const double* theta, double* out,
             int64_t ld_out);

/* ExactLFM.h(j, k, t1, t2) (src/model.py:315-365), elementwise over n tuples; j, k are gene indices
 * stored as doubles like the gene column of X. */
int lfm_h(lfm_stream_t stream, int64_t n, const double* j, const double* k, const double* t1,
          const double* t2, int G, const double* theta, double* out);

/* ExactLFM.mean_function(x) (src/model.py:124-149): (B/D)[i / (N/G)] * flag_i.  N % G must be 0. */
int lfm_mean_function(lfm_stream_t stream, int64_t N, const double* X, int G, const double* theta,
                      double* out);

/* tfp bijector forward / inverse applied leaf-wise, as gpjax Module.constrain()/unconstrain()
 * (src/trainer.py:75,103,218; bijectors at src/model.py:66,79,86,93,111).  B vectors of P=3G+2. */
int lfm_constrain(lfm_stream_t stream, int64_t B, int G, const double* theta_unc, double* theta);
int lfm_unconstrain(lfm_stream_t stream, int64_t B, int G, const double* theta, double* theta_unc);

/* ---- (b,c) objective and its gradient ------------------------------------------------------- */

size_t lfm_nlml_workspace_bytes(int64_t N, int G);

/* CustomConjMLL(negative=True)(model, Dataset(X, y)) (src/objectives.py:21-78):
 * Sigma = K + jitter I + sigma^2 I; out[0] = 1/2 [N log 2pi + log det Sigma + z^T Sigma^-1 z].
 * TRAINING ROWS MUST ALL CARRY FLAG 1: Sigma is built from k_xx alone (every training row of the reference has flag
 * 1, src/dataset.py:388); for a flag-0 row objectives.py:70 would blend k_xf / k_ff in, which this path (and the
 * posteriors' training covariance, and the batched fits) does not do.  The *_host entry points and the Python layer
 * reject such X (LFM_ERR_UNSUPPORTED / ValueError); device-pointer callers are trusted. */
int lfm_nlml(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
             const double* theta, double jitter, void* ws, size_t ws_bytes, double* out, int* info);

/* jax.value_and_grad(JaxTrainer.loss) (src/trainer.py:86-103,126) in CONSTRAINED coordinates:
 * out[0] = NLML, out[1..P] = dNLML/dtheta.  dK/dtheta blocks are contracted with
 * K_bar = 1/2 (Sigma^-1 - alpha alpha^T) on the fly and never materialised. */
int lfm_nlml_grad(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
                  const double* theta, double jitter, void* ws, size_t ws_bytes, double* out, int* info);

/* Same, differentiated w.r.t. the UNCONSTRAINED leaves -- the exact quantity the optimiser in
 * src/trainer.py:126-128 consumes.  out[0] = NLML, out[1..P] = gradient. */
int lfm_nlml_grad_unc(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
                      const double* theta_unc, double jitter, void* ws, size_t ws_bytes, double* out,
                      int* info);

/* ---- time-grid variants ----------------------------------------------------------------------
 * `time_grid` is an upper bound on the number of DISTINCT times among the rows of X (0 = unknown;
 * lfm_count_distinct_times gives it from a host copy).  The reference's layout observes every gene on
 * the same few time points (src/dataset.py:380-391), and the exp/erf factors of h (src/model.py:315-365)
 * depend on (gene, t, t') only: when the bound is small the library finds the distinct times on the
 * device, tabulates those factors once per evaluation (G T^2 entries instead of N^2) and builds Sigma
 * and the dK/dtheta contraction from the tables.  The tables hold the very values the direct path
 * computes; results agree to rounding.  If X has more distinct times than the bound, the kernels
 * detect it on the device and evaluate directly.  The plain entry points above are time_grid = 0. */
int64_t lfm_count_distinct_times(int64_t N, const double* X_host);
size_t lfm_nlml_workspace_bytes_tg(int64_t N, int G, int64_t time_grid);
int lfm_nlml_tg(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y, const double* theta,
                double jitter, int64_t time_grid, void* ws, size_t ws_bytes, double* out, int* info);
int lfm_nlml_grad_tg(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
                     const double* theta, double jitter, int64_t time_grid, void* ws, size_t ws_bytes,
                     double* out, int* info);
int lfm_nlml_grad_unc_tg(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
                         const double* theta_unc, double jitter, int64_t time_grid, void* ws, size_t ws_bytes,
                         double* out, int* info);

/* ---- heteroscedastic objective ----------------------------------------------------------------
 * Sigma = K + diag(variances) + jitter I + sigma^2 I: the measurement variances of dataset_3d
 * (src/dataset.py:396-397) inside the training covariance, the convention of the reference's GPyTorch twin when it
 * trains (src/gpytorch_alfi/model_alfi.py:294-299: K_xx += 1e-4 I; K_xx += self.variance).  `variances` is N doubles
 * (device) or NULL, in which case these ARE the entry points above.  The gradient formulas do not change
 * (d Sigma / d theta has no variance term); only the diagonal tiles of the Sigma build read `variances`. */
int lfm_nlml_het_tg(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y, const double* variances,
                    const double* theta, double jitter, int64_t time_grid, void* ws, size_t ws_bytes, double* out,
                    int* info);
int lfm_nlml_grad_het_tg(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
                         const double* variances, const double* theta, double jitter, int64_t time_grid, void* ws,
                         size_t ws_bytes, double* out, int* info);
int lfm_nlml_grad_unc_het_tg(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
                             const double* variances, const double* theta_unc, double jitter, int64_t time_grid,
                             void* ws, size_t ws_bytes, double* out, int* info);

/* ---- (d) latent posterior -------------------------------------------------------------------- */

size_t lfm_latent_posterior_workspace_bytes(int64_t N, int G, int64_t Tstar);

/* ExactLFM.latent_predict(test_inputs, train_data) (src/model.py:420-463):
 * Sigma_p = K + diag(variances) + jitter I; mean = mean_t + K_fx Sigma_p^-1 (y - mean_x);
 * var_i = k(t*_i,t*_i) + 2 jitter - k_i^T Sigma_p^-1 k_i.  Only the diagonal of the predictive
 * covariance is produced (the reference builds T* x T* and keeps the diagonal, :459-461). */
int lfm_latent_posterior(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
                         const double* variances, const double* theta, double jitter, int64_t Tstar,
                         const double* Xstar, void* ws, size_t ws_bytes, double* out_mean,
                         double* out_var, int* info);

/* ExactLFM.multi_gene_predict(test_inputs, train_data) (src/model.py:465-514; SURVEY 8f "next" row 1):
 * Sigma_g = K + diag(variances) + sigma^2 I (no jitter); mean = mean_t + K_tx Sigma_g^-1 (y - mean_x);
 * cov = K_tt - K_tx Sigma_g^-1 K_xt + jitter I.  out_cov (T* x T* row-major) and out_var (its diagonal)
 * may each be NULL.  Tstar % G must be 0 (mean_function's reshape). */
size_t lfm_gene_posterior_workspace_bytes(int64_t N, int G, int64_t Tstar);
int lfm_gene_posterior(lfm_stream_t stream, int64_t N, int G, const double* X, const double* y,
                       const double* variances, const double* theta, double jitter, int64_t Tstar,
                       const double* Xstar, void* ws, size_t ws_bytes, double* out_mean, double* out_cov,
                       double* out_var, int* info);

/* ---- batched multi-start path (many independent small LFMs per GPU) -------------------------- */

/* Rows of the duplicate-row-compressed problem for a HOST copy of X: the number of distinct rows when every distinct
 * (time, gene, flag) row occurs the same number of times R > 1 (the p53 layout repeats each row once per replicate),
 * else N -- the batched kernels compress only uniform multiplicities, and this mirrors their rule.  Passing it as
 * `unique_rows_hint` lets them size their shared memory for the compressed problem; 0 means "unknown" (sized for N).
 * A hint smaller than what the kernel finds makes it refuse with info = -1. */
int lfm_count_unique_rows(int64_t N, const double* X_host);

/* B independent value_and_grad evaluations sharing (X, y): theta_unc is B x P, out_val B,
 * out_grad B x P, info B ints.  N <= 128. */
int lfm_batched_nlml_grad_unc(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X,
                              const double* y, const double* theta_unc, double jitter,
                              int unique_rows_hint, double* out_val, double* out_grad, int* info);

/* B independent JaxTrainer.fit loops (src/trainer.py:162-228) with optax.adam(lr) restated
 * (b1,b2,eps as given; src/main.py:45) and the "fix p21" hook of trainer.py:133-160,205-210,218-220.
 * theta_unc_io is B x P UNCONSTRAINED (in: start / current iterate, out: iterate after the last step
 * of this call).  The fit may be split into chunks of steps [first_step, first_step + steps) of a
 * total_steps-long fit (with a collective in between); adam_state (B x 2P doubles: m then v) carries
 * the moments between calls and may be NULL only when the whole fit is one call.  out_hist
 * (B x ld_hist) receives the loss at every step at column first_step + s.  When the call reaches
 * total_steps, out_theta (B x P, may be NULL) receives constrain(theta_unc) with the constrained-space
 * hook of trainer.py:218-220 applied. */
int lfm_batched_fit(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                    double* theta_unc_io, double* adam_state, double jitter, double lr, double b1,
                    double b2, double eps, int first_step, int steps, int total_steps, int fix_params,
                    int steps_per_epoch, int unique_rows_hint, double* out_hist, int64_t ld_hist,
                    double* out_theta, int* info);

/* Device state of B fits in ONE launch: theta_unc = unconstrain(theta0) (src/trainer.py:75), adam_state (B x 2P, may be
 * NULL) = 0, hist (n_hist doubles, may be NULL) = NaN, info (B ints, may be NULL) = 0, keys (n_keys int64 words for
 * best_key / step_keys, may be NULL) = INT64_MAX. */
int lfm_batched_fit_init(lfm_stream_t stream, int64_t B, int G, const double* theta0, double* theta_unc,
                         double* adam_state, double* hist, int64_t n_hist, int* info, long long* keys, int64_t n_keys);

/* Time-grid variants of the two batched entry points: `time_grid_hint` is an upper bound on the number of
 * DISTINCT times among the rows of X (lfm_count_distinct_times; 0 = unknown).  With both hints set and
 * the problem inside the limits of the one-warp-per-LFM kernel (unique rows <= 36, G T^2 <= 2048), every
 * LFM is fitted by a single warp with the exp/erf pair terms tabulated once per step in shared memory;
 * otherwise the one-CTA-per-LFM kernel runs.  A hint smaller than the true count gives info = -2. */
int lfm_batched_nlml_grad_unc_tg(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X,
                                 const double* y, const double* theta_unc, double jitter, int unique_rows_hint,
                                 int time_grid_hint, double* out_val, double* out_grad, int* info);
int lfm_batched_fit_tg(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                       double* theta_unc_io, double* adam_state, double jitter, double lr, double b1, double b2,
                       double eps, int first_step, int steps, int total_steps, int fix_params,
                       int steps_per_epoch, int unique_rows_hint, int time_grid_hint, double* out_hist,
                       int64_t ld_hist, double* out_theta, int* info, long long* best_key, void* structure_cache);
/* Per-LFM observations: LFM b fits y + b * y_stride (y_stride >= N; 0 = every LFM fits the same y, which is what the
 * entry points above do).  X -- and with it the duplicate-row / time-grid structure -- stays shared, so this is the
 * batch over replicas, gene subsets of equal size and candidate transcription factors of north_star: same design
 * points, different expression data, independent hyper-parameters.  Everything else as lfm_batched_fit_tg /
 * lfm_batched_nlml_grad_unc_tg. */
int lfm_batched_fit_multi(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                          int64_t y_stride, double* theta_unc_io, double* adam_state, double jitter, double lr,
                          double b1, double b2, double eps, int first_step, int steps, int total_steps,
                          int fix_params, int steps_per_epoch, int unique_rows_hint, int time_grid_hint,
                          double* out_hist, int64_t ld_hist, double* out_theta, int* info, long long* best_key,
                          void* structure_cache);
int lfm_batched_nlml_grad_unc_multi(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X,
                                    const double* y, int64_t y_stride, const double* theta_unc, double jitter,
                                    int unique_rows_hint, int time_grid_hint, double* out_val, double* out_grad,
                                    int* info);
/* lfm_batched_fit_multi plus `step_keys` (may be NULL): total_steps device words, initialised to INT64_MAX by the caller;
 * word s receives atomicMin over the batch of the order-preserving image of every LFM's loss at optimiser step s (see
 * best_key below).  The best objective of EVERY step of a sharded fit is then ONE integer MIN all-reduce of that vector
 * after the launch, however many steps the launch ran -- the per-step reduction of north_star without a launch boundary
 * per step. */
int lfm_batched_fit_trace(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                          int64_t y_stride, double* theta_unc_io, double* adam_state, double jitter, double lr,
                          double b1, double b2, double eps, int first_step, int steps, int total_steps,
                          int fix_params, int steps_per_epoch, int unique_rows_hint, int time_grid_hint,
                          double* out_hist, int64_t ld_hist, double* out_theta, int* info, long long* best_key,
                          long long* step_keys, void* structure_cache);
/* The WHOLE fit (steps 0 .. total_steps) in one launch, with `queue_ws` (lfm_batched_queue_bytes() device bytes, may be
 * NULL = plain launch): the CTAs become persistent workers that take "the next chunk_steps steps of LFM b" tasks from a
 * device-side queue, so an LFM moves to whichever resident slot is free after every chunk.  The library uses the queue
 * when a static one-CTA-per-LFM assignment would be unbalanced (more LFMs than SMs, fewer than resident team slots, not
 * a whole number per SM -- e.g. the 512-LFM shard of 4096 restarts over 8 GPUs: 4 teams on 68 SMs and 3 on 80 for the
 * whole fit otherwise) and ignores it elsewhere; results do not depend on it beyond the rounding of Adam's running bias
 * products at chunk boundaries.  adam_state is required with a queue (the moments travel between workers through it);
 * the CTA-per-LFM fallback kernel ignores the queue.  LFM_BATCHED_QUEUE = 0 | 1 in the environment forces it off / on. */
size_t lfm_batched_queue_bytes(int64_t B, int total_steps, int chunk_steps);
int lfm_batched_fit_queue(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                          int64_t y_stride, double* theta_unc_io, double* adam_state, double jitter, double lr,
                          double b1, double b2, double eps, int total_steps, int fix_params, int steps_per_epoch,
                          int unique_rows_hint, int time_grid_hint, double* out_hist, int64_t ld_hist,
                          double* out_theta, int* info, long long* best_key, long long* step_keys,
                          void* structure_cache, int chunk_steps, void* queue_ws, size_t queue_bytes);
/* structure_cache (may be NULL): lfm_batched_structure_bytes() device bytes the caller keeps between the calls of ONE
 * chunked fit.  The call with first_step == 0 stores the structure of X (duplicate rows, distinct times and time
 * differences, pair table) there; calls with first_step > 0 load it instead of repeating the O(N^2) scans. */
size_t lfm_batched_structure_bytes(int64_t N, int G, int unique_rows_hint, int time_grid_hint);
/* ---- batched fits with measurement variances: the heteroscedastic objective of lfm_nlml_grad_unc_het_tg ------------
 * Sigma = K + diag(v) + (jitter + sigma^2) I, i.e. noise c_i = v_i + jitter + sigma^2 per point.  `variances` is N
 * device doubles shared by every LFM (var_stride 0) or one row per LFM at variances + b * var_stride (var_stride >= N),
 * as y / y_stride; NULL means exactly lfm_batched_nlml_grad_unc_multi / lfm_batched_fit_trace / _fit_queue.
 * The duplicate-row compression stays exact with a noise per point (same rule for U and R as above): per unique row u
 *   omega_u = sum_{i in u} 1/c_i, omega2_u = sum_{i in u} 1/c_i^2, cbar_u = R / omega_u, q_u = cbar_u sum_{i in u} z_i/c_i,
 *   M = diag(cbar) + R K_u,  beta = M^-1 q = P^T alpha,  K_u beta = (q - cbar o beta) / R,
 *   log det Sigma = sum_i log c_i - sum_u log cbar_u + log det M,
 *   z^T Sigma^-1 z = sum_i z_i^2/c_i - sum_u (q_u/cbar_u) (K_u beta)_u,
 *   P^T Kbar P = 1/2 (R M^-1 - beta beta^T) (the kernel-parameter weights: unchanged),
 *   diag(P^T Kbar P K_u)_u = 1/2 (1 - cbar_u M^-1_uu - beta_u (K_u beta)_u),   alpha_i = (z_i - (K_u beta)_u(i)) / c_i,
 *   tr Sigma^-1 = sum_i 1/c_i - sum_u omega2_u/omega_u + R sum_u omega2_u M^-1_uu / omega_u^2,
 *   dNLML/dsigma = sigma (tr Sigma^-1 - alpha^T alpha);
 * with v = 0 every line is the homoscedastic one.  Every c_i must be > 0: otherwise (or with NaN variances) info = 1 and
 * the loss / gradient are NaN, as for a failed factorisation. */
int lfm_batched_nlml_grad_unc_het(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                                  int64_t y_stride, const double* variances, int64_t var_stride,
                                  const double* theta_unc, double jitter, int unique_rows_hint, int time_grid_hint,
                                  double* out_val, double* out_grad, int* info);
/* lfm_batched_fit_trace with variances; with `queue_ws` non-NULL it is lfm_batched_fit_queue instead (then first_step must
 * be 0 and steps == total_steps: the queue runs the whole fit). */
int lfm_batched_fit_het(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                        int64_t y_stride, const double* variances, int64_t var_stride, double* theta_unc_io,
                        double* adam_state, double jitter, double lr, double b1, double b2, double eps, int first_step,
                        int steps, int total_steps, int fix_params, int steps_per_epoch, int unique_rows_hint,
                        int time_grid_hint, double* out_hist, int64_t ld_hist, double* out_theta, int* info,
                        long long* best_key, long long* step_keys, void* structure_cache, int chunk_steps,
                        void* queue_ws, size_t queue_bytes);
/* ---- batched posteriors: latent_predict / multi_gene_predict of B fitted LFMs in one launch ---------------------------
 * B LFMs share X (N <= 128 rows) and the test inputs Xstar (T* rows); LFM b has its own CONSTRAINED theta (theta +
 * b * P), observations (y, y_stride) and variances (variances, var_stride), with the meaning of lfm_batched_fit_het
 * (stride 0: shared; N or more: one row per LFM).  `variances` is required, as for lfm_latent_posterior.  The
 * duplicate-row compression of the batched fits (same rule for U and R, unique_rows_hint as there) with a noise c_i
 * per point: omega_u = sum_{i in u} 1/c_i, cbar_u = R / omega_u, q_u = cbar_u sum_{i in u} z_i / c_i,
 * M = diag(cbar) + R K_u = L L^T, beta = M^-1 q = P^T alpha, and P^T Sigma^-1 P = R M^-1.  With k_*u the
 * cross-covariance of a test row with the U unique rows (the flag-aware pair function of lfm_cross_covariance):
 *   latent (c_i = v_i + jitter):   mean = mean_t + k_*u^T beta,  var = k(t*,t*) + 2 jitter - R ||L^-1 k_*u||^2;
 *   gene   (c_i = v_i + sigma^2):  mean = mean_t + k_*u^T beta,  cov = K_tt - R V^T V + jitter I, V = L^-1 K_ut,
 *                                  var = diag(cov);
 * mean_t, k(t*,t*) and the positional blocks T* / G as lfm_latent_posterior / lfm_gene_posterior.  Outputs are B x T*
 * (out_mean, out_var) and B x T* x T* (out_cov, may be NULL; out_var of the gene posterior may be NULL too); info
 * (B ints): 0, k > 0 the failing pivot of M, 1 some c_i <= 0 or NaN, -1 unique_rows_hint smaller than U.  A failed LFM
 * gets NaN outputs and affects no other.  LFM b's outputs are bit-identical whatever B is and wherever b sits.  The
 * workspace (lfm_batched_posterior_workspace_bytes, full_cov = out_cov != NULL) holds the structure of X and, with
 * the full covariance, V of every LFM (B x U x T* doubles).  N > 128: LFM_ERR_UNSUPPORTED; Tstar % G must be 0 for the
 * gene posterior. */
size_t lfm_batched_posterior_workspace_bytes(int64_t B, int64_t N, int G, int64_t Tstar, int unique_rows_hint,
                                             int full_cov);
int lfm_batched_latent_posterior(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                                 int64_t y_stride, const double* variances, int64_t var_stride, const double* theta,
                                 double jitter, int64_t Tstar, const double* Xstar, int unique_rows_hint, void* ws,
                                 size_t ws_bytes, double* out_mean, double* out_var, int* info);
int lfm_batched_gene_posterior(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                               int64_t y_stride, const double* variances, int64_t var_stride, const double* theta,
                               double jitter, int64_t Tstar, const double* Xstar, int unique_rows_hint, void* ws,
                               size_t ws_bytes, double* out_mean, double* out_cov, double* out_var, int* info);

/* best_key (may be NULL): one device word that receives atomicMin over the batch of the order-preserving integer
 * image of each LFM's loss after the last step of this call (finite losses only; initialise it to INT64_MAX).
 * key(v) = bits(v) for v >= 0, bits(v) ^ 0x7fff...f otherwise -- monotone in v, so the global best objective of a
 * chunk of steps is ONE integer MIN all-reduce of that word across ranks (north_star: "one NCCL allreduce of
 * best-objective ... state per step"). */

/* Warps per LFM the batched entry points use for a batch of B LFMs of this shape on the current device: 1 (one warp per
 * LFM, register-resident Cholesky; a full GPU), 4 (a team of four warps per LFM, symmetric sweep in register tiles;
 * shards that leave SMs idle, e.g. 4096 restarts over 8 GPUs), or 0 when the shape runs the CTA-per-LFM kernel.
 * LFM_BATCHED_TEAM = 1 | 4 | 8 in the environment overrides the choice (measurements).  The answer is for the entry
 * points without variances: the _het ones keep N + 2U more doubles per LFM in shared memory and choose from their own
 * occupancy. */
int lfm_batched_team_size(int64_t B, int64_t N, int G, int unique_rows_hint, int time_grid_hint);

/* Winner of a shard after a fit: out_packed (P + 2 doubles) = [loss, id, theta(P)] of the LFM with the smallest FINITE
 * hist[b * ld_hist + col] (ties: smallest b), id = id0 + b; [inf, -1, inf...] when no loss is finite.  One launch of
 * one CTA; what multi_start_fit all-gathers across ranks (P + 2 doubles per rank). */
int lfm_batched_best(lfm_stream_t stream, int64_t B, int P, const double* hist, int64_t ld_hist, int64_t col,
                     const double* theta, double id0, double* out_packed);

/* ---- collective of the sharded batched path (SURVEY.md 8b / 8e) --------------------------------------------------
 * A holder of one ncclComm_t with the two collectives the path has: the integer MIN all-reduce of the best-objective
 * keys (best_key / step_keys above; in place, stream-ordered, 8 bytes per chunk or per step) and the all-gather of the
 * per-rank winners (lfm_batched_best, P + 2 doubles per rank).  NCCL is bound at run time (dlopen libnccl.so.2, or the
 * path in LFM_NCCL_LIB): the library itself links against libcudart only; without NCCL these return LFM_ERR_COMM.
 * Rank 0 calls lfm_comm_unique_id and ships the LFM_COMM_ID_BYTES bytes to the other ranks by any means (a file, a TCP
 * store, torch.distributed); every rank then calls lfm_comm_create on its own device (collective call). */
#define LFM_COMM_ID_BYTES 128
typedef struct lfm_comm lfm_comm;
int lfm_comm_available(void);
int lfm_comm_unique_id(void* id_out);
int lfm_comm_create(lfm_comm** out, int world, int rank, const void* id_bytes);
int lfm_comm_world(const lfm_comm* c);
int lfm_comm_rank(const lfm_comm* c);
int lfm_comm_allreduce_min_i64(lfm_comm* c, long long* buf, size_t count, lfm_stream_t stream);
int lfm_comm_allgather_f64(lfm_comm* c, const double* send, double* recv, size_t count, lfm_stream_t stream);
int lfm_comm_destroy(lfm_comm* c);

/* ---- host-buffer entry points (H2D / D2H inside; what a ctypes/cgo caller with numpy arrays
 * binds).  They allocate device scratch on first use per (N,G) and cache it in a handle. -------- */

/* ---- evaluation plans -------------------------------------------------------------------------
 * One lfm_nlml_grad[_unc]_tg evaluation over FIXED device buffers, captured once as a CUDA graph (the ~140
 * launches and ~70 cross-stream event edges of an N = 4000 evaluation replay with ~1 us between dependent
 * kernels).  A fit loop writes the next theta into the bound `theta` buffer and launches the plan again
 * (src/trainer.py:201-216 evaluates the same (X, y) at every step).  create runs the evaluation once eagerly
 * (validation, lazy initialisation) and synchronises; launch is stream-ordered and never synchronises. */
typedef struct lfm_plan lfm_plan;
int lfm_nlml_grad_plan_create(lfm_plan** out_plan, int64_t N, int G, const double* X, const double* y,
                              const double* theta, double jitter, int64_t time_grid, int unconstrained, void* ws,
                              size_t ws_bytes, double* out, int* info);
/* same with the heteroscedastic objective: `variances` (N device doubles, bound like X and y) or NULL */
int lfm_nlml_grad_plan_create_het(lfm_plan** out_plan, int64_t N, int G, const double* X, const double* y,
                                  const double* variances, const double* theta, double jitter, int64_t time_grid,
                                  int unconstrained, void* ws, size_t ws_bytes, double* out, int* info);
int lfm_plan_launch(lfm_plan* plan, lfm_stream_t stream);
int lfm_plan_destroy(lfm_plan* plan);

typedef struct lfm_handle lfm_handle;
int lfm_handle_create(lfm_handle** out);
int lfm_handle_destroy(lfm_handle* h);

int lfm_nlml_grad_host(lfm_handle* h, int64_t N, int G, const double* X, const double* y,
                       const double* theta, double jitter, int unconstrained, double* out, int* info);
/* heteroscedastic objective from host buffers: `variances` N host doubles or NULL (= lfm_nlml_grad_host) */
int lfm_nlml_grad_het_host(lfm_handle* h, int64_t N, int G, const double* X, const double* y, const double* variances,
                           const double* theta, double jitter, int unconstrained, double* out, int* info);
int lfm_latent_posterior_host(lfm_handle* h, int64_t N, int G, const double* X, const double* y,
                              const double* variances, const double* theta, double jitter,
                              int64_t Tstar, const double* Xstar, double* out_mean, double* out_var,
                              int* info);
int lfm_batched_fit_host(lfm_handle* h, int64_t B, int64_t N, int G, const double* X, const double* y,
                         const double* theta0, double jitter, double lr, double b1, double b2,
                         double eps, int steps, int fix_params, int steps_per_epoch, double* out_theta,
                         double* out_hist, int* info);
/* lfm_batched_fit_host with measurement variances (N host doubles, staged in the same single host->device copy as X, y
 * and theta0; the objective of lfm_batched_fit_het) or NULL (= lfm_batched_fit_host). */
int lfm_batched_fit_het_host(lfm_handle* h, int64_t B, int64_t N, int G, const double* X, const double* y,
                             const double* variances, const double* theta0, double jitter, double lr, double b1,
                             double b2, double eps, int steps, int fix_params, int steps_per_epoch, double* out_theta,
                             double* out_hist, int* info);

/* ---- diagnostics used by bench.py for the roofline denominators ------------------------------ */

/* Plain C = A B^T fp64 GEMM through the library's own DMMA kernel (M,N % 128 == 0, K % 16 == 0). */
int lfm_debug_dgemm_nt(lfm_stream_t stream, int64_t M, int64_t N, int64_t K, const double* A,
                       const double* B, double* C);
/* Every launch the dense path's DMMA GEMM can make: C = alpha op(A) op(B) + beta C, row-major, the fields of the
 * library's internal launch descriptor (csrc/lfm_common.cuh, LfmGemm).  transA = 1: A stored K x M; transB = 1: B stored
 * N x K.  kmode restricts each output tile's k-range: 0 full, 1 k < row tile end, 3 k >= row tile start, 4 k >= max(row,
 * column) tile start, 5 as 4 for the tile rows >= k_split and k in [k_split, K) accumulating (beta = 1) above them.  The
 * range is then clipped to [k_lo, k_hi) (multiples of 16); with beta = 1 and alpha = +-1, a tile whose range is empty is
 * left untouched.  lower_only skips the tiles above the diagonal and, with tri_skip, those of the first tri_skip rows.
 * batch > 1 runs problem y at A + y strideA, B + y strideB, C + y strideC.  tile: 0 heuristic, 1 16 x 128, 2 128 x 128,
 * 3 64 x 64 tiles.  LFM_ERR_INVALID before any launch for a base pointer that is not 16-byte aligned or an odd leading
 * dimension or stride.  *variant receives the instantiation that ran, TA TBN WM WN GM as decimal digits (0 if none). */
typedef struct lfm_gemm_desc {
  int transA, transB;
  int64_t M, N, K;
  const double* A; int64_t lda;
  const double* B; int64_t ldb;
  double* C; int64_t ldc;
  double alpha, beta;
  int lower_only, kmode, batch;
  int64_t strideA, strideB, strideC;
  int tile, tri_skip;
  int64_t k_split, k_lo, k_hi;
} lfm_gemm_desc;
int lfm_debug_dgemm(lfm_stream_t stream, const lfm_gemm_desc* desc, int* variant);
/* In-place dense lower Cholesky / inverse of an n x n row-major matrix (n % 128 == 0): after the
 * call A holds L (lower), and if Sinv != NULL it receives Sigma^-1 (lower triangle valid).
 * W is an n x n scratch matrix. */
int lfm_debug_potrf_potri(lfm_stream_t stream, int64_t n, double* A, double* W, double* Sinv, int* info);
/* The same factorisation and inverse in the sequence the NLML gradient runs: W = L^-1 (lower), diag(L) into ldiag
 * (n doubles), Sigma^-1 = W^T W started early where the sweep does so, and after the call A holds Sigma^-1 (lower
 * triangle valid).  chain_ready != 0: info is zeroed and an event recorded on `stream`, and the factorisation's chain
 * starts behind that event, as behind the first two block columns of Sigma (one-sweep sizes: n / 128 a power of two,
 * 4 <= n / 128 <= 32; ignored otherwise).  *early_done (host int, may be NULL) receives 1 when Sigma^-1 was finished by
 * the late half of the product (lfm_lauum_late) and 0 when by one full product. */
int lfm_debug_potrf_potri_eval(lfm_stream_t stream, int64_t n, double* A, double* W, double* ldiag, int chain_ready,
                               int* early_done, int* info);
/* C (lower tiles, m x m) -= P P^T, P m x K: the trailing update of the blocked Cholesky (roofline helper). */
int lfm_debug_syrk(lfm_stream_t stream, int64_t m, int64_t K, const double* P, int64_t ldp, double* C, int64_t ldc);
/* The same launch with 8 debug words per CTA in `stamps` (tiles of the launch x 8 int64): [0] SM id, clock64 at [1] entry,
 * [2] first operand unit landed, [3] last DMMA issued, [4] stores issued, [7] address set-up done (nothing requested yet);
 * globaltimer at [5] entry and [6] exit (tools/tile_life.py). */
int lfm_debug_syrk_stamps(lfm_stream_t stream, int64_t m, int64_t K, const double* P, int64_t ldp, double* C, int64_t ldc,
                          long long* stamps);

/* One 128 x 128 leaf factorisation with clock64() stamps at its phase boundaries (16 values). */
int lfm_debug_leaf_profile(lfm_stream_t stream, double* A, double* W, int* info, long long* stamps);
/* clock64 stamps at the phase boundaries of the second optimiser step of LFM 0 (warp-per-LFM kernel; tools/). */
int lfm_debug_batched_stamps(lfm_stream_t stream, int64_t B, int64_t N, int G, const double* X, const double* y,
                             double* theta_unc_io, double* adam_state, double jitter, int steps, int unique_rows_hint,
                             int time_grid_hint, double* out_hist, int* info, long long* stamps);
/* Number of CUDA kernels this library has launched since load (bench.py's gpu_launches). */
unsigned long long lfm_debug_launch_count(void);
/* Bracket every DMMA GEMM launch with CUDA events on its stream between begin and end; end
 * synchronises the device and reports the kernel time, the flops the tiles executed and the number of
 * launches.  Launches on the factorisation's streams overlap: the time is the length of the UNION of the
 * launch intervals (lfm_debug_profile_sum_ms gives the plain sum). */
int lfm_debug_profile_begin(void);
int lfm_debug_profile_end(double* total_ms, double* exec_flops, long long* launches);
double lfm_debug_profile_sum_ms(void);
/* the last session grouped by tile variant, as a JSON list (launches, summed launch time, executed flops per variant);
 * copies at most n - 1 characters into out and returns the full length */
size_t lfm_debug_profile_variants(char* out, size_t n);
/* the 16 x 128-tile launches of the factorisation's look-ahead chain, accounted separately (call after _end) */
int lfm_debug_profile_chain(double* total_ms, double* exec_flops, long long* launches);

#ifdef __cplusplus
}
#endif
#endif /* LFM_B200_H */
