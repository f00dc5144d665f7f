/*
 * elfi_b200.h -- C ABI of libelfi_b200.so: the B200 (sm_100a) implementation of ELFI's
 * data-parallel sampler / BOLFI hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  ELFI is pure Python: the binding a
 * maintainer adds on the reference side is a ctypes stub (see INTEGRATION.md) called from
 * the node operations that `elfi.executor.Executor._run` invokes (elfi/executor.py:143-159)
 * and from the sampler bookkeeping in elfi/methods/inference/samplers.py.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error (ELFI_B200_ERR_*); the message for
 *     the calling host thread is available from elfi_b200_last_error();
 *   - all array arguments are caller-allocated DEVICE pointers unless the name ends in
 *     `_host`; matrices are row-major with a leading dimension given in ELEMENTS;
 *   - sizes are int64_t; `stream` is a cudaStream_t passed as void* (NULL = legacy default
 *     stream); kernels are asynchronous on that stream;
 *   - the context owns only scratch memory; it never takes ownership of caller buffers;
 *   - one context per device; a context may be used by one host thread and one stream at a
 *     time (its scratch arena is ordered by that stream; growing it synchronises the device).
 */
#ifndef ELFI_B200_H
#define ELFI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ELFI_B200_VERSION 100

#define ELFI_B200_OK 0
#define ELFI_B200_ERR_ARG (-1)     /* invalid argument (shape, alignment, NULL) */
#define ELFI_B200_ERR_CUDA (-2)    /* a CUDA runtime / driver call failed */
#define ELFI_B200_ERR_NOMEM (-3)   /* scratch allocation failed */
#define ELFI_B200_ERR_UNSUPPORTED (-4)

#define ELFI_B200_MAX_NESTED 32    /* max nested distance columns K */

typedef struct elfi_b200_ctx elfi_b200_ctx;

/* ---- context ------------------------------------------------------------------------ */

int elfi_b200_version(void);
const char* elfi_b200_last_error(void);

/* Creates the context of CUDA device `device` (must be compute capability 10.x). */
int elfi_b200_ctx_create(int device, elfi_b200_ctx** out);
int elfi_b200_ctx_destroy(elfi_b200_ctx* ctx);
/* Number of SMs of the context's device (grid sizing is a multiple of this). */
int elfi_b200_ctx_sm_count(const elfi_b200_ctx* ctx);

/* ---- single-process multi-GPU exchange ----------------------------------------------------
 * The per-generation all-gather of accepted particles / weights (SURVEY.md section 8e; the
 * reference merges the batches of its workers in the master, samplers.py:140-237) for a process
 * that drives several GPUs itself (one context per GPU, e.g. the thread-per-GPU client): GPU g
 * contributes send[g] (rows x width doubles in ITS memory) and receives the context-ordered
 * concatenation (n_ctx * rows x width) in recv[g].  ctxs / send / recv / streams are HOST arrays
 * of n_ctx entries; streams[g] is the stream of GPU g on which send[g] was produced and on which
 * recv[g] is consumed afterwards (the call only enqueues copies and event waits).  Copies are
 * peer-to-peer (NVLink when peer access can be enabled, otherwise staged by the driver).
 * One-process-per-GPU runs use torch.distributed / NCCL instead (DESIGN.md section 5). */
int elfi_b200_allgather_particles(elfi_b200_ctx* const* ctxs, int64_t n_ctx,
                                  const double* const* send, int64_t rows, int64_t width,
                                  double* const* recv, void* const* streams);

/* ---- distance + acceptance ------------------------------------------------------------
 * Replaces, for the Euclidean family, the body of
 *   elfi/model/utils.py:37-52        distance_as_discrepancy  (column_stack + dist + flatten)
 *   elfi/model/elfi_model.py:1037    Distance -> scipy.spatial.distance.cdist(X, obs, 'euclidean')
 *   elfi/model/elfi_model.py:1135-1151  AdaptiveDistance.nested_distance (K weighted columns)
 * and the acceptance test of
 *   elfi/methods/inference/samplers.py:223-225   accepted = all_k(d[:, k] <= thr[k])
 *
 *   d[i, k] = sqrt( sum_j  W[k, j] * (S[i, j] - obs[j])^2 ),   j = 0 .. D-1 strictly in order,
 * every multiply and add rounded separately in fp64 (SciPy's order: bit-identical results).
 *
 *   S        (B, D) row-major, leading dimension ldS (elements)
 *   obs      (D)
 *   W        (K, D) row-major weights (cdist's `w`, i.e. 1/scale^2), or NULL = unweighted
 *            (K must then be 1; a row of ones is bit-identical to the unweighted form)
 *   K        number of nested distance columns, 1 <= K <= ELFI_B200_MAX_NESTED
 *   thr_host HOST pointer to K thresholds, or NULL = no acceptance test
 *   d_out    (B, K) row-major distances
 *   acc_idx  int32[B] ascending indices of accepted rows, or NULL (requires thr_host)
 *   n_acc    device int64[1] number of accepted rows (written when thr_host != NULL), or NULL
 */
int elfi_b200_dist_euclid_thr_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                  int64_t D, const double* obs, const double* W, int64_t K,
                                  const double* thr_host, double* d_out, int32_t* acc_idx,
                                  int64_t* n_acc, void* stream);

/* Same with the K thresholds in DEVICE memory (thr_dev, not NULL): a threshold that was itself
 * computed on the device -- the weighted quantile of the previous population
 * (samplers.py:542-549), the running n-th best distance of the buffer (samplers.py:243) -- feeds
 * the next distance call without a host round trip. */
int elfi_b200_dist_euclid_thr_dev_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                      int64_t D, const double* obs, const double* W, int64_t K,
                                      const double* thr_dev, double* d_out, int32_t* acc_idx,
                                      int64_t* n_acc, void* stream);

/* Distances + acceptance AND the per-column moments of the same batch from ONE read of S:
 * AdaptiveDistance evaluates its K nested columns (elfi_model.py:1135-1151) and then feeds the
 * batch to add_data (elfi_model.py:1104-1125); the reference reads S K + 1 times for that.
 * moments (2, D) device: row 0 = column means of the batch, row 1 = M2 = sum_i (x_ij - mean_j)^2
 * (what elfi_b200_colmoments_f64 returns; Chan-merged into (n, mean, M2) by the caller).
 * Thresholds: thr_host or thr_dev (at most one non-NULL; both NULL = no acceptance test).
 * W may be NULL only when the stand-alone moments pass is acceptable (the fused kernel is the
 * weighted / nested row stream; pass a row of ones for plain Euclidean distances). */
int elfi_b200_dist_euclid_mom_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                  int64_t D, const double* obs, const double* W, int64_t K,
                                  const double* thr_host, const double* thr_dev, double* d_out,
                                  int32_t* acc_idx, int64_t* n_acc, double* moments, void* stream);

/* Same computation with HOST buffers (pageable or pinned): rows are streamed to the device
 * in chunks on two copy streams overlapped with the kernel; distances, accepted indices
 * and the count are copied back.  Blocks until the results are in host memory.
 * d_out_host may be NULL (then only accepted indices / count come back). */
int elfi_b200_dist_euclid_thr_f64_host(elfi_b200_ctx* ctx, const double* S_host, int64_t ldS,
                                       int64_t B, int64_t D, const double* obs_host,
                                       const double* W_host, int64_t K, const double* thr_host,
                                       double* d_out_host, int32_t* acc_idx_host,
                                       int64_t* n_acc_host);

/* Other cdist metrics that elfi.Distance forwards to SciPy (elfi/model/elfi_model.py:1016-1037):
 *   SQEUCLIDEAN  sum_j (S_ij - obs_j)^2          CITYBLOCK  sum_j |S_ij - obs_j|
 *   CHEBYSHEV    max_j |S_ij - obs_j|            MINKOWSKI  (sum_j |S_ij - obs_j|^pexp)^(1/pexp)
 * accumulated left to right in fp64 like SciPy does (the first three are bit-identical to cdist,
 * Minkowski to the accuracy of pow).  Unweighted, one distance column; otherwise the arguments and
 * the acceptance outputs are those of elfi_b200_dist_euclid_thr_f64 (d_out has B entries). */
#define ELFI_B200_METRIC_SQEUCLIDEAN 1
#define ELFI_B200_METRIC_CITYBLOCK 2
#define ELFI_B200_METRIC_CHEBYSHEV 3
#define ELFI_B200_METRIC_MINKOWSKI 4
int elfi_b200_dist_metric_thr_f64(elfi_b200_ctx* ctx, int32_t metric, double pexp, const double* S,
                                  int64_t ldS, int64_t B, int64_t D, const double* obs,
                                  const double* thr_host, double* d_out, int32_t* acc_idx,
                                  int64_t* n_acc, void* stream);

/* cdist(S, obs, 'seuclidean', V=V) (elfi/model/elfi_model.py:1016-1037 with the V keyword of the
 * Distance docstring, elfi_model.py:996-1003): d_i = sqrt(sum_j (S_ij - obs_j)^2 / V_j) in the
 * summation order of SciPy's compiled loop -- two running sums over the even and the odd columns of
 * the first D - D%2 columns, their sum, then the last term when D is odd -- with an IEEE division
 * per term, so the result is bit-identical to cdist.  V (D) device, strictly positive.  Other
 * arguments and the acceptance outputs as for elfi_b200_dist_metric_thr_f64. */
int elfi_b200_dist_seuclidean_thr_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                      int64_t D, const double* obs, const double* V,
                                      const double* thr_host, double* d_out, int32_t* acc_idx,
                                      int64_t* n_acc, void* stream);

/* ---- summary statistics ----------------------------------------------------------------
 * Row-wise summaries with NumPy's pairwise summation order (bit-identical results).
 *
 * elfi_b200_summary_autocov_f64 replaces elfi/examples/ma2.py:40-59 (autocov):
 *   out[i*ld_out + l] = mean_j( X[i, j+lag_l] * X[i, j] ),  j = 0 .. n-lag_l-1
 * for every lag in lags_host (HOST int32 array, 1 <= lag < n).  All lags of a call are
 * evaluated from one pass over X where possible (lags {1,2} fused), and written straight
 * into the column-stacked (B, nlags) summary matrix that the distance kernel consumes
 * (this is the np.column_stack of elfi/model/utils.py:39, done for free).
 *
 * elfi_b200_summary_meanvar_f64 replaces elfi/examples/gauss.py:142-173 (ss_mean, ss_var):
 *   out[i*ld_out + col_mean] = np.mean(X[i]),  out[i*ld_out + col_var] = np.var(X[i])
 * (either column index may be -1 to skip that statistic).
 */
int elfi_b200_summary_autocov_f64(elfi_b200_ctx* ctx, const double* X, int64_t ldX, int64_t B,
                                  int64_t n, const int32_t* lags_host, int64_t nlags, double* out,
                                  int64_t ld_out, void* stream);
int elfi_b200_summary_meanvar_f64(elfi_b200_ctx* ctx, const double* X, int64_t ldX, int64_t B,
                                  int64_t n, double* out, int64_t ld_out, int32_t col_mean,
                                  int32_t col_var, void* stream);

/* ---- ordering primitives ---------------------------------------------------------------
 * elfi_b200_sort_pairs_f64: stable ascending argsort of n fp64 keys (NaN last).  Replaces
 * np.argsort in Rejection._merge_batch (elfi/methods/inference/samplers.py:232-237) and in
 * weighted_sample_quantile (elfi/methods/utils.py:397).  keys_sorted and perm may each be
 * NULL.  (NumPy's default argsort is unstable; the two agree whenever keys are distinct.)
 *
 * elfi_b200_gather_rows_f64: dst[i, 0:width] = src[idx[i], 0:width] -- the fancy-index
 * permutation `v[:] = v[sort_mask]` / `batch[node][accepted]` (samplers.py:228-237).
 *
 * elfi_b200_gather2_rows_f64: same from the virtual concatenation [A (nA rows); B], where B
 * rows may be indirected through mapB (the accepted indices of the new batch): the running
 * top-n merge without materialising the (n + batch) buffers of samplers.py:196-205.
 * perm == NULL means the identity.
 *
 * elfi_b200_accept_append_f64: `v[-num_accepted:] = batch[node][accepted]` for every output node
 * (samplers.py:228-230) with the counts read ON THE DEVICE, so a threshold-mode batch needs no
 * host round trip between the distance kernel and the merge: rows acc_idx[0 .. *n_acc) (acc_idx
 * == NULL: rows 0 .. *n_acc) of n_src <= 8 source arrays (src_host[k] = device pointer of a
 * (B, width_host[k]) array with leading dimension ld_src_host[k]; the three descriptor arrays
 * themselves are HOST arrays) are written side by side behind row *count of the packed candidate
 * buffer dst (capacity rows); *count += rows appended; rows that do not fit are dropped and
 * counted in *dropped (may be NULL).  n_acc, count, dropped are DEVICE int64.  max_rows bounds
 * *n_acc (sizes the launch).  The best n rows are taken once, when the population is extracted
 * (sort_pairs on the distance column + gather_rows) -- the same rows the reference's per-batch
 * argsort over n + batch_size rows leaves in its buffer (samplers.py:232-237).
 */
int elfi_b200_sort_pairs_f64(elfi_b200_ctx* ctx, const double* keys, int64_t n,
                             double* keys_sorted, int32_t* perm, void* stream);
int elfi_b200_gather_rows_f64(elfi_b200_ctx* ctx, const double* src, int64_t ld_src,
                              const int32_t* idx, int64_t n, int64_t width, double* dst,
                              int64_t ld_dst, void* stream);
int elfi_b200_accept_append_f64(elfi_b200_ctx* ctx, const int32_t* acc_idx, const int64_t* n_acc,
                                int64_t max_rows, int64_t n_src, const double* const* src_host,
                                const int64_t* ld_src_host, const int64_t* width_host, double* dst,
                                int64_t ld_dst, int64_t capacity, int64_t* count, int64_t* dropped,
                                void* stream);
/* One batch of a threshold-mode rejection round in one call (Rejection.update ->
 * _merge_batch, samplers.py:140-230): elfi_b200_dist_euclid_thr[_dev]_f64 followed by
 * elfi_b200_accept_append_f64 of the rows [d (K columns) | extra sources] -- four launches, no
 * synchronisation, one host -> library transition.  Exactly one of thr_host / thr_dev is given. */
int elfi_b200_rejection_batch_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B,
                                  int64_t D, const double* obs, const double* W, int64_t K,
                                  const double* thr_host, const double* thr_dev, double* d_out,
                                  int32_t* acc_idx, int64_t* n_acc, int64_t n_extra,
                                  const double* const* extra_host, const int64_t* ld_extra_host,
                                  const int64_t* width_extra_host, double* dst, int64_t ld_dst,
                                  int64_t capacity, int64_t* count, int64_t* dropped, void* stream);
int elfi_b200_gather2_rows_f64(elfi_b200_ctx* ctx, const double* A, int64_t ldA, int64_t nA,
                               const double* B, int64_t ldB, const int32_t* mapB,
                               const int32_t* perm, int64_t n, int64_t width, double* dst,
                               int64_t ld_dst, void* stream);

/* elfi_b200_topn_merge_f64: Rejection._merge_batch (samplers.py:226-237) in one call.  The
 * reference appends the accepted rows of a batch behind its best-n buffers, argsorts the distance
 * column over n + batch rows and permutes every output; here the virtual concatenation
 *     [A (nA rows of the current best-n) ; B[mapB] (nB accepted rows of the batch, mapB NULL = 0..nB-1)]
 * is ranked by its keys (keysA / keysB: the LAST distance column, addressed with a leading
 * dimension so that a column of a (rows, K) matrix can be passed in place; stable, NaN last) and
 * the n_keep smallest rows of each of the n_out outputs are gathered from their two sources:
 *     dst_host[k] (n_keep, width_host[k]) <- rows of A_host[k] (nA, width) / B_host[k] (batch, width).
 * The seven descriptor arrays are HOST arrays of length n_out; destinations must not alias sources.
 * merge_keys + 8-bit radix passes + one gather per output on `stream`, no synchronisation. */
int elfi_b200_topn_merge_f64(elfi_b200_ctx* ctx, const double* keysA, int64_t ld_keysA, int64_t nA,
                             const double* keysB, int64_t ld_keysB, const int32_t* mapB, int64_t nB,
                             int64_t n_keep, int64_t n_out, const double* const* A_host,
                             const int64_t* ldA_host, const double* const* B_host,
                             const int64_t* ldB_host, const int64_t* width_host,
                             double* const* dst_host, const int64_t* ld_dst_host, void* stream);

/* elfi_b200_wquantile_f64: weighted_sample_quantile (elfi/methods/utils.py:379-411).
 *   x (n), w (n) or NULL (equal weights), 0 <= alpha <= 1.
 *   out[0] = alpha-quantile (an element of x), out[1] = its rank in sorted order (as double).
 * np.sum (pairwise) and np.cumsum (sequential) are reproduced in the reference's order, so
 * the selected element is identical even when alpha falls exactly on a cumulative weight
 * (equal weights + round alpha, the normal case in SMC round 0).  A parallel scan with a rigorous
 * error bound answers first; the sequential kernel only runs when alpha is within that bound of a
 * cumulative weight.  With w == NULL the position follows in closed form from n and alpha (the
 * sequential sum of n copies of 1/n is an arithmetic progression per binade) and nothing is
 * scanned.  The call synchronises `stream` unless w == NULL. */
int elfi_b200_wquantile_f64(elfi_b200_ctx* ctx, const double* x, const double* w, int64_t n,
                            double alpha, double* out, void* stream);

/* ---- SMC population arithmetic ---------------------------------------------------------
 * elfi_b200_colmoments_f64: per-column mean and M2 = sum_i (x_ij - mean_j)^2 of one (B, D)
 * batch: out[0:D] = mean, out[D:2D] = M2.  The host merges batches with Chan's formula,
 * which is algebraically AdaptiveDistance.add_data (elfi/model/elfi_model.py:1104-1125);
 * parity is tolerance-level (the reference itself only promises np.std agreement,
 * tests/unit/test_elfi_model.py:185-253).
 *
 * elfi_b200_weighted_stats_f64: weighted_var and its ingredients (elfi/methods/utils.py:108-139):
 *   stats = [V1 = sum w, V2 = sum w^2, xbar_0..p-1 = np.average(x, weights=w),
 *            s2_0..p-1 = sum w (x - xbar)^2 / (V1 - V2/V1)],   w == NULL means all ones.
 *
 * elfi_b200_gm_logpdf_f64: GMDistribution.logpdf (elfi/methods/utils.py:146-197) --
 *   logq[i] = log sum_j (w_j / sum w) N(x_i; means_j, Sigma), plain sum of densities as in the
 *   reference (no log-sum-exp shift), Sigma shared.  Linv_host = inverse of the lower Cholesky
 *   factor of Sigma (HOST, p x p row-major), logdet = log det Sigma.  p <= 16.
 *   Tolerance: <= 1e-8 relative on q (range-reduced exp with a degree-6 minimax polynomial, max
 *   term error 1.9e-9; fp64 accumulation).
 * elfi_b200_gm_logpdf_mixed_f64: the same density with 2^f taken from the special-function unit in
 *   fp32 (range reduction and accumulation stay fp64): 1.3x faster, term error <= 2e-7 (measured
 *   2.4e-8 on the density of a 1e6-component mixture) -- used where parity with the reference is
 *   statistical anyway (throughput mode: device RNG), 50x inside the 1e-5 tolerance on SMC weights.
 *
 * elfi_b200_smc_weights_f64: w_i = exp(logprior_i - logq_i) (samplers.py:514).
 */
int elfi_b200_colmoments_f64(elfi_b200_ctx* ctx, const double* S, int64_t ldS, int64_t B, int64_t D,
                             double* out, void* stream);
int elfi_b200_weighted_stats_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, const double* w,
                                 int64_t N, int64_t p, double* stats, void* stream);
int elfi_b200_gm_logpdf_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t N,
                            const double* means, int64_t ldm, const double* w, int64_t M, int64_t p,
                            const double* Linv_host, double logdet, double* logq, void* stream);
int elfi_b200_gm_logpdf_mixed_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t N,
                                  const double* means, int64_t ldm, const double* w, int64_t M,
                                  int64_t p, const double* Linv_host, double logdet, double* logq,
                                  void* stream);
int elfi_b200_smc_weights_f64(elfi_b200_ctx* ctx, const double* logprior, const double* logq,
                              int64_t n, double* w, void* stream);

/* ---- BOLFI Gaussian-process surrogate (fp64) -------------------------------------------------
 * RBF + bias kernel k(a, b) = kernel_var * exp(-|a-b|^2 / (2 lengthscale^2)) + bias_var, Gaussian
 * noise.  These replace the GPy calls behind elfi/methods/bo/gpy_regression.py:
 *   update()/_init_gp() (242-315): Gram + Cholesky of Ky = K + noise_var I  -> elfi_b200_gp_fit_f64
 *   predict()/predict_mean() (98-163), incl. the cached-RBF restatement (127-140)
 *                                                                   -> elfi_b200_gp_predict_f64
 *   predictive_gradients() (186-223, restatement 206-218)           -> elfi_b200_gp_predict_grad_f64
 * and LCBSC.evaluate / evaluate_gradient (elfi/methods/bo/acquisition.py:262-301)
 *                                                                   -> `acq` outputs / elfi_b200_lcbsc_f64
 *
 * Factor storage (caller-allocated, n_pad x n_pad row-major, n_pad = elfi_b200_gp_padded_size(n)):
 *   L lower Cholesky factor (padded with the identity), W = L^-1, U = W^T;  alpha = Ky^-1 y (n).
 * noise_var must already include any jitter (GPy adds 1e-8).  info (device int32) is 0 on
 * success or 1 + the index of the first non-positive pivot.
 * gp_predict: mean/var/acq may each be NULL; var = k** - |W k|^2 + noise_add; acq = mean -
 * sqrt(beta * (noiseless var)).  Queries are processed in chunks through context scratch.
 */
int64_t elfi_b200_gp_padded_size(int64_t n);
int elfi_b200_gp_fit_f64(elfi_b200_ctx* ctx, const double* X, int64_t ldX, const double* y,
                         int64_t n, int64_t p, double kernel_var, double lengthscale,
                         double bias_var, double noise_var, double* L, double* W, double* U,
                         int64_t n_pad, double* alpha, int32_t* info, void* stream);
int elfi_b200_gp_predict_f64(elfi_b200_ctx* ctx, const double* Xq, int64_t ldq, int64_t m,
                             const double* X, int64_t ldX, int64_t n, int64_t p, const double* W,
                             int64_t n_pad, const double* alpha, double kernel_var,
                             double lengthscale, double bias_var, double noise_add, double beta,
                             double* mean, double* var, double* acq, void* stream);
int elfi_b200_gp_predict_grad_f64(elfi_b200_ctx* ctx, const double* Xq, int64_t ldq, int64_t m,
                                  const double* X, int64_t ldX, int64_t n, int64_t p,
                                  const double* W, const double* U, int64_t n_pad,
                                  const double* alpha, double kernel_var, double lengthscale,
                                  double bias_var, double* mean, double* var, double* grad_mean,
                                  double* grad_var, void* stream);
int elfi_b200_lcbsc_f64(elfi_b200_ctx* ctx, const double* mean, const double* var,
                        const double* grad_mean, const double* grad_var, int64_t m, int64_t p,
                        double beta, double* acq, double* grad_acq, void* stream);

/* Posterior cross-covariance of the GP between two sets of points, as ExpIntVar needs it
 * (elfi/methods/bo/acquisition.py:776-821; the reference re-factorises Ky on every evaluation,
 * :807).  With W from gp_fit, cov(x_a, x_b) = k(x_a, x_b) - (W k_a) . (W k_b):
 *   gp_whiten:    T[q, 0:n] = W k_q,  k_q[j] = k(Xq[q], X[j])  (RBF + bias);  T is (m, ldT), ldT >= n
 *   gp_cross_cov: cov[b * ma + a] = k(Xa[a], Xb[b]) - Ta[a, :] . Tb[b, :]     (mb x ma, row-major) */
int elfi_b200_gp_whiten_f64(elfi_b200_ctx* ctx, const double* Xq, int64_t ldq, int64_t m,
                            const double* X, int64_t ldX, int64_t n, int64_t p, const double* W,
                            int64_t n_pad, double kernel_var, double lengthscale, double bias_var,
                            double* T, int64_t ldT, void* stream);
/* out[q, 0:n] = W^T T[q, 0:n] (U = W^T from gp_fit): with T = gp_whiten(X_new) these are the rows
 * T W that a rank-b update of the factor (b new evidence points appended, no refit) needs. */
int elfi_b200_gp_apply_wt_f64(elfi_b200_ctx* ctx, const double* T, int64_t ldT, int64_t m,
                              const double* U, int64_t n_pad, int64_t n, double* out, int64_t ldo,
                              void* stream);
int elfi_b200_gp_cross_cov_f64(elfi_b200_ctx* ctx, const double* Xa, int64_t lda, int64_t ma,
                               const double* Ta, int64_t ldTa, const double* Xb, int64_t ldb,
                               int64_t mb, const double* Tb, int64_t ldTb, int64_t n, int64_t p,
                               double kernel_var, double lengthscale, double bias_var, double* cov,
                               void* stream);

/* Measures the sustained fp64 throughput of this device: tflops_host[0] = DFMA (vector pipe),
 * tflops_host[1] = DMMA (mma.sync m8n8k4.f64).  Roofline denominators for the compute-bound
 * kernels (mixture density, GP products); blocks the host for a few milliseconds. */
int elfi_b200_probe_fp64_f64(elfi_b200_ctx* ctx, double* tflops_host);

/* ---- throughput mode: device-side generation (SURVEY.md section 8f, N2) --------------------
 * Counter-based Philox4x32-10 streams keyed by (seed, offset + row): statistically equivalent to,
 * not bit-identical with, the reference's host RandomState.  `offset` = global index of the first
 * row of this call (e.g. batch_index * batch_size), so that any row sharding yields the same
 * particles.
 *   elfi_b200_prior_ma2_f64     CustomPrior1 / CustomPrior2 draws (elfi/examples/ma2.py:96-186);
 *                               mode 0 = (t1, t2) jointly, 1 = t1 only, 2 = t2 given the t1 passed in
 *   elfi_b200_logprior_ma2_f64  their joint log density (what ModelPrior.logpdf returns for MA2)
 *   elfi_b200_sim_ma2_f64       MA2 simulator (ma2.py:11-37); writes X (B, n_obs) and/or, fused,
 *                               the lag-1 / lag-2 autocovariances S (B, 2) (ma2.py:40-59, NumPy
 *                               pairwise order) so that X never has to touch HBM
 *   elfi_b200_gm_rvs_f64        GMDistribution.rvs (elfi/methods/utils.py:200-261): component by
 *                               weight, + MVN(0, Sigma) with Sigma = L L^T (Lchol_host, p <= 4),
 *                               redrawn until inside the support (0 = none, 1 = MA2 prior support,
 *                               2 = box: box_host = [lo_0..lo_{p-1}, hi_0..hi_{p-1}])
 *   elfi_b200_gm_cdf_f64        inclusive running sum of the (unnormalised) component weights, the
 *                               table np.random.choice(p=weights) builds on every call
 *                               (utils.py:239); one per population, reused by every batch of it
 *   elfi_b200_gm_rvs_cdf_f64    gm_rvs with that table (`cumw`, device, N) instead of the weights
 */
int elfi_b200_prior_ma2_f64(elfi_b200_ctx* ctx, int64_t B, uint64_t seed, uint64_t offset,
                            int32_t mode, double* t1, double* t2, void* stream);
int elfi_b200_logprior_ma2_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t B,
                               double* out, void* stream);
int elfi_b200_sim_ma2_f64(elfi_b200_ctx* ctx, const double* t1, const double* t2, int64_t B,
                          int64_t n_obs, uint64_t seed, uint64_t offset, double* X, int64_t ldX,
                          double* S, int64_t ldS, void* stream);
int elfi_b200_gm_rvs_f64(elfi_b200_ctx* ctx, const double* means, int64_t ldm, const double* weights,
                         int64_t N, int64_t p, const double* Lchol_host, int64_t B, uint64_t seed,
                         uint64_t offset, int32_t support, const double* box_host, double* out,
                         int64_t ldo, void* stream);
int elfi_b200_gm_cdf_f64(elfi_b200_ctx* ctx, const double* weights, int64_t N, double* cumw,
                         void* stream);
int elfi_b200_gm_rvs_cdf_f64(elfi_b200_ctx* ctx, const double* means, int64_t ldm, const double* cumw,
                             int64_t N, int64_t p, const double* Lchol_host, int64_t B, uint64_t seed,
                             uint64_t offset, int32_t support, const double* box_host, double* out,
                             int64_t ldo, void* stream);

/* Gaussian noise model of elfi/examples/gauss.py (1-d case): priors mu ~ U(prm[0], prm[0]+prm[1]),
 * sigma ~ truncnorm(prm[2], prm[3]) (gauss.py:118-126); simulator y = mu + sigma z (gauss.py:11-35)
 * with np.mean / np.var summaries (gauss.py:142-173, pairwise order) fused in the same kernel
 * (S (B, 2) = [mean, var]); Y (B, n_obs) is written only when requested. */
int elfi_b200_prior_gauss_f64(elfi_b200_ctx* ctx, int64_t B, uint64_t seed, uint64_t offset,
                              const double* prm_host, double* mu, double* sigma, void* stream);
int elfi_b200_logprior_gauss_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t B,
                                 const double* prm_host, double* out, void* stream);
int elfi_b200_sim_gauss_f64(elfi_b200_ctx* ctx, const double* mu, const double* sigma, int64_t B,
                            int64_t n_obs, uint64_t seed, uint64_t offset, double* Y, int64_t ldY,
                            double* S, int64_t ldS, void* stream);

/* g-and-k model of elfi/examples/gnk.py (throughput mode, statistical parity).
 * sim_gnk: Y[i, j] = A_i + B_i (1 + c (1 - exp(-g_i z)) / (1 + exp(-g_i z))) (1 + z^2)^k_i z with
 * z = z_ij ~ N(0, 1) from the Philox stream (seed, offset + i, j) (gnk.py:11-68); Y is (B, n_obs)
 * with leading dimension ldY.  The order-statistic summary is elfi_b200_rowsort_f64 on Y.
 * logprior_box: sum of independent uniform log densities, box_host = [lo (p), width (p)], p <= 8
 * (the priors A, B, g, k ~ uniform(0, 10) of gnk.py:99-103); -inf outside. */
int elfi_b200_sim_gnk_f64(elfi_b200_ctx* ctx, const double* A, const double* Bs, const double* g,
                          const double* k, double c, int64_t B, int64_t n_obs, uint64_t seed,
                          uint64_t offset, double* Y, int64_t ldY, void* stream);
int elfi_b200_logprior_box_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t B, int64_t p,
                               const double* box_host, double* out, void* stream);

/* ---- KLIEP density-ratio estimation (AdaptiveThresholdSMC) -------------------------------------
 * DensityRatioEstimation.fit + max_ratio (elfi/methods/density_ratio_estimation.py:71-207):
 * basis centres = first n_basis rows of x, A = RBF(x, centres), b = weighted RBF mean over y,
 * <= max_iter projected-gradient steps with a convergence check every conv_check_interval
 * steps.  wx (unnormalised, as the reference passes it) and wy may be NULL (ones).
 * alpha_out: device (n_basis);  result_host[0] = max_i r(x_i), result_host[1] = steps taken.
 * Blocks until done (the convergence test needs the host). */
int elfi_b200_kliep_fit_f64(elfi_b200_ctx* ctx, const double* x, int64_t ldx, int64_t Nx,
                            const double* y, int64_t ldy, int64_t Ny, int64_t p, const double* wx,
                            const double* wy, double sigma, int64_t n_basis, double epsilon,
                            int64_t max_iter, double abs_tol, int64_t conv_check_interval,
                            double* alpha_out, double* result_host);

/* elfi_b200_rowsort_f64: out[i, :] = np.sort(X[i, :]) (ascending, NaN last), 1 <= n <= 2048.
 * Order-statistic summaries such as the g-and-k model's (elfi/examples/gnk.py:145-161; the
 * 2-d form np.sort(y[:, :, 0], axis=1) that an (B, n_obs) summary matrix needs, SURVEY 8d #5). */
int elfi_b200_rowsort_f64(elfi_b200_ctx* ctx, const double* X, int64_t ldX, int64_t B, int64_t n,
                          double* out, int64_t ld_out, void* stream);

/* ---- BSL synthetic likelihood (fp64) ----------------------------------------------------------
 * elfi_b200_synlik_f64: the Gaussian synthetic log-likelihood of P groups of simulated summaries,
 *   GAUSSIAN      gaussian_syn_likelihood             (elfi/methods/bsl/pdf_methods.py:77-135)
 *   GHURYE_OLKIN  gaussian_syn_likelihood_ghurye_olkin (elfi/methods/bsl/pdf_methods.py:138-176)
 * Group g is rows g*group_stride .. g*group_stride + n - 1 of S ((rows, d) row-major, leading
 * dimension ldS); group_stride > n uses the first n rows of each block (array n_sim of
 * log_SL_stdev / select_penalty without copies).  Per group: column mean mu and the np.cov
 * covariance Sigma (ddof 1); with Wh (d x d device, row-major, or NULL) mu' = Wh mu,
 * Sigma' = Wh Sigma Wh^T, obs' = Wh obs; for each of the L Warton parameters gamma_host[l] (HOST,
 * in [0, 1]; the reference's cov_warton(Sigma, gamma) = gamma Sigma + (1 - gamma) diag(Sigma_ii +
 * 1e-5)), a Cholesky factor and
 *   loglik[g*L + l] = -(|L^-1 (obs - mu)|^2 + log det Sigma + d log 2 pi) / 2.
 * gamma_host == NULL means no shrinkage (L must be 1).  GHURYE_OLKIN takes neither Wh nor gammas;
 * its log|det psi| = d log(n-1) + log det Sigma + log|1 - q n / (n-1)^2| with
 * q = (obs-mu)^T Sigma^-1 (obs-mu) comes from the same factor (sign-blind like the reference's
 * slogdet).  -inf: a non-finite value in the group, or a pivot <= 1e6 eps max_j A_jj of the
 * factored matrix A (SciPy's _PSD cutoff constant applied to pivots; this covers n <= d).  A nearly
 * singular Sigma between that criterion and SciPy's eigenvalue test may be -inf in one
 * implementation and finite in the other.
 * Limits: 1 <= d <= ELFI_B200_SYNLIK_MAX_D, n >= 2, group_stride >= n, L >= 1, else ERR_ARG. */
#define ELFI_B200_SYNLIK_MAX_D 128
#define ELFI_B200_SYNLIK_GAUSSIAN 0
#define ELFI_B200_SYNLIK_GHURYE_OLKIN 1
int elfi_b200_synlik_f64(elfi_b200_ctx* ctx, int32_t estimator, const double* S, int64_t ldS,
                         int64_t P, int64_t n, int64_t group_stride, int64_t d, const double* obs,
                         const double* Wh, const double* gamma_host, int64_t L, double* loglik,
                         void* stream);

#ifdef __cplusplus
}
#endif

#endif /* ELFI_B200_H */
