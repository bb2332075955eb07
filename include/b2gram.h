/*
 * b2gram.h -- C-ABI of libb2gram.so: the B200 (sm_100a) retrain hot path of
 * AlexIoannides/bodywork-mlops-demo, i.e. the least-squares / ridge fit that
 * mlops_simulation/stage_1_train_model.py performs through scikit-learn.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.
 * The reference is pure Python, so the binding a maintainer adds is a ctypes stub
 * (see INTEGRATION.md); every entry point cites the reference call it replaces.
 *
 * Conventions
 *   - every function returns int: 0 = ok, <0 = error (B2_E_*); text via b2_last_error()
 *     (thread-local).  No exceptions cross the boundary.
 *   - the caller owns every buffer it passes; b2_ctx owns device scratch, streams, the
 *     fp64 sufficient statistic S and (optionally) one NCCL communicator.
 *   - one b2_ctx == one GPU; one process per GPU for multi-GPU (rows shard by rank, the
 *     only exchange is b2_gram_allreduce).  A ctx is not re-entrant.
 *   - there is NO CPU fallback: without a usable CUDA device every compute entry point
 *     fails with B2_E_CUDA.
 *
 * Sufficient statistic.  S = [X 1 y]^T [X 1 y], (D+2) x (D+2), row-major fp64, index
 * order: features 0..D-1, the ones column (D), y (D+1).  S[D][D] is the row count.
 */
#ifndef B2GRAM_H_
#define B2GRAM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_ABI_VERSION 2
#define B2_MAX_D 128

/* element type of X */
#define B2_F32 0
#define B2_BF16 1
#define B2_F64 2 /* b2_metrics, b2_upload_columns */

/* where a caller buffer lives */
#define B2_MEM_DEVICE 0 /* device pointer (HBM)                                   */
#define B2_MEM_HOST 1   /* host pointer (pinned preferred); streamed in row blocks */

/* kernel selection for b2_gram_accumulate */
#define B2_KERNEL_AUTO 0   /* d <= 16: NARROW; wider: TCGEN05; odd layouts / tiny blocks: SIMT */
#define B2_KERNEL_SIMT 1   /* fp64-accumulating CUDA-core kernel (any D <= 128)       */
#define B2_KERNEL_TCGEN05 2 /* TMA -> smem -> bf16 hi/lo split -> tcgen05.mma -> TMEM   */
#define B2_KERNEL_NARROW 3  /* D <= 16: TMA bulk-copy pipeline -> fp32 FMA on CUDA cores */
/* tcgen05 path requirements: 4 <= d <= 128, row bytes and row pitch multiples of 16, X / y / row_mask 16-byte
 * aligned, n_rows >= 64.  Contiguous rows with 17 <= d <= 64 are packed min(5, 128 / d) per 128-wide super-row.
 * narrow path requirements: d <= 16, contiguous rows (ldx == d), X / y / row_mask 16-byte aligned.
 * AUTO uses NARROW from 4096 rows and TCGEN05 from 2048 rows per call; smaller blocks (the reference's 1 440-row
 * daily tranche, stage_3_synthetic_data_generation.py:19) and every other layout take the exact fp64 SIMT kernel. */

/* operand precision of the tcgen05 Gram kernel (b2_ctx_set_precision) */
#define B2_PRECISION_SPLIT 0 /* bf16 hi + lo operands (16 mantissa bits), default: coef error ~2e-6 at any n */
#define B2_PRECISION_BF16 1  /* single bf16 operand ("bf16-accum", BASELINE.json configs[1]): error ~2.4e-2/sqrt(n) */

/* error codes */
#define B2_OK 0
#define B2_E_ARG (-1)
#define B2_E_CUDA (-2)
#define B2_E_STATE (-3)
#define B2_E_SINGULAR (-4) /* Cholesky met a non-positive pivot (rank-deficient, alpha == 0) */
#define B2_E_COMM (-5) /* NCCL failure, or a peer did not deliver its partial statistic within the timeout */
#define B2_E_NCCL B2_E_COMM
#define B2_E_UNSUPPORTED (-6)

typedef struct b2_ctx b2_ctx;

/* ---- library / context ------------------------------------------------------------ */
int b2_abi_version(void);
const char* b2_last_error(void);
int b2_device_count(int* n_out);
int b2_ctx_create(int device, b2_ctx** out);
int b2_ctx_destroy(b2_ctx* ctx);
int b2_ctx_sync(b2_ctx* ctx);
/* name, SM count, HBM bytes of the ctx's device (name_cap bytes incl. NUL) */
int b2_ctx_info(b2_ctx* ctx, char* name, int name_cap, int* sm_count, size_t* hbm_bytes);
/* force a kernel family (B2_KERNEL_*); default AUTO */
int b2_ctx_set_kernel(b2_ctx* ctx, int kernel);
/* rows of fp32 tensor-core accumulation before a TMEM drain into fp64 (default 8192) */
int b2_ctx_set_drain_rows(b2_ctx* ctx, int rows);
/* the persistent Gram kernel uses at most n_sms SMs (0 = all): leaves room for other work on the device */
int b2_ctx_set_sm_limit(b2_ctx* ctx, int n_sms);
/* B2_PRECISION_*: operand precision of the tensor-core path (the CUDA-core kernel is always exact) */
int b2_ctx_set_precision(b2_ctx* ctx, int precision);

/* ---- caller-owned buffers (helpers; the Python shim has no other CUDA binding) ------------ */
int b2_dev_alloc(b2_ctx* ctx, size_t bytes, void** out);
int b2_dev_free(b2_ctx* ctx, void* p);
int b2_host_alloc(b2_ctx* ctx, size_t bytes, void** out); /* pinned */
int b2_host_free(b2_ctx* ctx, void* p);
int b2_copy_h2d(b2_ctx* ctx, void* dst, const void* src, size_t bytes); /* sync on return */
int b2_copy_d2h(b2_ctx* ctx, void* dst, const void* src, size_t bytes); /* sync on return */
int b2_copy_d2d(b2_ctx* ctx, void* dst, const void* src, size_t bytes); /* on the context's stream, asynchronous: bench.py
                                                                         times it as this box's own copy bandwidth */
int b2_dev_memset(b2_ctx* ctx, void* dst, int value, size_t bytes);
/* DataFrame columns -> row-major float32 rows in HBM.  reference: stage_1_train_model.py:95-96
 * (`X = data['X'].values.reshape(-1, 1)`): pandas hands every column over as its own strided array.  cols[j] = address of
 * row 0 of feature column j, strides[j] = bytes between consecutive rows of it, dtype = B2_F64 (pandas' default) or B2_F32;
 * X_dev: caller-owned device buffer of n_rows x d floats, row-major.  Host threads gather and convert into a pinned ring
 * while the previous block is on the wire; sync on return. */
int b2_upload_columns(b2_ctx* ctx, const void* const* cols, const int64_t* strides, int dtype, int64_t n_rows, int d,
                      float* X_dev);
/* The gather + conversion of b2_upload_columns alone, host to host (no device, no context): out[n_rows][d] float32, e.g. a
 * caller's own pinned block.  Multi-threaded like the upload. */
int b2_pack_columns(const void* const* cols, const int64_t* strides, int dtype, int64_t n_rows, int d, float* out);

/* ---- Gram accumulation: replaces LinearRegression.fit's pass over the rows -----------------
 * reference: stage_1_train_model.py:105-106 -> sklearn/linear_model/_base.py (centre + gelsd). */
int b2_gram_reset(b2_ctx* ctx, int d);
/* S += [X 1 y]^T [X 1 y] over the rows of this block (this rank's shard).
 *   X        n_rows x d, row-major, leading dimension ldx (elements), dtype x_dtype
 *   y        n_rows fp32
 *   row_mask NULL, or one byte per row: a row is used iff row_mask[r] == mask_keep.
 *            (lets train_test_split's shuffled 80/20 membership -- stage_1_train_model.py:98-103 --
 *            be applied without gathering rows)
 *   mem_kind where X / y / row_mask live (all three the same)                                */
int b2_gram_accumulate(b2_ctx* ctx, const void* X, int x_dtype, const float* y, int64_t n_rows,
                       int d, int64_t ldx, int mem_kind, const uint8_t* row_mask, int mask_keep);
/* sum S over the ranks of the communicator (one ncclAllReduce of (d+2)^2 doubles) */
int b2_gram_allreduce(b2_ctx* ctx);
/* copy S out / in (incremental-refit state).  S_out/S_in: (d+2)^2 doubles on the host */
int b2_gram_export(b2_ctx* ctx, double* S_out, int64_t* n_rows_out);
int b2_gram_import(b2_ctx* ctx, const double* S_in, int d);
/* which kernel families added to the resident S since the last b2_gram_reset / b2_gram_import / b2_fit:
 * *kernels_out = OR of (1 << B2_KERNEL_SIMT / _TCGEN05 / _NARROW) (0 after an import: the source is the caller's).
 * A statistic from the tensor-core or narrow kernel resolves eigenvalues only down to ~eps_kernel of the largest, so a
 * caller that finds the centred Gram near singular can rebuild S on the exact kernel (B200LinearRegression.fit does). */
int b2_gram_kernels(b2_ctx* ctx, int* kernels_out);

/* ---- split: the row membership of train_test_split(X, y, test_size, random_state=seed) ---------------------------
 * reference: stage_1_train_model.py:98-103 -> sklearn ShuffleSplit: perm = RandomState(seed).permutation(n_rows);
 * test = perm[:n_test], train = the rest.  mask_out[r] = 0 for test rows, 1 for train rows (n_rows bytes, host) --
 * the row_mask b2_gram_accumulate / b2_fit (keep 1) and b2_score (keep 0) consume.  Host-side by nature (MT19937 +
 * Fisher-Yates are sequential); bit-exact with numpy's legacy generator, ~10x its speed at 10^8 rows. */
int b2_split_mask(int64_t n_rows, int64_t n_test, uint32_t seed, uint8_t* mask_out);

/* ---- the whole fit in one call: LinearRegression(fit_intercept).fit(X, y) / Ridge(alpha) ----------------------
 * reference: stage_1_train_model.py:105-106.  Equivalent to b2_gram_reset + b2_gram_accumulate + b2_gram_allreduce +
 * b2_solve with the same arguments.  Device-resident rows that take the tensor-core kernel skip the memset, the separate
 * scatter / gather launches and the D2H copy: the finalize kernel behind the Gram kernel folds the partials and stores
 * S into the peers' exchange slots (when a peer exchange is attached), the solve kernel sums the peers' slots, factors
 * and writes coef / intercept to the host. */
int b2_fit(b2_ctx* ctx, const void* X, int x_dtype, const float* y, int64_t n_rows, int d, int64_t ldx,
           int mem_kind, const uint8_t* row_mask, int mask_keep, double alpha, int fit_intercept,
           double* coef, double* intercept);

/* ---- solve: replaces scipy.linalg.lstsq + _set_intercept ----------------------------------------
 * reference: sklearn/linear_model/_base.py (lstsq on centred data; intercept_ = y_mean - x_mean.coef_)
 * Single-SM fp64 LDL^T (square-root-free Cholesky) of (Xc^T Xc + alpha I).  coef: d doubles, intercept: 1 double
 * (host).  fit_intercept = 0 solves the uncentred problem.  Returns B2_E_SINGULAR on a non-positive pivot and
 * B2_E_COMM when the preceding peer-memory exchange timed out (S incomplete). */
int b2_solve(b2_ctx* ctx, double alpha, int fit_intercept, double* coef, double* intercept);
/* eigenvalues of the centred Gram (device Jacobi) -> singular_ (descending, d doubles) and rank_
 * (count of singular values > cond * max), plus the minimum-norm coefficients gelsd would return.
 * Any output pointer may be NULL. */
int b2_solve_spectral(b2_ctx* ctx, double cond, int fit_intercept, double* coef, double* intercept,
                      double* singular, int* rank);

/* singular_ (descending, d doubles) and rank_ only -- the attributes LinearRegression.fit stores beside coef_
 * (sklearn/linear_model/_base.py) -- as sqrt of the eigenvalues of the centred Gram: Householder tridiagonalisation +
 * Sturm multisection on one SM, no eigenvectors (b2_solve_spectral is only needed when rank < d). */
int b2_solve_eigvals(b2_ctx* ctx, double cond, int fit_intercept, double* singular, int* rank,
                     int64_t* n_rows_out /* rows in S; may be NULL */);

/* ---- scoring: replaces model.predict and model_metrics ------------------------------------------
 * reference: stage_1_train_model.py:107 / stage_2_serve_model.py:78 (X @ coef_ + intercept_)
 *            stage_1_train_model.py:79-90 (MAPE, r2_score, max_error)
 * yhat may be NULL (metrics only); y may be NULL (predict only; stats_out untouched).
 * stats_out (host, 10 doubles):
 *   [0] sum |yhat-y|/max(|y|,eps_f64)  [1] sum (y-yhat)^2  [2] sum y  [3] sum y^2  [4] max |y-yhat|  [5] rows used
 *   [6] sum yhat  [7] sum yhat^2  [8] sum y*yhat  [9] max |yhat/y - 1|
 *   ([0]-[5]: stage_1's model_metrics; [6]-[9]: stage_4_test_model_scoring_service.py:89,101-105 -- APE,
 *    Pearson "r_squared", max APE.)
 * With a communicator, b2_score_allreduce combines the ten across ranks (sums; [4] and [9] by max). */
int b2_score(b2_ctx* ctx, const void* X, int x_dtype, int64_t n_rows, int d, int64_t ldx,
             int mem_kind, const double* coef, double intercept, const float* y,
             const uint8_t* row_mask, int mask_keep, float* yhat, double* stats_out);
int b2_score_allreduce(b2_ctx* ctx, double* stats_inout);
/* model_metrics(y_actual, y_predicted) (stage_1_train_model.py:79-90) on two vectors of dtype B2_F32 or B2_F64
 * (the reference works on float64 arrays): the same ten reductions as b2_score, divisions correctly rounded. */
int b2_metrics(b2_ctx* ctx, const void* y_actual, const void* y_predicted, int dtype, int64_t n_rows,
               int mem_kind, double* stats_out);

/* ---- synthetic rows on the device (benchmarks): stage_3_synthetic_data_generation.py:36-43 --------
 * X_ij ~ U(0,100), eps ~ N(0,1), y = alpha + beta * sum_j X_ij + sigma * eps   (Philox4x32-10,
 * counter = global row index + row_offset, so shards of one dataset can be drawn independently). */
int b2_synth(b2_ctx* ctx, uint64_t seed, int64_t row_offset, int64_t n_rows, int d, int64_t ldx,
             int x_dtype, double alpha, double beta, double sigma, void* X_dev, float* y_dev);

/* One reference tranche (D = 1) of day `day` >= 1, exactly as generate_dataset draws it
 * (stage_3_synthetic_data_generation.py:28-43): alpha(day) = 1 + 0.5 sin(2 pi 6 (day - 1) / 364), X ~ U(0,100),
 * y = alpha + beta X + sigma eps, rows with y < 0 dropped, order kept.  X_dev / y_dev hold n_rows floats; the
 * number of rows written comes back in *n_kept_out. */
int b2_synth_tranche(b2_ctx* ctx, uint64_t seed, int64_t n_rows, int day, double beta, double sigma,
                     float* X_dev, float* y_dev, int64_t* n_kept_out);

/* ---- multi-GPU (one process per GPU; NCCL is dlopen'ed on first use) ------------------------------ */
int b2_comm_unique_id(char* id_out /* 128 bytes */);
int b2_comm_init(b2_ctx* ctx, int n_ranks, int rank, const char* id /* 128 bytes */);
int b2_comm_destroy(b2_ctx* ctx);
int b2_comm_barrier(b2_ctx* ctx);
/* Optional one-shot peer-memory exchange for b2_gram_allreduce (2..8 ranks of one NVLink box): every rank exports
 * the CUDA-IPC handle of its exchange buffer (64 bytes), the caller gathers the handles of all ranks in rank
 * order and attaches them.  Once attached, b2_gram_allreduce stores S into every peer's buffer over NVLink and
 * sums the n slots in rank order (no NCCL launch; bit-identical S on every rank); NCCL stays the fallback. */
int b2_comm_p2p_export(b2_ctx* ctx, char* handle_out /* 64 bytes */);
int b2_comm_p2p_attach(b2_ctx* ctx, int n_ranks, int rank, const char* handles /* n_ranks x 64 bytes */);
int b2_comm_p2p_detach(b2_ctx* ctx); /* back to the NCCL all-reduce (all ranks must detach together) */
/* the same exchange between contexts of ONE process (several GPUs driven by one C client, or two contexts on one
 * GPU): peers[r] is rank r's context, peers[rank] == ctx.  Every context of the group calls it once. */
int b2_comm_p2p_attach_local(b2_ctx* ctx, int n_ranks, int rank, b2_ctx* const* peers);
/* how long a rank waits for a peer's partial statistic before the exchange fails with B2_E_COMM (default 10 000 ms) */
int b2_comm_set_timeout_ms(b2_ctx* ctx, int64_t ms);
/* ranks, this rank, and which exchange b2_gram_allreduce / b2_fit use (B2_EXCHANGE_*) */
#define B2_EXCHANGE_NONE 0
#define B2_EXCHANGE_NCCL 1
#define B2_EXCHANGE_PEER 2
int b2_comm_info(b2_ctx* ctx, int* n_ranks_out, int* rank_out, int* exchange_out);

/* ---- timing (CUDA events on the ctx stream) ---------------------------------------------------------
 * b2_timer_start/stop bracket any sequence of calls; *_ms is device time between the two events.
 * b2_last_kernel_ms: summed device time of the tcgen05 Gram kernel launches (one CUDA-event pair each, at most
 * the 64 most recent) since the previous call to this function, and how many launches that sum covers. */
int b2_timer_start(b2_ctx* ctx);
int b2_timer_stop(b2_ctx* ctx, double* ms_out);
int b2_last_kernel_ms(b2_ctx* ctx, double* gram_ms_out, int* launches_out);
/* total number of kernels this ctx has launched since creation (bench.py's gpu_launches) */
int b2_launch_count(b2_ctx* ctx, int64_t* n_out);
/* out3[0] fits that took the fused path of b2_fit, [1] peer exchanges started, [2] kernels launched */
int b2_ctx_stats(b2_ctx* ctx, int64_t* out3);

#ifdef __cplusplus
}
#endif
#endif /* B2GRAM_H_ */
