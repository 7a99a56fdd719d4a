/*
 * cvmx.h - C ABI of the B200-native fold-wise training-matrix engine (libcvmx.so).
 *
 * This is the drop-in boundary for the hot path of sm00thix/cvmatrix (reference v3.2.1):
 *     CVMatrix.fit -> Partitioner index sets -> CVMatrix.training_XTX / training_XTY /
 *     training_XTX_XTY / training_statistics.
 * The reference has no FFI of its own (pure Python over numpy); the entry points below are
 * what a binding for this path would call - INTEGRATION.md shows the ctypes stub.  Each
 * declaration cites the reference code it replaces (file:line under the reference root).
 *
 * Conventions
 *   - every function returns a cvmx_status (0 = CVMX_OK); no exception crosses the boundary;
 *     cvmx_last_error() gives the message of the last failure on a handle (or on the calling
 *     thread when no handle exists yet).
 *   - plain pointers and sizes only.  `mem` says whether the pointers of that call are HOST
 *     or DEVICE addresses (on the handle's device).  Host pointers are only read/written
 *     during the call; the library owns its device copies; callers own every output buffer.
 *   - matrices are row-major.  dtype: 0 = float32, 1 = float64 (all floating-point buffers of
 *     a handle have the handle's dtype); indices and counts are int64.
 *   - flags  = center_X | center_Y << 1 | scale_X << 2 | scale_Y << 3
 *     want   = CVMX_WANT_XTX | CVMX_WANT_XTY | CVMX_WANT_STATS
 *   - one host thread drives a handle at a time.  All device work of a handle is issued on
 *     the handle's stream (cvmx_set_stream; default: a private non-blocking stream).
 *   - there is NO CPU fallback: without a CUDA device cvmx_create fails with CVMX_ERR_CUDA.
 */
#ifndef CVMX_H_
#define CVMX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CVMX_VERSION 100 /* 0.1.0 */

typedef struct cvmx_handle cvmx_t;

typedef enum {
  CVMX_OK = 0,
  CVMX_ERR_INVALID = 1,    /* bad argument / call order                                   */
  CVMX_ERR_CUDA = 2,       /* CUDA runtime failure (message in cvmx_last_error)            */
  CVMX_ERR_NEG_WEIGHT = 3, /* -> ValueError("Weights must be non-negative.")  cvmatrix/cvmatrix.py:1186-1189 */
  CVMX_ERR_INDEX = 4,      /* validation index outside [-N, N)  -> IndexError (numpy fancy indexing) */
  CVMX_ERR_NO_Y = 5,       /* XTY wanted but fit() had no Y     cvmatrix/cvmatrix.py:810-811 */
  CVMX_ERR_NOMEM = 6
} cvmx_status;

enum { CVMX_F32 = 0, CVMX_F64 = 1 };
enum { CVMX_HOST = 0, CVMX_DEVICE = 1 };
enum { CVMX_CENTER_X = 1, CVMX_CENTER_Y = 2, CVMX_SCALE_X = 4, CVMX_SCALE_Y = 8 };
enum { CVMX_WANT_XTX = 1, CVMX_WANT_XTY = 2, CVMX_WANT_STATS = 4 };

/* per-fold status bits written by the training calls (0 = fine):
 *   bit 0: weighted and no non-zero weight is left in the training set  (cvmatrix/cvmatrix.py:625-629)
 *   bit 1: number of non-zero training weights <= ddof                   (cvmatrix/cvmatrix.py:1074-1078)
 * Whether a bit is an error depends on which statistics the caller's method computes
 * (cvmatrix/cvmatrix.py:693-699, 722-725); that decision stays with the host wrapper. */
enum { CVMX_FOLD_NO_NONZERO_W = 1, CVMX_FOLD_NNZ_LE_DDOF = 2 };

int32_t cvmx_version(void);
const char* cvmx_last_error(const cvmx_t* h); /* h may be NULL */

/* Replaces CVMatrix.__init__ (cvmatrix/cvmatrix.py:157-205).  `resolution` is
 * np.finfo(dtype).resolution * 10 evaluated by the caller in the model dtype (cvmatrix.py:187). */
int32_t cvmx_create(int32_t device, int32_t dtype, uint32_t flags, int64_t ddof, double resolution,
                    cvmx_t** out);
int32_t cvmx_destroy(cvmx_t* h);

/* Use the caller's CUDA stream (a cudaStream_t passed as void*) for all later work. NULL restores
 * the private stream. */
int32_t cvmx_set_stream(cvmx_t* h, void* cuda_stream);
int32_t cvmx_sync(cvmx_t* h);

/*
 * Replaces CVMatrix.fit (cvmatrix/cvmatrix.py:207-328 -> _init_mats :1153-1191,
 * _init_weighted_mats :1193-1207, _init_matrix_products :1209-1217, _init_stats :1219-1243).
 * X is N x K with row pitch ldx (elements), Y is N x M (NULL/M = 0: no responses), w has N
 * entries (NULL: unweighted).  The library keeps a device copy Z = [X | Y | 0-pad] and w.
 * It computes   XtWX, XtWY (one weighted Gram pass on FP64 tensor cores),
 *               sum w (numpy pairwise order), count_nonzero(w),
 *               column sums of WX, WY, WX.X, WY.Y (numpy order: sequential per column).
 * [gram_row_begin, gram_row_end) restricts the Gram pass to a row slab (multi-GPU row sharding:
 * the caller all-reduces cvmx_totals_ptr() across ranks and then calls cvmx_commit_totals);
 * pass 0, N for the whole matrix.  Moment sums always cover all N rows (their order cannot be
 * sharded).  Returns CVMX_ERR_NEG_WEIGHT if any weight is negative.
 */
int32_t cvmx_fit(cvmx_t* h, const void* X, int64_t N, int64_t K, int64_t ldx, const void* Y, int64_t M,
                 int64_t ldy, const void* w, int32_t mem, int64_t gram_row_begin, int64_t gram_row_end);

/*
 * The same fit fed in row blocks (streaming / sharded upload), replacing the same reference code as cvmx_fit
 * (cvmatrix/cvmatrix.py:207-328, 1131-1243).  Use it when the matrix does not exist in one piece on the host (it is
 * produced on the device, or it is larger than host memory: 180 GB of HBM hold N = 2M x K = 5000 float64), or when
 * several GPUs share the upload: every rank copies only its own row slab over PCIe and the slabs are exchanged over
 * NVLink straight into cvmx_data_ptr() (cvmatrix_b200/distributed.py: fit_sharded_upload).
 *   cvmx_fit_begin : allocates Z = [X | Y | 0-pad] (N x ld), w and the totals; max_block_rows bounds the blocks.
 *   cvmx_fit_rows  : rows [row0, row0 + nrows) from X (pitch ldx), Y (pitch ldy; ignored when M = 0), w (ignored when
 *                    unweighted); `mem` = CVMX_HOST or CVMX_DEVICE.  With gram != 0 the block's weighted Gram
 *                    X^T diag(w) [X | Y] is added to a float64 accumulator; blocks may come in any order, every row
 *                    must be contracted by exactly one rank.  Returns after the block buffers may be reused.
 *   cvmx_fit_end   : accumulator -> cvmx_totals_ptr(); sum w / count_nonzero(w) over all N rows (they must all be
 *                    present by now); numpy-order column sums for column groups col_shard, col_shard + n, ...
 *                    (others zero).  One GPU: cvmx_fit_end(h, 0, 1) completes the fit.  Several: all-reduce(sum)
 *                    cvmx_totals_ptr() and cvmx_moments_ptr() across ranks, then cvmx_commit_totals.
 */
int32_t cvmx_fit_begin(cvmx_t* h, int64_t N, int64_t K, int64_t M, int32_t weighted, int64_t max_block_rows);
int32_t cvmx_fit_rows(cvmx_t* h, int64_t row0, int64_t nrows, const void* X, int64_t ldx, const void* Y, int64_t ldy,
                      const void* w, int32_t mem, int32_t gram);
int32_t cvmx_fit_end(cvmx_t* h, int32_t col_shard, int32_t n_col_shards);
/* Device addresses of Z (N x ld, handle dtype), w (N) and of the two moment rows (ld elements each). */
int32_t cvmx_data_ptr(cvmx_t* h, void** Z, void** w, int64_t* ld);
int32_t cvmx_moments_ptr(cvmx_t* h, void** sum_z, void** sumsq_z, int64_t* count);

/* Device address and element count of the K x ld [XtWX | XtWY] totals (handle dtype), for an
 * external all-reduce (NCCL) between cvmx_fit on a row slab and cvmx_commit_totals. */
int32_t cvmx_totals_ptr(cvmx_t* h, void** dev_ptr, int64_t* count, int64_t* ld);
int32_t cvmx_commit_totals(cvmx_t* h);

/* Host copies of the public fit attributes XTX, XTY, sum_X, sum_Y, sum_sq_X, sum_sq_Y, sum_w,
 * num_nonzero_w (cvmatrix/cvmatrix.py:233-314).  Any pointer may be NULL.  Dense outputs:
 * XTX K*K, XTY K*M, sums K / M.  sum_w is returned as double (exact for float32 too). */
int32_t cvmx_get_totals(cvmx_t* h, void* XTX, void* XTY, void* sum_X, void* sum_Y, void* sum_sq_X,
                        void* sum_sq_Y, double* sum_w, int64_t* nnz_w);

/*
 * Device-resident CSR of validation index sets: replaces the per-fold index arrays of
 * Partitioner.folds_dict (cvmatrix/partitioner.py:89-107) as consumed by
 * _get_val_matrices (cvmatrix/cvmatrix.py:924-937).  offsets has P + 1 entries, indices
 * offsets[P].  Indices may be unsorted / repeated / negative (numpy wrap-around); anything
 * outside [-N, N) gives CVMX_ERR_INDEX.  Needs a prior cvmx_fit.
 */
int32_t cvmx_set_folds(cvmx_t* h, const int64_t* offsets, const int64_t* indices, int64_t P, int32_t mem);

/*
 * cvmx_fit + cvmx_set_folds in one call (host pointers).  When the folds are a TRUE partition of the rows (every row in
 * exactly one fold, indices ascending inside a fold - what Partitioner produces, cvmatrix/partitioner.py:89-107) and
 * the matrix takes the chunk-pipelined upload, XtWX = sum over folds of the fold Grams: every row is contracted ONCE,
 * per fold, behind the host->device copy, the raw fold Grams are kept, and a later cvmx_training_batch(XTX|XTY) only
 * runs the statistics and the centering / scaling epilogue (the reference evaluates 2 N K (K+M) flops in fit and the
 * same again over the folds, cvmatrix/cvmatrix.py:1215-1217 and :1001).  Otherwise it behaves exactly like the two
 * separate calls.  is_partition != 0 skips the O(N) verification (the caller vouches for it).
 * cvmx_folds_are_cached: 1 while the kept fold Grams match the current CSR.
 */
int32_t cvmx_fit_folds(cvmx_t* h, const void* X, int64_t N, int64_t K, int64_t ldx, const void* Y, int64_t M, int64_t ldy,
                       const void* w, int32_t mem, const int64_t* offsets, const int64_t* indices, int64_t P,
                       int32_t is_partition);
int32_t cvmx_folds_are_cached(const cvmx_t* h);

/*
 * Batched replacement of _training_matrices / training_statistics for folds
 * [fold_begin, fold_end) of the CSR (cvmatrix/cvmatrix.py:754-896, 519-574; per fold:
 * _get_sum_w_train_and_num_nonzero_w_train :589-630, _compute_training_stats :632-752,
 * _compute_std_divisor :1045-1079, _compute_training_mat_std :1081-1129,
 * _training_kernel_matrix :943-1010).  With P' = fold_end - fold_begin:
 *   out_XTX   [P', K, K]   if want & CVMX_WANT_XTX   (else may be NULL)
 *   out_XTY   [P', K, M]   if want & CVMX_WANT_XTY
 *   out_stats [P', 2, K+M] rows: weighted mean, weighted std of the training set over the columns of
 *                          [X | Y]; entries the flags do not define are 0
 *   out_scal  [P', 2]      sum of training weights, number of non-zero training weights
 *   out_status[P']         int32 bits CVMX_FOLD_*
 * out_stats / out_scal / out_status may be NULL.  `mem` applies to all five output pointers.
 * Centering / scaling of each matrix follows the handle flags exactly as the reference does
 * (XTX centred iff center_X, XTY centred iff center_X|center_Y, ... :843-864, 1001-1009).
 */
int32_t cvmx_training_batch(cvmx_t* h, int64_t fold_begin, int64_t fold_end, uint32_t want, void* out_XTX,
                            void* out_XTY, void* out_stats, void* out_scal, int32_t* out_status, int32_t mem);

/* Same for ONE ad-hoc validation index set (the reference's per-call signature
 * training_XTX_XTY(validation_indices), cvmatrix/cvmatrix.py:330-517).  Does not disturb the CSR. */
int32_t cvmx_training_indices(cvmx_t* h, const int64_t* val_idx, int64_t n_val, int32_t idx_mem, uint32_t want,
                              void* out_XTX, void* out_XTY, void* out_stats, void* out_scal,
                              int32_t* out_status, int32_t out_mem);

/*
 * Sharded evaluation of a fold batch across several handles (one per GPU / rank).  The path shards two ways
 * (SURVEY.md 8e): many folds -> give each rank its own fold range with cvmx_training_batch (no collective);
 * few large folds -> split every fold's ROWS across ranks with the three phases below, the caller all-reducing
 * (NCCL) the two buffers in between - one fused all-reduce in cvmatrix_b200/distributed.py.  All pointers are DEVICE pointers; every rank holds the full data and the CSR.
 *   1. cvmx_sharded_stats : statistics of folds [f0, f1) for column groups col_shard, col_shard + n_col_shards, ...
 *        (the sequential per-column chains cannot be split by rows, so they are split by columns).  Returns the
 *        device address / element count (handle dtype) of the [P'][2][ld] buffer: entries of other shards are zero,
 *        so all-reduce(sum) in place assembles it.  The per-fold scalars are computed redundantly on every rank.
 *   2. cvmx_sharded_gram  : raw weighted Gram of row shard `row_shard` of every fold -> gram_dev, float64,
 *        cvmx_sharded_gram_count() elements (internal tile/fragment order); all-reduce(sum) across ranks.
 *   3. cvmx_sharded_finish: downdate + centering + scaling epilogue for folds [f0, f1) (a sub-range of the batch
 *        that started at batch_f0 - typically the folds this rank owns) from the reduced Gram; outputs as in
 *        cvmx_training_batch, indexed from f0.
 * Replaces, together, the same reference code as cvmx_training_batch.
 */
int32_t cvmx_sharded_stats(cvmx_t* h, int64_t f0, int64_t f1, int32_t col_shard, int32_t n_col_shards, void** stats_dev,
                           int64_t* stats_count);
int32_t cvmx_sharded_stats_wait(cvmx_t* h); /* phase 1 runs on a side stream beside phase 2: call this before touching its result */
int64_t cvmx_sharded_gram_count(cvmx_t* h, int64_t f0, int64_t f1, uint32_t want);
int32_t cvmx_sharded_gram(cvmx_t* h, int64_t f0, int64_t f1, uint32_t want, int32_t row_shard, int32_t n_row_shards,
                          double* gram_dev);
int32_t cvmx_sharded_finish(cvmx_t* h, int64_t batch_f0, int64_t f0, int64_t f1, uint32_t want, const double* gram_dev,
                            void* out_XTX, void* out_XTY, void* out_stats, void* out_scal, int32_t* out_status);

/* Phase 3 without the all-reduce: the raw Grams (and, behind them at element gram_count, the statistics rows widened to
 * float64) of ALL ranks live in buffers of the same layout that are mapped into this process over NVLink (symmetric
 * memory; peer_bufs[q] = rank q's buffer, this rank's own included, at most 8).  The owner of folds [f0, f1) sums the
 * peers' fragments on the fly inside the epilogue kernel (P2P loads) and the peers' statistics rows for the batch
 * [batch_f0, batch_f1) with a small kernel.  The caller provides the cross-GPU barrier between phase 2 and this call
 * (cvmatrix_b200/distributed.py: symmetric-memory barrier).  float64 handles.  gram_count < 0: the statistics of the
 * batch are already complete in this handle (row-slab mode, cvmx_slab_finalize_stats) and only the Grams are summed. */
int32_t cvmx_sharded_finish_peers(cvmx_t* h, int64_t batch_f0, int64_t batch_f1, int64_t f0, int64_t f1, uint32_t want,
                                  const void* const* peer_bufs, int32_t n_peers, int64_t gram_count, void* out_XTX,
                                  void* out_XTY, void* out_stats, void* out_scal, int32_t* out_status);

/*
 * Row-slab mode (BASELINE config 5: N = 2M x K = 5000 float64 is 80 GB - the rows are sharded across the GPUs of a box
 * instead of replicated).  One handle per rank holds rows [row0, row0 + N_local) of the N_glob-row data set; the same
 * reference code as cvmx_fit / cvmx_training_batch is replaced (cvmatrix/cvmatrix.py:1209-1243 fit, :589-752 fold
 * statistics, :1001-1009 kernel matrices), with the row dimension of every reduction cut at the slab boundaries:
 *   - Gram totals and fold Grams are sums over rows: per-slab partials, reduced across ranks by the caller
 *     (all-reduce of cvmx_totals_ptr(); cvmx_sharded_gram with row shard 0 of 1 + cvmx_sharded_finish_peers);
 *   - numpy's column sums are sequential over rows, so they are CHAINED slab to slab: a rank continues the running
 *     sums it receives from the previous rank and hands them on (carry buffers in the model dtype);
 *   - numpy's weight sums are pairwise trees over all rows, which cannot be cut: every rank keeps the whole weight
 *     vector and the global validation index sets (small) and evaluates them itself.
 * Folds must list their rows in ascending order (a Partitioner always does), so that a fold's rows on rank r all
 * precede those on rank r + 1.  K >= 2 and M != 1 (a single column is summed pairwise over all rows by numpy).
 *   cvmx_fit_end_slab        : completes cvmx_fit_begin(N_local, ...) / cvmx_fit_rows.  carry_sum / carry_sumsq: device
 *                              rows of ld elements (NULL on the first rank) = the moment chains after the previous
 *                              slab; afterwards cvmx_moments_ptr() holds the chains after THIS slab (send them on; the
 *                              last rank's are final: write them back into cvmx_moments_ptr() on every rank).  w_glob:
 *                              device vector of all N_glob weights (NULL when unweighted), copied.  cvmx_totals_ptr()
 *                              holds this slab's partial [XtWX | XtWY]: all-reduce(sum) it across ranks.
 *   cvmx_set_folds           : the LOCAL validation sets (rows of this slab, numbered from 0), as usual;
 *   cvmx_set_weight_folds    : the same folds as GLOBAL row numbers (host arrays), for the weight sums;
 *   cvmx_slab_fold_sums      : carry [f1 - f0][2][ld] (device, model dtype, in / out): the folds' raw column sums
 *                              (sum w z, sum w z z) after the previous slab -> after this slab (zeros on the first rank);
 *   cvmx_slab_finalize_stats : raw = the completed sums of the last rank (same layout) -> weight masses, means, stds of
 *                              folds [f0, f1) in the handle's statistics buffer, ready for cvmx_sharded_finish_peers
 *                              (called with gram_count < 0: no statistics rows to sum).
 */
int32_t cvmx_fit_end_slab(cvmx_t* h, const void* carry_sum, const void* carry_sumsq, const void* w_glob, int64_t N_glob, int64_t row0);

/* Decoupled slab chain (float64).  The chained column sums above make rank r wait for rank r - 1, but only the LAST pass of
 * the binade scan (kernels_scan.cuh: one exact addition per 256 rows) needs the exact incoming chains; the streaming
 * passes need the running sum at the slab's first row only approximately - and that is the sum of the earlier slabs'
 * approximate totals, which the ranks all-gather (4 ld values per slab and fold).  The same numpy sums are replaced
 * (cvmatrix/cvmatrix.py:1231-1241 fit, :709-737 folds); results stay bit-identical to the sequential chain.
 *   cvmx_slab_scan_local   : f0 < 0: the fit totals of this slab, after the last cvmx_fit_rows (w_glob / N_glob / row0 as
 *                            for cvmx_fit_end_slab, which must follow with the same values; also runs everything of it
 *                            that does not depend on the previous slab).  f0 >= 0: folds [f0, f1) of the local CSR.
 *                            tot_out [folds][2 chains][2][ld] float64 (device): this slab's approximate sums and sums of
 *                            magnitudes.  *applicable = 0: slab too small / float32 - nothing was done, use the plain
 *                            chained calls.  Every rank must take the same path (all-reduce the flag).
 *   cvmx_slab_scan_prepare : start = the sum of tot_out over all EARLIER slabs (zeros on the first), same layout.
 *   then cvmx_fit_end_slab / cvmx_slab_fold_sums with the exact carry as before: they run only the last pass. */
/* Optional, right after cvmx_fit_begin of a row slab: hands over the global weights early (same w_glob / N_glob / row0 as
 * the cvmx_fit_end_slab that follows) so that the weight sums - ONE CTA walking numpy's pairwise tree over all N_glob
 * weights (cvmatrix/cvmatrix.py:1219-1229), ~1 ms at N = 1M - run on a side stream while the rows are still uploading. */
int32_t cvmx_slab_begin(cvmx_t* h, const void* w_glob, int64_t N_glob, int64_t row0);
int32_t cvmx_slab_scan_local(cvmx_t* h, int64_t f0, int64_t f1, const void* w_glob, int64_t N_glob, int64_t row0, double* tot_out,
                             int32_t* applicable);
int32_t cvmx_slab_scan_prepare(cvmx_t* h, int64_t f0, int64_t f1, const double* start);
int32_t cvmx_set_weight_folds(cvmx_t* h, const int64_t* offsets, const int64_t* indices, int64_t P);
int32_t cvmx_slab_fold_sums(cvmx_t* h, int64_t f0, int64_t f1, void* carry);
int32_t cvmx_slab_finalize_stats(cvmx_t* h, int64_t f0, int64_t f1, const void* raw);

/* The validation rows of CSR fold `fold` for the caller's next step (predicting the held-out rows with a model built
 * from the training matrices - what ikpls does after training_XTX_XTY, cvmatrix/partitioner.py:27-31): out_X [n_val, K]
 * = X[val], out_Y [n_val, M] = Y[val] (either may be NULL), optionally centred / scaled with training-set statistics:
 * `stats` is [2][K+M] (mean row, std row: the out_stats layout of cvmx_training_batch) in `mem`, `apply` a mask of
 * CVMX_CENTER_X | CVMX_CENTER_Y | CVMX_SCALE_X | CVMX_SCALE_Y; each op is individually rounded, so the result equals
 * numpy's (X[val] - X_mean) / X_std bit for bit.  `mem` applies to stats and to both outputs. */
int32_t cvmx_validation_rows(cvmx_t* h, int64_t fold, const void* stats, uint32_t apply, void* out_X, void* out_Y,
                             int32_t mem);

/*
 * Cross-validated PLS regression over folds [fold_begin, fold_end) of the CSR - the consumer of the training matrices
 * (ikpls after training_XTX_XTY, cvmatrix/partitioner.py:27-31).  Per fold, from XTX / XTY and the statistics exactly as
 * cvmx_training_batch(XTX | XTY) forms them: Improved Kernel PLS, Algorithm 2 (Dayal & MacGregor 1997) with A =
 * n_components components in float64 (M > 1: the direction is the dominant eigenvector of XTY_a^T XTY_a; a fold stops
 * early when ||XTY_a q|| <= 64 eps ||XTY_0||_F or t^T t <= 0, later coefficients repeat the last ones), then the
 * validation rows x_i of the fold predict y^_i = ((x_i - mu_X) / sigma_X) B_a * sigma_Y + mu_Y (each statistic applied
 * iff its flag is set) for a = 0 .. A-1.  With P' = fold_end - fold_begin, in the handle's dtype unless noted:
 *   out_press      [P', A, M]     sum over the validation rows (as stored: repeats count) of w_i (y_im - y^_im)^2
 *   out_sum_w_val  [P']           sum of the validation weights (row count when unweighted)
 *   out_B          [P', A, K, M]  coefficients B_a (may be NULL)
 *   out_n_fitted   [P'] int32     components fitted before the fold stopped (<= A)
 *   out_status     [P'] int32     CVMX_FOLD_* bits
 * Folds whose status bits make training_XTX_XTY raise (cvmatrix/cvmatrix.py:625-629, 1074-1078) get NaN press and B and
 * n_fitted = 0.  The range is processed in windows of about 1 GiB of device scratch; a range that fits one window reuses
 * the fold Grams kept by cvmx_fit_folds.  M = 0 gives CVMX_ERR_NO_Y; A outside [1, K] or M > 128 CVMX_ERR_INVALID.
 * `mem` applies to all five outputs.  Results do not depend on the launch geometry: identical calls give identical bits.
 */
int32_t cvmx_pls_cv(cvmx_t* h, int64_t fold_begin, int64_t fold_end, int64_t n_components, void* out_press,
                    void* out_sum_w_val, void* out_B, int32_t* out_n_fitted, int32_t* out_status, int32_t mem);

/*
 * Cross-validated ridge regression over folds [fold_begin, fold_end) of the CSR for L penalties - the other linear model
 * fitted from the training matrices (the caller's per-fold np.linalg.solve(XTX + lambda I, XTY) after
 * training_XTX_XTY, cvmatrix/partitioner.py:27-31).  Per fold f and penalty lambda_l = alphas[l] (a HOST array of L
 * finite values >= 0, 1 <= L <= 1024; copied to the device once per call), from XTX / XTY and the statistics exactly
 * as cvmx_training_batch(XTX | XTY) forms them: B = (XTX + lambda_l I)^-1 XTY by a blocked Cholesky factorisation in
 * float64 (lambda is added to the diagonal of the matrix as formed, so with scale_X it penalises the standardised
 * coefficients), then the validation rows x_i of the fold predict y^_i = ((x_i - mu_X) / sigma_X) B * sigma_Y + mu_Y
 * (each statistic applied iff its flag is set).  With P' = fold_end - fold_begin, in the handle's dtype unless noted:
 *   out_press      [P', L, M]     sum over the validation rows (as stored: repeats count) of w_i (y_im - y^_im)^2
 *   out_sum_w_val  [P']           sum of the validation weights (row count when unweighted)
 *   out_B          [P', L, K, M]  coefficients (may be NULL)
 *   out_info       [P', L] int32  0, or the 1-based column of the first pivot that was not > 0 (NaN included), as
 *                                 LAPACK dpotrf reports it; such a pair gets NaN press and B
 *   out_status     [P'] int32     CVMX_FOLD_* bits
 * Folds whose status bits make training_XTX_XTY raise (cvmatrix/cvmatrix.py:625-629, 1074-1078) get NaN press and B for
 * every penalty and info 0.  Folds are processed in windows and the penalties of a window in passes, as
 * cvmx_ridge_plan says; a range that fits one window reuses the fold Grams kept by cvmx_fit_folds.  M = 0 gives
 * CVMX_ERR_NO_Y; M > 128, a bad penalty list, a row-slab handle or a shape cvmx_ridge_plan calls infeasible give
 * CVMX_ERR_INVALID before anything is launched.  `mem` applies to all five outputs.  Results do not depend on the launch
 * geometry, the windows or the passes: identical calls give identical bits.
 */
int32_t cvmx_ridge_cv(cvmx_t* h, int64_t fold_begin, int64_t fold_end, const double* alphas, int64_t L, void* out_press,
                      void* out_sum_w_val, void* out_B, int32_t* out_info, int32_t* out_status, int32_t mem);

/*
 * cvmx_pls_cv / cvmx_ridge_cv that also return the out-of-fold predictions (cvmx_pls_cv and cvmx_ridge_cv are these
 * calls with out_pred = NULL; every other output is bit-identical with and without predictions).  The predictions are
 * in CSR order over the call's fold range: with off the CSR offsets and n = off[fold_end] - off[fold_begin], row j
 * belongs to CSR entry off[fold_begin] + j (repeats kept as stored), in the handle's dtype (float32: rounded once from
 * the float64 value), `mem` like the other outputs:
 *   PLS    out_pred [n, A, M]  row j, component a: the prediction with a + 1 components whose residual PRESS adds,
 *                              ((x - mu_X) / sigma_X) B_a * sigma_Y + mu_Y; a fold that stopped early repeats its last
 *                              fitted component's predictions; n_fitted = 0 predicts mu_Y if centred, else 0
 *   ridge  out_pred [n, L, M]  the same for penalty l; NaN for a pair with info != 0
 * Rows of a fold refused by its status bits are NaN; empty folds have no rows.  out_pred may be NULL.  Host outputs are
 * staged through at most 256 MiB of device memory per PRESS launch, or one 32-row chunk's predictions if that is larger.
 */
int32_t cvmx_pls_cv_predict(cvmx_t* h, int64_t fold_begin, int64_t fold_end, int64_t n_components, void* out_press,
                            void* out_sum_w_val, void* out_B, int32_t* out_n_fitted, int32_t* out_status,
                            void* out_pred, int32_t mem);
int32_t cvmx_ridge_cv_predict(cvmx_t* h, int64_t fold_begin, int64_t fold_end, const double* alphas, int64_t L,
                              void* out_press, void* out_sum_w_val, void* out_B, int32_t* out_info, int32_t* out_status,
                              void* out_pred, int32_t mem);

/* Host-only (no CUDA call): the launch plan cvmx_ridge_cv uses for K columns of X, M of Y, L penalties and P folds of
 * the given dtype, output memory (`mem`) and whether B is wanted.  plan[CVMX_RIDGE_PLAN_LEN] receives the folds per
 * window, the penalties per pass, the device scratch bytes of a pass and the byte offset at which each of its arrays
 * ends, the PRESS partials of one launch, the largest grid (x, y) of every kernel (CVMX_RIDGE_GRID + 2 * CVMX_RK_*) and
 * its dynamic shared memory (CVMX_RIDGE_SMEM + CVMX_RK_*).  A pass holds every penalty of its folds, or one fold.
 * Returns CVMX_OK with plan[CVMX_RIDGE_FEASIBLE] = 1, or CVMX_ERR_INVALID (feasible = 0) for arguments out of range or a
 * shape that cannot run within the device limits (grid dimensions, 227 KB of shared memory a block, 32 GiB of scratch
 * for one fold and one penalty). */
int32_t cvmx_ridge_plan(int64_t K, int64_t M, int64_t L, int64_t P, int32_t dtype, int32_t mem, int32_t want_B, int64_t* plan);

enum {
  CVMX_RK_LOAD = 0, CVMX_RK_POTRF, CVMX_RK_TRSM, CVMX_RK_SYRK, CVMX_RK_BSOLVE_DIAG, CVMX_RK_BSOLVE_UPDATE,
  CVMX_RK_PRESS, CVMX_RK_PRESS_ACCUM, CVMX_RK_FINISH, CVMX_RK_COEFS, CVMX_RK_COUNT
};
enum {
  CVMX_RIDGE_FEASIBLE = 0, CVMX_RIDGE_FOLDS_PER_WINDOW, CVMX_RIDGE_PENALTIES_PER_PASS, CVMX_RIDGE_SCRATCH_BYTES,
  CVMX_RIDGE_END_A, CVMX_RIDGE_END_STATE, CVMX_RIDGE_END_ACC, CVMX_RIDGE_END_ACC_W, CVMX_RIDGE_END_PRESS,
  CVMX_RIDGE_END_INFO, CVMX_RIDGE_END_B, CVMX_RIDGE_END_SUM_W, CVMX_RIDGE_END_STATUS,
  CVMX_RIDGE_WINDOW_BYTES,       /* XTX / XTY of one window (model dtype) */
  CVMX_RIDGE_PART_BYTES,         /* PRESS partials of one launch */
  CVMX_RIDGE_CHUNKS_PER_LAUNCH,  /* PRESS chunks of one launch */
  CVMX_RIDGE_GRID = 16,
  CVMX_RIDGE_SMEM = CVMX_RIDGE_GRID + 2 * CVMX_RK_COUNT,
  CVMX_RIDGE_PLAN_LEN = CVMX_RIDGE_SMEM + CVMX_RK_COUNT
};

/* Per-kernel device timing for bench.py's roofline line: while enabled, CUDA events are recorded on the
 * handle's stream around the statistics kernels (ms[0]), the Gram kernel (ms[1]) and the split-reduce
 * kernel (ms[2]); cvmx_profile_read synchronises, returns the accumulated milliseconds and span counts
 * (arrays of 3) since the last read, and resets them. */
int32_t cvmx_profile_enable(cvmx_t* h, int32_t on);
int32_t cvmx_profile_read(cvmx_t* h, double* ms, int64_t* count);

/* Host-only helper (no CUDA call): CSR of validation sets from integer fold labels, replacing the Python loop of
 * Partitioner._init_folds_dict (cvmatrix/partitioner.py:101-107).  labels[i] in [lo, lo + span); folds are ordered
 * by first appearance; first_rows[k] = first row of fold k, offsets / indices = CSR (indices ascending per fold).
 * scratch needs 2 * span int64.  Returns the number of folds, or -1 on bad arguments. */
int64_t cvmx_partition_labels(const int64_t* labels, int64_t n, int64_t lo, int64_t span, int64_t* scratch,
                              int64_t* first_rows, int64_t* offsets, int64_t* indices);

/* Introspection used by tests / bench: number of kernels launched by this handle so far, and
 * the padded leading dimension of the device matrices. */
int64_t cvmx_launch_count(const cvmx_t* h);
int64_t cvmx_ld(const cvmx_t* h);

/* Column sums in numpy's order (np.sum(A, axis=0): sequential per column, cvmatrix/cvmatrix.py:709, 716, 727, 737,
 * 1231-1241) are evaluated either as dependent-add chains or, for float64, by the bit-identical "binade scan"
 * (csrc/kernels_scan.cuh).  mode 0: chains only; 1 (default): scan when the chains are on the critical path;
 * 2: scan whenever a fold has >= 1024 rows.  Also settable with the environment variable CVMX_SCAN at cvmx_create.
 * cvmx_scan_launch_count: how many moment launches went through the scan so far. */
int32_t cvmx_set_scan_mode(cvmx_t* h, int32_t mode);
int64_t cvmx_scan_launch_count(const cvmx_t* h);

/* Leave-one-out and leave-few-out batches (every fold of a cvmx_training_batch range holds at most 16 rows; the rank-n
 * downdate of cvmatrix/cvmatrix.py:1001-1009 is bound by writing K x (K + M) results).  mode 0 (default): streaming
 * form - operand rows prepared once per fold, per element a few FMAs and a multiplication by precomputed reciprocal
 * standard deviations, matrices within ~1e-15 (relative Frobenius) of the reference and exactly symmetric; mode 1: exact
 * form - numpy's operation order with IEEE division, matrices bit-identical to the reference for one-row folds.
 * Statistics are bit-identical in both.  Also settable with the environment variable CVMX_LOO_EXACT=1 at cvmx_create. */
int32_t cvmx_set_loo_mode(cvmx_t* h, int32_t mode);

#ifdef __cplusplus
}
#endif
#endif /* CVMX_H_ */
