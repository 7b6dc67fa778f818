/*
 * rs_knn.h — C ABI of the B200-native KNN hot path (librs_knn_b200.so).
 *
 * This is the drop-in boundary for Oneaccount1/recommend-sys' memory-based KNN
 * recommender.  Each entry point names the reference interface it replaces (paths are
 * relative to the reference repository).  The reference-side binding (cgo) is in
 * recommend-sys_b200/go/ and INTEGRATION.md.
 *
 * Conventions
 *   - plain C types only: pointers + sizes, no torch / C++ types in any signature;
 *   - every function returns RS_OK (0) or a negative RS_ERR_* code; rs_last_error()
 *     returns a thread-local message for the last failure on the calling thread;
 *   - host-pointer entry points borrow their arguments for the duration of the call only
 *     (cgo forbids C retaining Go pointers); `_device` variants take CUDA device pointers
 *     that must stay valid until the handle's stream has drained;
 *   - ids are INNER ids (core/data.go:137-151 — order of first appearance), -1 is the
 *     reference's `newID` (core/data.go:129);
 *   - "left" is the side similarities are computed over (users if userBased, else items,
 *     core/knn.go:154-162), "right" is the other side;
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails
 *     with RS_ERR_CUDA;
 *   - threading: distinct handles may be used concurrently from any threads; calls on ONE handle
 *     are serialised internally (a per-handle mutex held for the whole call), so concurrent
 *     Predict calls on a fitted estimator are safe, as they are in the reference;
 *   - Fit is asynchronous: rs_knn_fit returns once the inputs are consumed and validated, the
 *     similarity kernel may still be running.  A device fault in it surfaces on the next call that
 *     waits for the stream; callers that want Fit errors eagerly call rs_knn_synchronize.
 */
#ifndef RS_KNN_H
#define RS_KNN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RS_OK 0
#define RS_ERR_INVALID (-1)     /* bad argument / call order                              */
#define RS_ERR_CUDA (-2)        /* CUDA runtime or driver failure (incl. no device)       */
#define RS_ERR_UNSUPPORTED (-3) /* input outside what the device path supports            */
#define RS_ERR_OOM (-4)         /* device allocation failed                               */
#define RS_ERR_DUPLICATE (-5)   /* the same (left,right) pair appears twice in the ratings */

/* core/sim.go: Cosine :10, MSD :28, Pearson :47.  PEARSON_BASELINE is an extension
 * (named by the north star, absent from the reference). */
enum rs_sim { RS_SIM_COSINE = 0, RS_SIM_MSD = 1, RS_SIM_PEARSON = 2, RS_SIM_PEARSON_BASELINE = 3,
              /* SURVEY.md §8 f-2, the step next to the KNN path: the Slope One deviation matrix
               * (core/slope_one.go:47-93) instead of a similarity.  Fit with left = items, right =
               * users; rs_knn_sims_rows returns dev rows (0 = unset, antisymmetric);
               * rs_knn_predict_batch(left = item, right = user) is SlopeOne.Predict
               * (core/slope_one.go:22-45).  Integer ratings only (tensor path). */
              RS_SIM_SLOPE_ONE = 4 };
/* core/knn.go:10-15 and the four constructors core/knn.go:50-73 */
enum rs_knn_type { RS_KNN_BASIC = 0, RS_KNN_CENTERED = 1, RS_KNN_ZSCORE = 2, RS_KNN_BASELINE = 3 };
/* How Pearson is evaluated.
 *   EXACT: FP64 replay of core/sim.go:65-80 in the reference's accumulation order
 *          (ascending right id) — bit-identical similarities and neighbour lists.
 *   SUMS : the six integer co-rating sums on int8 tensor cores + an FP64 epilogue that forms
 *          L / (sqrt(Mi) * sqrt(Ni)) from exact integers: within 4 ulps of the exact value (6 once
 *          |L|, Mi or Ni pass 2^53), NaN exactly where Mi * Ni == 0, +0.0 where L == 0, symmetric;
 *          equal to EXACT within 1e-9*max(1,|s|), not bit-identical (SURVEY.md hazard 2). */
enum rs_pearson_mode { RS_PEARSON_EXACT = 0, RS_PEARSON_SUMS = 1 };
/* Which device kernel computes the similarities.
 *   AUTO  : Pearson in EXACT mode and any rating set that is not small integers run STREAM.
 *           Otherwise (Cosine / MSD / Pearson SUMS on integer ratings in [-11, 11], where both
 *           kernels are bit-exact or within the stated tolerance) the faster one by a two-term
 *           cost model: dense int8 work N(N-1)/2 * 2*G*K against the co-rated triples counted
 *           during Fit (csrc/api.cu tensor_faster; constants measured on B200).
 *   TENSOR: tcgen05.mma.kind::i8 masked contractions (fails with RS_ERR_UNSUPPORTED if
 *           the ratings are not small integers, or if its int32 sums could overflow: with
 *           m = the largest |rating| and n2 = the second-longest left row, 4 m^2 n2 > 2^31-1
 *           for MSD, m^2 n2 for Cosine and Pearson SUMS, 2 m n2 for Slope One; AUTO then runs
 *           STREAM).
 *   STREAM: FP64 CUDA-core sparse replay: work proportional to the co-rated triples,
 *           accumulation in the reference's order; accepts ANY float64 ratings (no limit on
 *           the number of distinct values; NaN ratings are refused). */
enum rs_sim_path { RS_PATH_AUTO = 0, RS_PATH_TENSOR = 1, RS_PATH_STREAM = 2 };
/* What Fit leaves resident in HBM.
 *   MATRIX: the dense similarity rows of this handle's shard (what core/knn.go:157,161
 *           keeps; required by Predict).
 *   TOPK  : only the per-row top-`topk` neighbour lists; the N x N matrix is never resident
 *           (BASELINE.json config 4).  With shard_count >= 1, Cosine / MSD on integer ratings and a
 *           problem large enough for the CTA-pair tensor kernel, the lists are selected IN the
 *           tensor kernel's epilogue (threshold compare, candidate append, merge between the waves
 *           of the tile schedule): no similarity row is ever stored.  Otherwise the rows are produced
 *           slab by slab into a bounded work buffer and reduced to the lists by selection kernels. */
enum rs_store { RS_STORE_MATRIX = 0, RS_STORE_TOPK = 1 };

typedef struct rs_knn rs_knn; /* opaque handle; one per estimator copy (core/eval.go:29-30) */

/* Mirrors the Parameters keys the path reads (core/knn.go:79-81,145-148) plus the
 * device-side choices.  Fill with rs_knn_params_default() first. */
typedef struct rs_knn_params {
    int32_t sim;          /* enum rs_sim;        Parameters["sim"], default MSD           */
    int32_t knn_type;     /* enum rs_knn_type;   fixed by the constructor                 */
    int32_t k;            /* Parameters["k"], default 40                                  */
    int32_t min_k;        /* Parameters["mink"], default 1                                */
    int32_t device;       /* CUDA device ordinal; -1 = the calling thread's current device */
    int32_t pearson_mode; /* enum rs_pearson_mode, default EXACT                          */
    int32_t sim_path;     /* enum rs_sim_path, default AUTO                               */
    int32_t store;        /* enum rs_store, default MATRIX                                */
    int32_t topk;         /* neighbours per row for RS_STORE_TOPK / rs_knn_topk           */
    int32_t reserved0;
    int64_t row_begin;    /* shard of left rows this handle owns: [row_begin,row_end);    */
    int64_t row_end;      /*   0,0 = all rows.  One handle per GPU when row-sharding.     */
    double shrinkage;     /* PearsonBaseline extension: (n-1)/(n-1+shrinkage), 0 = off    */
                          /* RS_STORE_MATRIX with shard_count >= 2: CYCLIC ROW SHARDS.  The left rows are   */
                          /*   dealt in blocks of 32 (block b -> shard b % shard_count); the handle        */
                          /*   computes ONE triangle of the rows it owns (every pair once across the       */
                          /*   shards, exact sparse path) and the other triangle is pulled from the peers'  */
                          /*   matrices over NVLink by rs_knn_mirror (after rs_knn_peer_import).  Predict   */
                          /*   then serves the test pairs whose left row the handle owns (NaN for others;  */
                          /*   rs_knn_predict_batch_sharded_device: +0.0 for others, for an all-reduce).   */
    int32_t shard_count;  /* RS_STORE_TOPK.  0 (default): the handle computes the full rows of             */
    int32_t shard_index;  /*   [row_begin,row_end) and keeps their lists.  >= 1: SYMMETRIC SLABS — the */
                          /*   left rows are cut into slabs dealt to the shards in snake order          */
                          /*   (0..c-1, c-1..0, ...); the handle computes its slabs, of each only the part */
                          /*   right of the diagonal; every pair {i,j} it computes feeds the list of  */
                          /*   row i AND of row j, so no pair is computed twice (half the work) and  */
                          /*   the handle holds PARTIAL lists for ALL n_left rows: complete when      */
                          /*   shard_count == 1, else to be united across the shard_count handles     */
                          /*   with rs_knn_topk_union_device after an all-gather.                      */
} rs_knn_params;

/* Per-handle counters since creation / the last rs_knn_profile_reset: device time of the
 * named kernels measured with CUDA events on the handle's stream, and launch counts. */
typedef struct rs_knn_profile {
    double sim_kernel_ms;      /* dominant similarity kernel (tensor or stream)            */
    double predict_kernel_ms;  /* gather-select-reduce kernel                              */
    double prep_ms;            /* CSR build, packing, statistics                           */
    int64_t sim_launches;
    int64_t predict_launches;
    int64_t total_launches;    /* every kernel this library launched on the handle         */
    int32_t sim_path_used;     /* enum rs_sim_path actually taken by the last Fit          */
    int32_t reserved0;
    double corated_triples;    /* sum over right rows of cnt*(cnt-1)/2 of the last Fit (rs_knn_update leaves it):
                                * the work of the exact sparse path, input of the RS_PATH_AUTO model */
} rs_knn_profile;

/* Thread-local message of the last error on this thread ("" if none). */
const char *rs_last_error(void);
/* Library/ABI version, and the number of visible CUDA devices (0 when there is none). */
int32_t rs_knn_abi_version(void);
int32_t rs_knn_device_count(void);

/* Defaults of core/knn.go:79-81,145-148 (sim=MSD, k=40, mink=1), device -1, AUTO path. */
int32_t rs_knn_params_default(rs_knn_params *p);

/* Replaces NewKNN / NewKNNWithMean / NewKNNWithZScore / NewKNNBaseLine (core/knn.go:50-73)
 * + SetParams (core/base.go:64-66). */
int32_t rs_knn_create(const rs_knn_params *p, rs_knn **out);
/* Go side: Close() + finalizer; the handle lives in an unexported field so the gob
 * round-trip in Copy (core/dump.go:37-43) never sees it. */
int32_t rs_knn_destroy(rs_knn *h);

/* Run all of this handle's work on `cuda_stream` (a cudaStream_t / CUstream; NULL is the
 * legacy default stream), e.g. the caller's current stream.  use_own != 0 switches back to
 * the non-blocking stream the handle created for itself (the default). */
int32_t rs_knn_set_stream(rs_knn *h, void *cuda_stream, int32_t use_own);

/* Replaces KNN.Fit (core/knn.go:143-217) after the Go side has built the inner-id COO:
 * left[i], right[i], rating[i] for i in dataset order (the order matters: Means/StdDevs are
 * accumulated in it, core/data.go:222-235, core/knn.go:167-177).
 *   global_mean       TrainSet.GlobalMean (core/data.go:134)
 *   left_bias         Bias of the left side for RS_KNN_BASELINE (core/knn.go:179-187), else NULL
 *   right_bias,global_bias  only for RS_SIM_PEARSON_BASELINE (both bias vectors), else NULL/0
 * Host pointers; copied to the device inside the call, and free to reuse when it returns.  The call
 * returns once the inputs are consumed and validated (errors in the data are reported here); the
 * similarity kernel may still be running — every call that needs its result is ordered behind it on
 * the handle's stream, and rs_knn_synchronize waits for it explicitly. */
int32_t rs_knn_fit(rs_knn *h, const int32_t *left, const int32_t *right, const double *rating,
                   int64_t nnz, int32_t n_left, int32_t n_right, double global_mean,
                   const double *left_bias, const double *right_bias, double global_bias);
/* Same with every array already resident in device memory. */
int32_t rs_knn_fit_device(rs_knn *h, const int32_t *d_left, const int32_t *d_right,
                          const double *d_rating, int64_t nnz, int32_t n_left, int32_t n_right,
                          double global_mean, const double *d_left_bias,
                          const double *d_right_bias, double global_bias);

/* Replaces DataSet.Predict (core/data.go:98-105) looping over KNN.Predict
 * (core/knn.go:75-141): out[i] = prediction for (left[i], right[i]); -1 on either side
 * returns GlobalMean.  Ties between equal similarities are broken by ascending inner id
 * (the canonical policy; Go's sort.Sort is unstable, SURVEY.md hazard 1).
 * Requires RS_STORE_MATRIX; left ids outside the handle's row shard yield NaN.  k <= 256. */
int32_t rs_knn_predict_batch(rs_knn *h, const int32_t *left, const int32_t *right, int64_t n,
                             double *out);
int32_t rs_knn_predict_batch_device(rs_knn *h, const int32_t *d_left, const int32_t *d_right,
                                    int64_t n, double *d_out);
/* The neighbours one prediction used, in accumulation order (for parity tests of the
 * neighbour indices).  Returns the count in *n_out (0 = GlobalMean branch). */
int32_t rs_knn_predict_neighbors(rs_knn *h, int32_t left, int32_t right, int32_t cap,
                                 int32_t *ids, double *sims, int32_t *n_out);

/* Backs the exported KNN.Sims field / gob Save on demand (core/knn.go:21, core/dump.go:11):
 * copies rows [row0,row0+nrows) of the N x N float64 matrix (NaN = unset, diagonal NaN,
 * core/utils.go:110-120) to `out` (nrows*N doubles).  Rows must lie in the shard. */
int32_t rs_knn_sims_rows(rs_knn *h, int64_t row0, int64_t nrows, double *out);

/* Per-row top-k neighbour lists of the shard under (similarity desc, id asc), NaN skipped,
 * unused slots idx=-1/sim=NaN: idx, sim are (row_end-row_begin) x k.  Not an artefact of
 * the reference (it selects per prediction); this is BASELINE.json config 4's output.
 * The _device variant writes into device memory (for an NCCL all-gather across shards). */
int32_t rs_knn_topk(rs_knn *h, int32_t k, int32_t *idx, double *sim);
int32_t rs_knn_topk_device(rs_knn *h, int32_t k, int32_t *d_idx, double *d_sim);

/* Integer co-rating sums {count, sum_x, sum_y, sum_xx, sum_yy, sum_xy} of left rows
 * [row0,row0+nrows) against all N rows, straight from the tensor-core contraction
 * (out: nrows*N*6 int32, host).  Parity surface for "integer co-rating sums bit-exact".
 * RS_ERR_UNSUPPORTED when the sums could leave int32: m^2 n1 > 2^31-1, m = the largest
 * |rating|, n1 = the longest left row (the sums of a row with itself run over all of it). */
int32_t rs_knn_cosums(rs_knn *h, int64_t row0, int64_t nrows, int32_t *out);

/* KNN.Means / KNN.StdDevs (core/knn.go:24-25): n_left doubles each, host. */
int32_t rs_knn_means(rs_knn *h, double *out);
int32_t rs_knn_stddevs(rs_knn *h, double *out);

/* EXTENSION (BASELINE.json config 3 "ALS baselines"; SURVEY.md §8 f-3) — an alternative to
 * BaseLine.Fit (core/base.go:135-163), whose sequential SGD stays on the host: alternating least
 * squares baseline estimates computed on `device` (-1 = current) from the inner-id COO (host
 * pointers, dataset order), Surprise-style
 *     b_i = sum_{u in R(i)} (r_ui - mu - b_u) / (reg_i + |R(i)|),  then  b_u likewise,  n_epochs times,
 * mu = global_mean.  Writes user_bias[n_users], item_bias[n_items]; pass them (and mu as
 * global_bias) to rs_knn_fit for KNNBaseline / PearsonBaseline.  Selected from the host API with
 * Parameters["baseline"] = "als" (defaults regU 15, regI 10, nEpochs 10).  Parity unpinned: the
 * reference has no ALS; checked against oracle/knn_oracle.c:or_baseline_als bit for bit. */
int32_t rs_baseline_als(int32_t device, const int32_t *users, const int32_t *items, const double *ratings,
                        int64_t nnz, int32_t n_users, int32_t n_items, double global_mean, double reg_u,
                        double reg_i, int32_t n_epochs, double *user_bias, double *item_bias);

/* Unites the partial neighbour lists of `n_lists` shards (device pointers, layout
 * [n_lists][n_rows][k], idx -1 = empty) into the final top-k lists [n_rows][k] (similarity desc, id
 * asc), on `cuda_stream`.  Every (row, neighbour) pair must occur in at most one partial list —
 * which is what symmetric-slab handles (shard_count >= 1) produce.  n_lists * k <= 2048. */
int32_t rs_knn_topk_union_device(int32_t n_lists, int64_t n_rows, int32_t k, const int32_t *d_idx_all,
                                 const double *d_sim_all, int32_t *d_idx, double *d_sim, void *cuda_stream);

/* TOP-N RECOMMENDATION.  A query is an inner id of one side; its TARGETS are all ids of the other side:
 *   RS_SIDE_RIGHT query q: score(t) = Predict(left = t, right = q) — item-based mode, the user is the right side;
 *   RS_SIDE_LEFT  query q: score(t) = Predict(left = q, right = t) — user-based mode.
 * Every score is bit-identical to what rs_knn_predict_batch returns for the same pair with the current k / mink
 * (rs_knn_set_k applies); NaN and +-Inf scores (sum of weights <= 0) are reproduced as they are.  Targets the query
 * rated (its row of the left or right ratings) are excluded: their score is NaN.  A query of -1 (newID) scores
 * GlobalMean everywhere.  The host variants refuse ids outside [-1, n_side) with RS_ERR_INVALID; the _device
 * variants treat them as -1.
 * Ranking: the top n_top targets by (score desc, target inner id asc) under the order-preserving key of the
 * neighbour lists; NaN is never listed, +Inf ranks first and -Inf last, +-0 tie by id and -0.0 is reported as
 * -0.0; unused slots are id -1 / score NaN.  A -1 query therefore lists the first n_top target ids.
 * Limits: 1 <= n_top <= 512, k <= 256, n >= 0.  Only RS_STORE_MATRIX handles that hold all rows: RS_STORE_TOPK is
 * refused like Predict refuses it, row shards (row_begin/row_end or shard_count >= 2) and RS_SIM_SLOPE_ONE with
 * RS_ERR_UNSUPPORTED.  Queries are scored in batches into a device slab of full score rows (~256 MiB). */
enum rs_side { RS_SIDE_LEFT = 0, RS_SIDE_RIGHT = 1 };
/* Full score rows: out[n][n_targets] (n_targets = n_right for left queries, n_left for right queries). */
int32_t rs_knn_score_all(rs_knn *h, int32_t side, const int32_t *queries, int64_t n, double *out);
int32_t rs_knn_score_all_device(rs_knn *h, int32_t side, const int32_t *d_queries, int64_t n, double *d_out);
/* The n_top best targets of each query: ids[n][n_top] (inner ids), scores[n][n_top]. */
int32_t rs_knn_recommend(rs_knn *h, int32_t side, const int32_t *queries, int64_t n, int32_t n_top, int32_t *ids,
                         double *scores);
int32_t rs_knn_recommend_device(rs_knn *h, int32_t side, const int32_t *d_queries, int64_t n, int32_t n_top,
                                int32_t *d_ids, double *d_scores);
/* TOP-N RECOMMENDATION ON ROW SHARDS (cyclic shards after rs_knn_mirror, or row_begin/row_end shards): every shard
 * gets the SAME queries and answers the part it owns ("owns": the cyclic block rule, resp. [row_begin, row_end)):
 *   RS_SIDE_RIGHT query q: the shard scores and lists only the targets (left rows) it owns; list ids are global inner
 *     ids.  A -1 query (an id out of range) scores GlobalMean on the shard's own targets.
 *   RS_SIDE_LEFT  query q: the owner of row q produces the whole list / row; every other shard an empty list (ids -1,
 *     scores NaN) or a +0.0 row.  A -1 query is answered by the shard that owns left row 0 only (cyclic shard 0, the
 *     contiguous shard with row_begin == 0), so that it is not listed twice.
 * rs_knn_recommend_sharded_device writes each shard's PARTIAL lists ids[n][n_top], scores[n][n_top]: all-gather them
 * and unite them with rs_knn_topk_union_device — in groups of at most 2048 / n_top lists, and the results again when
 * there are more shards; every target is in at most one partial list.  rs_knn_score_all_sharded_device writes rows
 * out[n][n_targets] in which the cells the shard does not answer are +0.0 (all bits zero) and its own rated targets
 * NaN: an integer SUM all-reduce of the 64-bit patterns over the shards assembles rs_knn_score_all.  Either way the
 * result is bit-identical to rs_knn_recommend / rs_knn_score_all on one handle of all rows at the same k / mink.
 * Refused: a handle that is not a row shard or a cyclic shard before rs_knn_mirror (RS_ERR_INVALID), RS_STORE_TOPK,
 * RS_SIM_SLOPE_ONE, and the limits of rs_knn_recommend.  The plain entry points keep refusing row shards. */
int32_t rs_knn_recommend_sharded_device(rs_knn *h, int32_t side, const int32_t *d_queries, int64_t n,
                                        int32_t n_top, int32_t *d_ids, double *d_scores);
int32_t rs_knn_score_all_sharded_device(rs_knn *h, int32_t side, const int32_t *d_queries, int64_t n,
                                        double *d_out);
/* TOP-N RECOMMENDATION FOR QUERIES GIVEN AS RATING LISTS ("fold-in"): users who signed up or rated after the Fit are
 * scored against the fitted model without a refit.  Query b is the list ids[ptr[b] .. ptr[b+1]), vals[...] of inner
 * ids of the TARGET side and their ratings, in the caller's order (it plays the role of the user's dataset order).
 *   RS_SIDE_RIGHT (item-based; ids are left ids): score(t) = Predict(left = t, right = q*), q* a right row whose
 *     ratings are the list.  The candidates are the list's entries in ascending id, their similarities row S[t], their
 *     statistics (means, stddevs, bias) the fitted ones.  The order of the list does not matter; a list equal to right
 *     row u's ratings gives rs_knn_score_all(RS_SIDE_RIGHT, u) bit for bit.
 *   RS_SIDE_LEFT (user-based; ids are right ids): S*[v] = Sim(list sorted by id, left row v) for every fitted left row
 *     v, with the reference's formulas, term order and IEEE operations (the exact sparse Fit's; Pearson's mean of the
 *     list summed in ascending id, NaN without a co-rating); then score(t) = Predict(left = q*, right = t) with the
 *     candidates R(t) weighted by S*.  The list's own mean / stddev (centered, z-score) are accumulated in the
 *     caller's order as Fit's are.  A list equal to left row u's ratings in dataset order gives
 *     rs_knn_score_all(RS_SIDE_LEFT, u) bit for bit.
 * The list's ids are the query's rated targets: NaN in score rows, never listed.  An empty list scores GlobalMean
 * everywhere (a -1 query).  Output layout, ranking rule, unused slots and n_top limits are rs_knn_score_all's /
 * rs_knn_recommend's.  NOT A REFIT: the given ratings enter neither the similarities between fitted rows, nor the
 * fitted means, nor GlobalMean.
 * Refused: RS_ERR_INVALID for an id outside [0, n_targets), ptr not starting at >= 0 or not non-decreasing, a NaN
 * rating; RS_ERR_DUPLICATE for an id twice in one list (the _device variants check on the device and read back a
 * few bytes); RS_ERR_UNSUPPORTED for RS_STORE_TOPK, RS_SIM_SLOPE_ONE, row shards, and for RS_SIDE_LEFT
 * RS_KNN_BASELINE / RS_SIM_PEARSON_BASELINE (no bias for the list's user) and Pearson in RS_PEARSON_SUMS mode (the
 * matrix is not the exact replay S* is); plus the limits of rs_knn_recommend.  Lists are scored in batches; for left
 * queries the S* rows share the ~256 MiB slab with the score rows. */
int32_t rs_knn_score_all_given(rs_knn *h, int32_t side, const int64_t *ptr, const int32_t *ids, const double *vals,
                               int64_t n, double *out);
int32_t rs_knn_score_all_given_device(rs_knn *h, int32_t side, const int64_t *d_ptr, const int32_t *d_ids,
                                      const double *d_vals, int64_t n, double *d_out);
int32_t rs_knn_recommend_given(rs_knn *h, int32_t side, const int64_t *ptr, const int32_t *ids, const double *vals,
                               int64_t n, int32_t n_top, int32_t *out_ids, double *out_scores);
int32_t rs_knn_recommend_given_device(rs_knn *h, int32_t side, const int64_t *d_ptr, const int32_t *d_ids,
                                      const double *d_vals, int64_t n, int32_t n_top, int32_t *d_out_ids,
                                      double *d_out_scores);

/* ADDING RATINGS TO A FITTED MODEL (an extension: the reference has no incremental Fit).  The ratings left[i],
 * right[i], rating[i] (inner ids, in call order) join the fitted ones, and the model becomes the one rs_knn_fit
 * returns for the union — the fitted ratings in their dataset order followed by these — with n_left x n_right ids and
 * GlobalMean global_mean, bit for bit: matrix, means, stddevs, Predict, recommendation and fold-in.  Only the
 * similarity rows (and columns) of the TOUCHED left ids are recomputed: the ids these ratings name, and the new ids
 * n_left_fitted .. n_left-1; a cell between two untouched rows keeps its value, which is the refit's (the same terms
 * in the same order).  n_left / n_right are the counts after the update, at least the fitted ones (larger ones add
 * ids; an id without ratings gets the empty row a Fit gives it).  nnz may be 0 (only new ids, or a new GlobalMean).
 * Host pointers are consumed when the call returns; the _device variant reads its arrays on the handle's stream.
 * The call returns once the ratings are validated and the work is queued; rs_knn_synchronize waits for it.
 * Refused before anything of the model is written, leaving it exactly as it was:
 *   RS_ERR_INVALID     the handle is not fitted, an id outside [0, n_left) x [0, n_right), a count smaller than the
 *                      fitted one, a null pointer with nnz > 0;
 *   RS_ERR_UNSUPPORTED a NaN rating; RS_STORE_TOPK; row shards (row_begin/row_end, shard_count >= 2);
 *                      RS_SIM_SLOPE_ONE; RS_KNN_BASELINE and RS_SIM_PEARSON_BASELINE (their biases come from a global
 *                      fit that every rating changes); Pearson in RS_PEARSON_SUMS mode (the recomputed rows are the
 *                      exact replay); a non-integer rating for a model fitted on integer ratings in [-11, 11] (such a
 *                      Fit keeps no dataset order of the values); more than 2^31-1 ratings in all;
 *   RS_ERR_DUPLICATE   a (left, right) pair the model holds already, or twice among these ratings;
 *   RS_ERR_OOM         the merged arrays or the grown matrix do not fit.
 * Memory: the merged arrays live in two blocks per array with a quarter of slack (the one the model reads and the one
 * the next update writes), so a sequence of updates stops allocating; a new left id grows the matrix in place while
 * ld = ceil(n_left / 16) * 16 does not change, else into a new block.  The int8 planes of rs_knn_cosums are dropped
 * and rebuilt for the union on its next call, into a block of their own that later rebuilds reuse while it is large
 * enough; rs_knn_profile's corated_triples stays the last Fit's. */
int32_t rs_knn_update(rs_knn *h, const int32_t *left, const int32_t *right, const double *rating, int64_t nnz,
                      int32_t n_left, int32_t n_right, double global_mean);
int32_t rs_knn_update_device(rs_knn *h, const int32_t *d_left, const int32_t *d_right, const double *d_rating,
                             int64_t nnz, int32_t n_left, int32_t n_right, double global_mean);
/* REMOVING OR CHANGING RATINGS OF A FITTED MODEL (an extension, the other half of rs_knn_update).  The pairs
 * (left[i], right[i]) are inner-id pairs the model holds.  rs_knn_remove drops them: the remaining ratings keep their
 * relative dataset order.  rs_knn_change gives pair i the rating rating[i] at its place in the dataset order (the same
 * value is allowed).  Afterwards the model is, bit for bit, what rs_knn_fit returns for the edited ratings in the edited
 * dataset order with the SAME n_left x n_right and GlobalMean global_mean: matrix, means, stddevs, Predict,
 * rs_knn_predict_neighbors, rs_knn_topk, score rows, recommendation lists, fold-in (_given) and rs_knn_cosums.  Inner
 * ids are never renumbered or dropped: an id left without ratings keeps the empty row a Fit gives it (NaN everywhere;
 * Predict falls back to GlobalMean).  Only the similarity rows (and columns) of the left ids the pairs name are
 * recomputed, as in rs_knn_update.  n may be 0 (a new GlobalMean only).  Host pointers are consumed when the call
 * returns; the _device variants read their arrays on the handle's stream.  The call returns once the pairs are
 * validated and the work is queued.
 * Refused before anything of the model is written, leaving it exactly as it was:
 *   RS_ERR_INVALID     the handle is not fitted, an id outside [0, n_left) x [0, n_right), a pair the model does not
 *                      hold, a null pointer with n > 0, a removal that would leave no rating (rs_knn_fit refuses
 *                      nnz = 0);
 *   RS_ERR_DUPLICATE   a pair named twice in one call;
 *   RS_ERR_UNSUPPORTED every model rs_knn_update refuses (RS_STORE_TOPK, row shards of both kinds, RS_SIM_SLOPE_ONE,
 *                      RS_KNN_BASELINE, RS_SIM_PEARSON_BASELINE, Pearson in RS_PEARSON_SUMS mode); a NaN change; a
 *                      change to a value outside the integers in [-11, 11] on a model fitted on that class;
 *   RS_ERR_OOM         as rs_knn_update.
 * The counts never change; rs_knn_profile's corated_triples stays the last Fit's, and the candidate bound of Predict
 * (the longest right row) is not lowered.  Memory as rs_knn_update: the edited arrays go to the same two blocks per
 * array.  To find a pair's place in the dataset order, a Fit that keeps the dataset-order values (non-integer ratings,
 * RS_KNN_ZSCORE) also keeps their right ids, 4 bytes per rating. */
int32_t rs_knn_remove(rs_knn *h, const int32_t *left, const int32_t *right, int64_t n, double global_mean);
int32_t rs_knn_remove_device(rs_knn *h, const int32_t *d_left, const int32_t *d_right, int64_t n, double global_mean);
int32_t rs_knn_change(rs_knn *h, const int32_t *left, const int32_t *right, const double *rating, int64_t n,
                      double global_mean);
int32_t rs_knn_change_device(rs_knn *h, const int32_t *d_left, const int32_t *d_right, const double *d_rating,
                             int64_t n, double global_mean);
/* ADDING RATINGS TO A CYCLIC ROW SHARD (after rs_knn_mirror).  rs_knn_update and rs_knn_update_device refuse every row
 * shard; this is their form for cyclic shards.  Every shard of the model is called with the same ratings, counts and
 * global_mean, and no data moves between them: each merges the ratings into its copies of both CSRs and of every row's
 * statistics, and recomputes the cells it stores — the full rows of the touched ids it owns, and the columns of the
 * touched ids other shards own in each of its rows.  Afterwards every shard holds, bit for bit, the rows that a cyclic
 * Fit of the union plus rs_knn_mirror gives it under the same block rule (blocks of 32 rows, block b on shard
 * b % shard_count); a new left id lands on the shard that rule names, so a shard that held no rows may gain some.
 * Inputs, return and memory as rs_knn_update_device.  Refused, leaving the shard exactly as it was:
 *   RS_ERR_INVALID     not a cyclic row shard (a handle with every row), a cyclic shard before rs_knn_mirror, and
 *                      every RS_ERR_INVALID case of rs_knn_update;
 *   RS_ERR_UNSUPPORTED a row_begin/row_end shard (its range is fixed at create and cannot take new ids), and every
 *                      RS_ERR_UNSUPPORTED case of rs_knn_update other than row shards;
 *   RS_ERR_DUPLICATE, RS_ERR_OOM as rs_knn_update.
 * The checks read only what every shard holds alike, so a refusal other than RS_ERR_OOM is the same on every shard.
 * After an update, rs_knn_mirror returns RS_ERR_INVALID until the next Fit: the shard's rows are complete. */
int32_t rs_knn_update_sharded_device(rs_knn *h, const int32_t *d_left, const int32_t *d_right, const double *d_rating,
                                     int64_t nnz, int32_t n_left, int32_t n_right, double global_mean);

/* Parameters["k"] / ["mink"] are read at Predict time by the reference (core/knn.go:80-81): change
 * them on a fitted handle without refitting.  The predict kernel supports k <= 256. */
int32_t rs_knn_set_k(rs_knn *h, int32_t k, int32_t min_k);

/* CYCLIC ROW SHARDS (RS_STORE_MATRIX, shard_count >= 2) — the exchange step of a Fit sharded over the
 * GPUs of one box; replaces the goroutine row split of core/knn.go:192-216.
 *   rs_knn_peer_export  : a CUDA IPC handle (64 bytes) + byte offset of this shard's matrix, to be
 *                         all-gathered by the host (torch.distributed / MPI / a pipe);
 *   rs_knn_peer_import  : attaches the matrices of all shard_count shards (handles: shard_count x 64
 *                         bytes, offsets: shard_count); mappings are cached for the life of the handle;
 *   rs_knn_peer_import_local : the same for shards that live in THIS process (one handle per GPU, or
 *                         several on one GPU in tests): peers[q] = handle of shard q;
 *   rs_knn_mirror       : fills the triangle this shard did not compute from the peers' matrices (P2P
 *                         loads over NVLink, transposed through shared memory).  The caller orders it
 *                         after every peer's Fit has finished (rs_knn_synchronize + a barrier) and
 *                         keeps the peers' matrices alive until it has finished.
 * Until rs_knn_mirror has run, Predict / sims_rows / topk on a cyclic shard fail with RS_ERR_INVALID, and after
 * rs_knn_update_sharded_device it returns RS_ERR_INVALID until the next Fit. */
/* Predict on a cyclic row shard for an all-reduce: the FULL test set goes to every shard; a pair whose left row
 * another shard owns yields +0.0 (all bits zero) instead of NaN, and a cold-start pair (left = -1) is answered by
 * shard (index % shard_count) only — so an integer SUM all-reduce of the 64-bit patterns over the shards assembles
 * the complete prediction vector, bit for bit, with no routing and no re-ordering on the host. */
int32_t rs_knn_predict_batch_sharded_device(rs_knn *h, const int32_t *d_left, const int32_t *d_right, int64_t n,
                                            double *d_out);
int32_t rs_knn_peer_export(rs_knn *h, unsigned char *handle64, int64_t *offset);
int32_t rs_knn_peer_import(rs_knn *h, int32_t n_peers, const unsigned char *handles, const int64_t *offsets);
int32_t rs_knn_peer_import_local(rs_knn *h, int32_t n_peers, rs_knn *const *peers);
int32_t rs_knn_mirror(rs_knn *h);

int32_t rs_knn_profile_get(rs_knn *h, rs_knn_profile *out);
int32_t rs_knn_profile_reset(rs_knn *h);
/* Destroyed handles park their device memory in a process-wide cache (estimator copies are
 * created and destroyed per fold, core/eval.go:29-35); this returns it to the driver. */
int32_t rs_knn_trim_cache(void);
/* Page-locked host memory for the host-pointer entry points (rs_knn_fit, rs_knn_predict_batch, ...): copies from
 * and to such buffers run at full PCIe speed and asynchronously, pageable buffers are staged by the driver
 * (a 4 M-pair test set: ~1.3 ms instead of ~6 ms for ids in + predictions out).  Blocks are cached per process
 * (cudaHostAlloc costs milliseconds); rs_knn_trim_cache returns them to the driver.  Optional: every entry
 * point accepts ordinary host memory (the reference's slices, core/data.go:18-22). */
int32_t rs_knn_host_alloc(size_t bytes, void **out);
int32_t rs_knn_host_free(void *p);
/* Block until everything queued on the handle's stream has finished. */
int32_t rs_knn_synchronize(rs_knn *h);

#ifdef __cplusplus
}
#endif
#endif /* RS_KNN_H */
