// common.cuh — shared declarations of librs_knn_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>

#include "rs_knn.h"

void rs_set_error(const char *fmt, ...);

#define RS_CUDA(expr)                                                                       \
    do {                                                                                    \
        cudaError_t e_ = (expr);                                                            \
        if (e_ != cudaSuccess) {                                                            \
            rs_set_error("%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return (e_ == cudaErrorMemoryAllocation) ? RS_ERR_OOM : RS_ERR_CUDA;            \
        }                                                                                   \
    } while (0)

#define RS_TRY(expr)              \
    do {                          \
        int32_t rc_ = (expr);     \
        if (rc_ != RS_OK) return rc_; \
    } while (0)

// Rating classes (how a rating is represented as one byte; 0 = missing).
//   RS_CLASS_INT8 : every rating is an integer in [-11,11]; code = rating + 12.
//   RS_CLASS_TABLE: any other float64 ratings; no byte code (stream path only, reads the values).
enum { RS_CLASS_INT8 = 0, RS_CLASS_TABLE = 1 };
constexpr int RS_INT8_BIAS = 12;

// Column-chunk width of the streaming similarity kernel (threads * bytes per thread).
// Streaming similarity kernel: warps per CTA, each an independent (row, column-chunk) work item.
// The chunk width (rs_knn::stream_jc, 128 or 256 columns = 3 x JC doubles of accumulators per
// warp) is chosen per Fit: 128 gives small problems enough work items to balance the SMs
// (MovieLens-1M shape: 1.6 ms vs 2.2 ms), 256 halves the per-chunk walk of the row on large sparse
// ones (MovieLens-20M item shape: 85 ms vs 128 ms); profiles/r01_stream_notes.md.
constexpr int RS_STREAM_WARPS = 8;

// Tensor-core similarity kernel tile: 128 left rows (MMA M) x 64 left rows (MMA N),
// K blocked by 128 bytes (one SWIZZLE_128B atom) per pipeline stage.
constexpr int RS_TC_BM = 128;
constexpr int RS_TC_BN = 64;
constexpr int RS_TC_BK = 128;
constexpr int RS_TC_KBLK = 256;   // bytes of K per block of the K-blocked plane layout [plane][K/256][row][256]

// Cyclic row shards (RS_STORE_MATRIX with shard_count >= 2): rows are dealt to the shards in blocks of
// RS_CYC_B (block b belongs to shard b % count), so every shard gets the same mix of long and short
// rows; a shard stores its rows densely in dealing order.
constexpr int RS_CYC_B = 32;
constexpr int RS_MAX_PEERS = 16;
__host__ __device__ inline int64_t rs_cyc_local(int64_t i, int count) {
    return (i / ((int64_t)RS_CYC_B * count)) * RS_CYC_B + i % RS_CYC_B;
}
__host__ __device__ inline bool rs_cyc_owns(int64_t i, int count, int index) {
    return (i / RS_CYC_B) % count == index;
}
// Global id of local row `loc` of shard `index`: the inverse of rs_cyc_local on the rows the shard owns.
__host__ __device__ inline int64_t rs_cyc_global(int64_t loc, int count, int index) {
    return ((loc / RS_CYC_B) * count + index) * RS_CYC_B + loc % RS_CYC_B;
}
inline int64_t rs_cyc_rows(int64_t n, int count, int index) {
    const int64_t nblk = (n + RS_CYC_B - 1) / RS_CYC_B;
    int64_t rows = 0;
    for (int64_t b = index; b < nblk; b += count) rows += (b + 1) * RS_CYC_B <= n ? RS_CYC_B : n - b * RS_CYC_B;
    return rows;
}

// The model arrays rs_knn_update, rs_knn_remove and rs_knn_change rewrite (update.cu); rs_knn::upd holds their blocks.
enum rs_upd_array {
    RS_UPD_L_PTR, RS_UPD_L_COL, RS_UPD_L_VAL, RS_UPD_L_CODE, RS_UPD_LD_VAL, RS_UPD_R_PTR, RS_UPD_R_COL, RS_UPD_R_VAL,
    RS_UPD_MEANS, RS_UPD_STDDEVS, RS_UPD_PMEANS, RS_UPD_ROW_CNT, RS_UPD_ROW_SUM, RS_UPD_LD_COL, RS_UPD_ARRAYS
};

struct rs_knn {
    std::recursive_mutex mu;             // serialises the ABI calls on this handle (api.cu Guard)
    rs_knn_params p{};
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaStream_t aux_stream = nullptr;   // read-backs of Fit statistics that must not wait for the similarity kernel
    cudaEvent_t ev_in = nullptr;         // the host inputs of rs_knn_fit have been consumed
    cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_c = nullptr, ev_d = nullptr, ev_e = nullptr;
    rs_knn_profile prof{};
    // pending event pairs whose elapsed time has not been folded into prof yet
    bool sim_pending = false, pred_pending = false, prep_pending = false;

    bool fitted = false;
    int32_t n_left = 0, n_right = 0;
    int64_t nnz = 0;
    int64_t row_begin = 0, row_end = 0;  // resolved shard
    int64_t col_begin = 0;               // symmetric slabs: similarity tiles left of this column are not needed
    bool force_sym = false;              // symmetric slabs: compute only j > i although the rows are a slab
    int64_t topk_rows = 0;               // rows covered by topk_idx / topk_sim
    // cyclic row shards: cyc_R >= 2 shards, this handle is shard cyc_r and stores rows_local rows
    int32_t cyc_R = 0, cyc_r = 0;
    int64_t rows_local = 0;              // rows of `sims` (== row_end - row_begin unless cyclic)
    int64_t n_work_rows = 0;             // entries of row_order the stream kernel walks
    const double *peer_sims[RS_MAX_PEERS] = {nullptr};   // the shards' matrices (peer memory over NVLink), [cyc_r] = own
    bool peers_ready = false;
    double global_mean = 0.0, global_bias = 0.0;
    int rating_class = RS_CLASS_INT8;

    // Grow-only device arena: Fit bump-allocates from it and the next Fit reuses the same
    // chunks, so a refit of the same shape performs no cudaMalloc / cudaFree at all.
    struct Chunk { char *p; size_t bytes; };
    std::vector<Chunk> chunks;
    size_t cur_chunk = 0, cur_off = 0;
    // cached tensor-path tile list
    void *tile_buf = nullptr;
    size_t tile_buf_bytes = 0;
    int64_t tile_key[5] = {-1, -1, -1, -1, -1};
    int32_t tile_count = 0;
    // fused top-k: band tile lists (all waves, concatenated) and the per-row selection state
    void *band_buf = nullptr;
    size_t band_buf_bytes = 0;
    int64_t band_key[4] = {-1, -1, -1, -1};
    std::vector<int64_t> band_off;
    unsigned long long *thr_key = nullptr;   // [n_left] k-th best key of the row's running list (0 = not full)
    int32_t *thr_id = nullptr;
    int32_t *cand_cnt = nullptr;             // [n_left] candidates appended since the last merge
    int32_t *cand_id = nullptr;              // [n_left][cand_cap]
    double *cand_sim = nullptr;
    int32_t cand_cap = 0;
    int32_t *row_flag = nullptr;             // [n_left] the row's buffer overflowed in the current band

    // CSR of the left rows, entries ascending by right id (core/data.go:236-243)
    int64_t *l_ptr = nullptr;
    int32_t *l_col = nullptr;
    double *l_val = nullptr;
    uint8_t *l_code = nullptr;
    double *ld_val = nullptr;  // left rows in DATASET order (means / std accumulate in it)
    int32_t *ld_col = nullptr; // their right ids, where Fit keeps ld_val (an edit finds its entry in that order by id)
    // CSR of the right rows, entries ascending by left id (Predict candidates)
    int64_t *r_ptr = nullptr;
    int32_t *r_col = nullptr;
    double *r_val = nullptr;

    double *means = nullptr;      // KNN.Means    (dataset order sum / count)
    double *stddevs = nullptr;    // KNN.StdDevs
    double *pmeans = nullptr;     // Pearson's own row means (sorted-order sum, core/sim.go:49-62)
    double *left_bias = nullptr;  // KNN.Bias
    int32_t *row_cnt = nullptr;   // ratings per left row and their integer sum (tensor path, Pearson)
    int32_t *row_sum = nullptr;
    // integer class: the largest |rating| and the two longest left rows, which bound every int32 accumulator of the
    // tensor path (tensor_eligible, api.cu)
    int32_t int_abs_max = 0;
    int64_t row_len1 = 0, row_len2 = 0;
    int32_t max_right_len = 0;    // longest right row = most candidates one prediction can have
    double triples = 0.0;         // co-rated triples of the full matrix: sum over right rows of cnt*(cnt-1)/2
    double *right_bias = nullptr;
    // Slope One: the right rows (users) in DATASET order — left ids only — and their means
    int32_t *rd_col = nullptr;
    double *right_means = nullptr;

    // stream path: b-side term of every rating in right-CSR order (value, value - row mean, ...),
    // chunk pointers cp[right][Q+1] into each right row, and l2r: left-CSR entry -> right-CSR (or walk-CSR) index
    double *r_dev = nullptr;
    int32_t *cp = nullptr;
    int32_t n_chunks = 0;
    int32_t stream_jc = 256;
    bool stream_lower = false;     // full-matrix stream Fit computes j < i (else j > i); chosen per Fit from the lookup counts
    double inc_upper = 0.0, inc_lower = 0.0;   // (entry, chunk) lookups of the two triangles (in label space with popular columns)
    int64_t *l2r = nullptr;
    int32_t *perm_lr = nullptr, *perm_rl = nullptr, *perm_tmp = nullptr;  // CSR position -> input row (arena, valid until the next Fit)
    int32_t *row_order = nullptr;  // left rows sorted by descending length
    // popular columns (sim_stream.cu: the dense items of sim_stream_kernel): the n_pop longest rows, longest first.
    // Their ratings are taken out of the right CSR the column walk reads (walk CSR: w_ptr / w_col / w_dev, `cp` and
    // `l2r` refer to it) and kept as a dense table pop_dense[n_right][pop_ld] instead (one byte per cell when every
    // rating is a small integer, else the b-side double; 0 / NaN = no rating).
    // Every row has a RANK, its position in the stable longest-first order of all rows: ranks below n_pop are the
    // popular list, and the other rows are the walk's columns under the LABEL rank - n_pop (the walk CSR holds
    // labels, ascending within each right row), so the long rows have the small labels.
    int32_t n_pop = 0, pop_ld = 0;
    bool pop_u8 = false;
    int32_t *rank = nullptr;       // [n_left] position in the longest-first order
    int32_t *lab_row = nullptr;    // [n_left - n_pop] the row of each label
    int32_t *pop_items = nullptr;  // [pop_ld] row id (-1 beyond n_pop)
    void *pop_dense = nullptr;
    int64_t *w_ptr = nullptr;
    int32_t *w_col = nullptr;      // labels
    double *w_dev = nullptr;
    int32_t *row_all = nullptr;    // every row of the shard, longest first (the dense pass visits them all)
    int64_t n_all_rows = 0;
    // int8 planes X^2, M, X of the left matrix, [3][k_pad / 256][n_pad][256] (tensor path)
    int8_t *planes = nullptr;
    int64_t tc_npad = 0, tc_kpad = 0;

    // outputs
    double *sims = nullptr;  // (row_end-row_begin) x ld_s, NaN = unset
    int64_t ld_s = 0;
    int32_t *topk_idx = nullptr;  // RS_STORE_TOPK: rows x topk
    double *topk_sim = nullptr;

    int32_t *d_flags = nullptr;  // small device scratch for validation flags
    // rs_knn_update (and the edits): the model arrays an update rewrote live in blocks of their own (the arena only grows until the
    // next Fit), two per array: the model's, p[cur], and the spare the next update merges into.  cur = -1 while
    // the model's array is the Fit's, in the arena.
    struct UpdArray { void *p[2] = {nullptr, nullptr}; size_t bytes[2] = {0, 0}; int cur = -1; };
    UpdArray upd[RS_UPD_ARRAYS];
    void *upd_sims = nullptr;    // the matrix, once an update has grown it out of the arena
    size_t upd_sims_bytes = 0;
    bool updated = false;        // an update has run since the last Fit: rs_prep_planes builds into upd_planes
    void *upd_planes = nullptr;
    size_t upd_planes_bytes = 0;
    void *ovf = nullptr;         // predict: overflow list (count + indices)
    size_t ovf_bytes = 0;
    std::vector<void *> scratch;         // device staging of the host-pointer entry points
    std::vector<size_t> scratch_bytes;
};

// ---- devmem.cu: process-wide cache of device allocations ----
// Estimator copies are created and destroyed per cross-validation fold (core/eval.go:29-35);
// freed device blocks are parked here and handed to the next handle on the same device, so a
// create/Fit/Predict/destroy cycle performs no cudaMalloc/cudaFree after the first one.
int32_t rs_cached_malloc(int device, void **out, size_t bytes, size_t *got);
void rs_cached_free(int device, void *p, size_t bytes);
void rs_cache_trim(void);

// ---- api.cu: grow-only per-handle device scratch (slot-indexed) ----
// A slot holds one buffer, and asking it for more bytes than it has frees that buffer and allocates a larger one.  So
// two buffers that are live at the same time need two slots.  ABI calls on one handle are serialised and run on its
// stream, so different calls may share a slot; the slots that are shared say so.
enum rs_scratch_slot {
    // api.cu: host arguments of rs_knn_predict_batch and rs_knn_predict_neighbors (one call at a time)
    RS_SCR_PRED_LEFT,
    RS_SCR_PRED_RIGHT,
    RS_SCR_PRED_OUT,
    RS_SCR_HOST_IDS,          // rs_knn_predict_neighbors' list, rs_knn_topk's lists
    RS_SCR_HOST_SIMS,
    RS_SCR_NB_COUNT,
    RS_SCR_COSUMS,
    RS_SCR_FIT_LEFT,          // rs_knn_fit's and rs_knn_update's inputs
    RS_SCR_FIT_RIGHT,
    RS_SCR_FIT_RATING,
    RS_SCR_FIT_LEFT_BIAS,
    RS_SCR_FIT_RIGHT_BIAS,
    // predict.cu: the pairs grouped by left row
    RS_SCR_PRED_KEYS_IN,
    RS_SCR_PRED_KEYS,
    RS_SCR_PRED_IOTA,
    RS_SCR_PRED_PERM,
    RS_SCR_PRED_SORT_TMP,
    RS_SCR_PRED_OWN_COUNT,
    // the work counter and the per-warp key spill of a select.cuh kernel: Predict, Slope One's Predict and
    // recommend_kernel share them.  A launch uses them alone; the next one zeroes the counter and sizes the spill after
    // it on the same stream (a larger spill is allocated only after that stream has drained).
    RS_SCR_WORK,
    RS_SCR_KEY_SPILL,
    // api.cu: host arguments of the recommendation entry points (by id or as lists; one call at a time)
    RS_SCR_REC_QUERIES,
    RS_SCR_REC_PTR,
    RS_SCR_REC_IDS,
    RS_SCR_REC_VALS,
    RS_SCR_REC_OUT,           // the score rows, or the list ids
    RS_SCR_REC_SCORES,        // the list scores
    // recommend.cu
    RS_SCR_REC_SLAB,          // a batch's score rows
    RS_SCR_REC_STAGE_IDS,     // a shard's lists of a batch, before they are placed
    RS_SCR_REC_STAGE_SCORES,
    RS_SCR_OWN_FLAG,          // the left queries a shard answers
    RS_SCR_OWN_QUERIES,
    RS_SCR_OWN_POS,
    RS_SCR_OWN_COUNT,
    RS_SCR_OWN_TMP,
    // given.cu and the given lists' statistics (recommend.cu)
    RS_SCR_GIVEN_COUNTER,
    RS_SCR_GIVEN_HDR,
    RS_SCR_GIVEN_PTR,
    RS_SCR_GIVEN_IDS,
    RS_SCR_GIVEN_VALS,
    RS_SCR_GIVEN_SORT_TMP,
    RS_SCR_GIVEN_MEANS,
    RS_SCR_GIVEN_STDDEVS,
    RS_SCR_GIVEN_PMEANS,
    RS_SCR_GIVEN_SIMS,        // a batch's S* rows
    // update.cu
    RS_SCR_UPD_WORK,          // the added ratings sorted both ways, their row pointers, the touched rows
    RS_SCR_UPD_SORT_TMP,
    RS_SCR_UPD_SLAB,          // a batch's recomputed rows
};
extern "C" int32_t rs_scratch_get(rs_knn *h, int slot, size_t bytes, void **out);

// The targets of a query of `side`: every id of the other side.
inline int64_t rs_n_targets(const rs_knn *h, int32_t side) { return side == RS_SIDE_RIGHT ? h->n_left : h->n_right; }

// ---- prep.cu ----
int32_t rs_prep_build(rs_knn *h, const int32_t *d_left, const int32_t *d_right, const double *d_rating,
                      const double *d_left_bias, const double *d_right_bias);
int32_t rs_dev_alloc(rs_knn *h, void **out, size_t bytes);
template <typename T>
inline int32_t rs_alloc(rs_knn *h, T **out, size_t count) {
    return rs_dev_alloc(h, reinterpret_cast<void **>(out), count * sizeof(T));
}
int32_t rs_prep_rt(rs_knn *h);
int32_t rs_prep_planes(rs_knn *h);
int32_t rs_row_stats_launch(rs_knn *h, const int64_t *ptr, const double *ld_val, const double *l_val, int64_t n,
                            int want_std, double *means, double *stddevs, double *pmeans);
int32_t rs_prep_stats(rs_knn *h);
// Words of h->d_flags (16 x int32) where rs_prep_stats leaves the tensor path's limits for integer ratings: the largest
// |rating|, and at the 8-byte aligned pair RS_FL_LEN_TOP2 the longest (high word) and second-longest (low) left row.
constexpr int RS_FL_ABS_MAX = 1, RS_FL_LEN_TOP2 = 12;
inline void rs_tensor_limits_read(rs_knn *h, const int32_t fl[16]) {
    unsigned long long t;
    std::memcpy(&t, fl + RS_FL_LEN_TOP2, 8);
    h->int_abs_max = fl[RS_FL_ABS_MAX];
    h->row_len1 = (int64_t)(t >> 32);
    h->row_len2 = (int64_t)(t & 0xFFFFFFFFull);
}
// Kernels of the CSR build that rs_knn_update runs on the added ratings as Fit runs them on all ratings.
enum rs_prep_flag { FLAG_BAD_ID = 1, FLAG_NOT_INT8 = 2, FLAG_DUP = 4, FLAG_NAN = 8, FLAG_MISSING = 16 };
__global__ void ptr_from_sorted_kernel(const int32_t *__restrict__ keys, int64_t nnz, int32_t n_rows,
                                       int64_t *__restrict__ ptr);
__global__ void gather_keys_kernel(const int32_t *__restrict__ src, const int32_t *__restrict__ perm, int64_t n,
                                   int32_t *__restrict__ out);
__global__ void dup_check_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col, int64_t nnz,
                                 int32_t *__restrict__ flags);

// ---- sim_stream.cu ----
int32_t rs_sim_stream_launch(rs_knn *h);
int32_t rs_symmetrize_launch(rs_knn *h);
int32_t rs_mirror_launch(rs_knn *h);

// ---- sim_tensor.cu ----
int32_t rs_sim_tensor_launch(rs_knn *h, int32_t *d_cosums, int64_t cos_row0, int64_t cos_nrows);
int32_t rs_tensor_band_count(const rs_knn *h);
int32_t rs_sim_tensor_band_launch(rs_knn *h, int32_t wave);
bool rs_tensor_topk_fused(const rs_knn *h);

// ---- predict.cu ----
int32_t rs_predict_launch(rs_knn *h, const int32_t *d_left, const int32_t *d_right, int64_t n, double *d_out,
                          int32_t *d_nb_ids, double *d_nb_sims, int32_t *d_nb_count, int32_t nb_cap, int32_t foreign_zero = 0);
int32_t rs_nb_cells_launch(rs_knn *h, const int32_t *d_left, const int32_t *d_nb_ids, const int32_t *d_nb_count,
                           double *d_nb_sims);
int32_t rs_slope_predict_launch(rs_knn *h, const int32_t *d_left, const int32_t *d_right, int64_t n, double *d_out);

// ---- topk.cu ----
// Neighbours per row of an RS_STORE_TOPK handle.
inline int32_t rs_list_k(const rs_knn *h) { return h->p.topk > 0 ? h->p.topk : h->p.k; }
int32_t rs_topk_check_k(int32_t k);
int32_t rs_topk_rows_launch(rs_knn *h, const double *src, int64_t ld, int32_t n, int64_t rows, int32_t k, int32_t *d_idx,
                            double *d_sim);
int32_t rs_fit_lists(rs_knn *h, int path);

// ---- recommend.cu ----
// One call of a recommendation entry point (include/rs_knn.h), checked by api.cu; every pointer is device memory.
struct rs_rec_call {
    int32_t side;                 // enum rs_side
    bool sharded;                 // a row shard's part (rs_knn_*_sharded_device)
    bool given;                   // the queries are rating lists (rs_knn_*_given), else inner ids
    bool lists;                   // the top-n_top lists, else the score rows
    const int32_t *queries;       // by id: [n]
    const int64_t *ptr;           // given: list b is ids / vals [ptr[b], ptr[b+1])
    const int32_t *ids;
    const double *vals;
    int64_t n;
    double *rows;                 // score rows [n][n_targets]
    int32_t n_top;                // lists [n][n_top]
    int32_t *top_ids;
    double *top_scores;
};
int32_t rs_recommend_run(rs_knn *h, const rs_rec_call &c);
// Rows per batch of a slab of `width` doubles per row: ~256 MiB (RS_KNN_REC_BATCH forces a size).
int64_t slab_batch(int64_t width, int64_t n);

// ---- given.cu ----
// The lists of rs_knn_*_given, validated and sorted: list b is entries ptr[b] .. ptr[b+1) of ids / vals (ascending id)
// and of vals_in (the caller's order).
struct rs_given_lists {
    const int64_t *ptr;      // [n + 1], ptr[0] = 0
    const int32_t *ids;
    const double *vals;
    const double *vals_in;
    int64_t nnz;
    int64_t max_len;         // the longest list
};
int32_t rs_given_prepare(rs_knn *h, int32_t n_targets, const int64_t *d_ptr, const int32_t *d_ids,
                         const double *d_vals, int64_t n, rs_given_lists *out);
// The similarity rows S*[b][v] = Sim(list b, left row v) of the lists ptr[0 .. nq) (ids: right ids), into out[nq][ld].
// With `rows`, list b is list rows[b] of ptr and its Pearson mean qpmeans[rows[b]].  With `own` (a cyclic row shard),
// only the rows the shard owns, at their local rows: out[nq][ld], ld >= rows_local.
int32_t rs_given_sims_launch(rs_knn *h, const int64_t *ptr, const int32_t *ids, const double *vals,
                             const double *qpmeans, int64_t nq, double *out, int64_t ld,
                             const int32_t *rows = nullptr, bool own = false);

// ---- update.cu ----
int32_t rs_update_run(rs_knn *h, const int32_t *d_left, const int32_t *d_right, const double *d_rating, int64_t nnz,
                      int32_t n_left, int32_t n_right, double global_mean);
// rs_knn_remove (remove) / rs_knn_change: the pairs d_left[e], d_right[e] the model holds, dropped or given d_rating[e]
int32_t rs_edit_run(rs_knn *h, bool remove, const int32_t *d_left, const int32_t *d_right, const double *d_rating,
                    int64_t nd, double global_mean);
void rs_update_release(rs_knn *h);

// First position in [lo, hi) of an ascending id array whose id is >= v: the searches of given.cu and update.cu.
__device__ __forceinline__ int64_t lower_bound_id(const int32_t *__restrict__ col, int64_t lo, int64_t hi, int32_t v) {
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (col[mid] < v) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// order-preserving map double -> uint64 (larger similarity = larger key); -0.0 folded to +0.0
__host__ __device__ inline uint64_t rs_sim_key(double s) {
    s = s + 0.0;  // -0.0 -> +0.0, every other value unchanged
#ifdef __CUDA_ARCH__
    uint64_t b = (uint64_t)__double_as_longlong(s);
#else
    uint64_t b;
    __builtin_memcpy(&b, &s, 8);
#endif
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__host__ __device__ inline double rs_key_sim(uint64_t k) {
    uint64_t b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
#ifdef __CUDA_ARCH__
    return __longlong_as_double((long long)b);
#else
    double s;
    __builtin_memcpy(&s, &b, 8);
    return s;
#endif
}
