// update.cu — rs_knn_update: ratings added to a fitted model without a refit.
//
// The updated model is the Fit of the union (the fitted ratings in their dataset order, then the added ones in call
// order), bit for bit (DESIGN.md §5.3d).  A left row is TOUCHED when an added rating names it, and every new left id
// is touched.
//   - The CSRs are merged: each left row holds its old entries and its new ones in ascending right id, and its
//     dataset-order values (ld_val) are the old ones followed by the new ones; each right row likewise in ascending
//     left id.  Old entries move by the number of new entries before them in their row, and new ones by the number
//     of old ones (a binary search in the short side): O(nnz) copies and no sort of the model.
//   - The statistics of every row are recomputed with Fit's kernels (rs_prep_stats, O(nnz)).
//   - The similarity rows of the touched ids are recomputed by given_sims_kernel on their merged left rows (the exact
//     sparse Fit's terms, order and IEEE operations) and written into their rows and columns, diagonal NaN.  A cell
//     between two untouched rows sums the same terms in the same order as before and their statistics do not change:
//     it is kept.
// Everything up to the one read-back of the checks goes to scratch; the model's merged arrays go to spare blocks
// (rs_knn::upd), and the model is written only when every check has passed and every block is allocated, so a
// refused update, or one that runs out of memory, leaves the model as it was.
#include <cub/cub.cuh>

#include <cstring>

#include "common.cuh"

namespace {

constexpr int T = 256;
inline unsigned blocks_for(int64_t n) { return (unsigned)((n + T - 1) / T); }

int bits_for(int32_t n) {
    int b = 1;
    while ((1ll << b) < (long long)n) b++;
    return b;
}

// The checks of Fit on the added ratings (ids in range, no NaN, the rating class), and the ids the sorts use: an id
// out of range becomes 0, so that every kernel before the read-back stays in bounds.
__global__ void upd_validate_kernel(const int32_t *__restrict__ left, const int32_t *__restrict__ right,
                                    const double *__restrict__ rating, int64_t nd, int32_t n_left, int32_t n_right,
                                    int32_t *__restrict__ idx, int32_t *__restrict__ ls, int32_t *__restrict__ rs,
                                    int32_t *__restrict__ flags) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nd) return;
    idx[e] = (int32_t)e;
    const int32_t l = left[e], r = right[e];
    const bool ok = l >= 0 && l < n_left && r >= 0 && r < n_right;
    ls[e] = ok ? l : 0;
    rs[e] = ok ? r : 0;
    const double v = rating[e];
    int f = ok ? 0 : FLAG_BAD_ID;
    if (v != v) f |= FLAG_NAN;
    if (!(v == rint(v) && fabs(v) <= 11.0)) f |= FLAG_NOT_INT8;
    if (f) atomicOr(flags, f);
}

// An added (left, right) pair the fitted left CSR holds already.  row / col: the added ratings in (left, right) order.
__global__ void upd_dup_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col, int64_t nd,
                               const int64_t *__restrict__ l_ptr, const int32_t *__restrict__ l_col, int32_t nl0,
                               int32_t *__restrict__ flags) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nd) return;
    const int32_t i = row[e], c = col[e];
    if (i >= nl0) return;
    const int64_t b = l_ptr[i], end = l_ptr[i + 1];
    const int64_t p = lower_bound_id(l_col, b, end, c);
    if (p < end && l_col[p] == c) atomicOr(flags, FLAG_DUP);
}

// The touched left rows, each keyed by its merged length + 1 (0: untouched) for a longest-first sort; flags[1] counts
// them.  d_ptr: the added ratings' row pointers.
__global__ void upd_touched_kernel(const int64_t *__restrict__ l_ptr, int32_t nl0, const int64_t *__restrict__ d_ptr,
                                   int32_t nl, uint32_t *__restrict__ key, int32_t *__restrict__ ids,
                                   int32_t *__restrict__ flags) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nl) return;
    const int64_t dl = d_ptr[i + 1] - d_ptr[i];
    const bool touched = dl > 0 || i >= nl0;
    key[i] = touched ? (uint32_t)((i < nl0 ? l_ptr[i + 1] - l_ptr[i] : 0) + dl + 1) : 0u;
    ids[i] = i;
    if (touched) atomicAdd(flags + 1, 1);
}

// The longest merged right row (Predict's candidate bound) into flags[2].
__global__ void upd_right_len_kernel(const int64_t *__restrict__ r_ptr, int32_t nr0, const int64_t *__restrict__ d_ptr,
                                     int32_t nr, int32_t *__restrict__ flags) {
    const int32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nr) return;
    const int64_t len = (c < nr0 ? r_ptr[c + 1] - r_ptr[c] : 0) + d_ptr[c + 1] - d_ptr[c];
    atomicMax(flags + 2, (int32_t)len);
}

// merged row pointers: old_ptr (n0 rows, ptr[n0] = nnz0) + the added ratings' d_ptr (n rows)
__global__ void upd_ptr_kernel(const int64_t *__restrict__ old_ptr, int32_t n0, const int64_t *__restrict__ d_ptr,
                               int32_t n, int64_t *__restrict__ out) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    out[i] = old_ptr[i < n0 ? i : n0] + d_ptr[i];
}

// The old entries of a CSR into the merged one, one warp per old row: entry x of row i moves to its place in the
// merged row, after the added entries of row i with a smaller id (d_col: the added entries' ids, row by row
// ascending; null: no added entry comes before an old one, the dataset order of ld_val).  code: the byte codes.
__global__ void upd_merge_old_kernel(const int64_t *__restrict__ old_ptr, const int32_t *__restrict__ old_col,
                                     const double *__restrict__ old_val, int32_t n0, const int64_t *__restrict__ d_ptr,
                                     const int32_t *__restrict__ d_col, const int64_t *__restrict__ new_ptr,
                                     int32_t *__restrict__ col, double *__restrict__ val, uint8_t *__restrict__ code) {
    const int32_t i = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n0) return;
    const int64_t b = old_ptr[i], e = old_ptr[i + 1], db = d_ptr[i], de = d_ptr[i + 1];
    const int64_t base = new_ptr[i] - b;
    for (int64_t x = b + lane; x < e; x += 32) {
        const double v = old_val[x];
        int64_t pos = base + x;
        if (d_col) {
            const int32_t c = old_col[x];
            pos += lower_bound_id(d_col, db, de, c) - db;
            col[pos] = c;
        }
        val[pos] = v;
        if (code) code[pos] = (uint8_t)((int)v + RS_INT8_BIAS);      // code_int8_kernel's byte
    }
}

// The added entries into the merged CSR, one thread each (in the order of the sort that grouped them by row: key = the
// row, perm = the added rating's position): after the old entries of the row with a smaller id (old_col null: after
// all of them).
__global__ void upd_merge_new_kernel(const int32_t *__restrict__ key, const int32_t *__restrict__ d_col,
                                     const int32_t *__restrict__ perm, const double *__restrict__ rating, int64_t nd,
                                     const int64_t *__restrict__ old_ptr, const int32_t *__restrict__ old_col,
                                     int32_t n0, const int64_t *__restrict__ d_ptr, const int64_t *__restrict__ new_ptr,
                                     int32_t *__restrict__ col, double *__restrict__ val, uint8_t *__restrict__ code) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nd) return;
    const int32_t i = key[e];
    const int64_t b = i < n0 ? old_ptr[i] : 0, end = i < n0 ? old_ptr[i + 1] : 0;
    int64_t pos = new_ptr[i] + (e - d_ptr[i]);
    const double v = rating[perm[e]];
    if (old_col) {
        const int32_t c = d_col[e];
        pos += lower_bound_id(old_col, b, end, c) - b;
        col[pos] = c;
    } else {
        pos += end - b;
    }
    val[pos] = v;
    if (code) code[pos] = (uint8_t)((int)v + RS_INT8_BIAS);
}

// Row i = rows[b] of the matrix and its column from the recomputed row slab[b]: S[i][v] = S[v][i] = slab[b][v], the
// diagonal NaN as Fit leaves it.  Two touched rows write the same bits into their common cells: Sim(i, j) and
// Sim(j, i) sum the same terms in the same order.
__global__ void upd_scatter_kernel(const double *__restrict__ slab, int64_t ld, const int32_t *__restrict__ rows,
                                   int64_t nb, int32_t n, double *__restrict__ sims) {
    const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= nb * n) return;
    const int64_t b = x / n;
    const int32_t v = (int32_t)(x - b * n);
    const int32_t i = rows[b];
    const double s = v == i ? __longlong_as_double(0x7ff8000000000001ll) : slab[b * ld + v];
    sims[(int64_t)i * ld + v] = s;
    sims[(int64_t)v * ld + i] = s;
}

// Carves the update's scratch arrays out of one block.
struct Carve {
    char *p;
    size_t off = 0;
    template <typename X>
    X *take(int64_t n) {
        X *r = reinterpret_cast<X *>(p ? p + off : nullptr);
        off += ((size_t)(n > 0 ? n : 1) * sizeof(X) + 255) & ~(size_t)255;
        return r;
    }
};

struct Work {
    int32_t *flags;           // [0] FLAG_*, [1] touched rows, [2] longest merged right row
    int32_t *idx, *ls, *rs, *keys_a, *keys_b, *keys_l, *keys_r;
    int32_t *perm_l, *perm_r, *perm_lr, *perm_rl, *col_lr, *col_rl;
    int64_t *ptr_l, *ptr_r;
    uint32_t *len, *len_sorted;
    int32_t *ids, *rows;
};

Work carve(void *base, int64_t nd, int32_t nl, int32_t nr, size_t *bytes) {
    Carve c{static_cast<char *>(base)};
    Work w;
    w.flags = c.take<int32_t>(4);
    int32_t **nd_arrays[] = {&w.idx, &w.ls, &w.rs, &w.keys_a, &w.keys_b, &w.keys_l, &w.keys_r, &w.perm_l,
                             &w.perm_r, &w.perm_lr, &w.perm_rl, &w.col_lr, &w.col_rl};
    for (int32_t **a : nd_arrays) *a = c.take<int32_t>(nd);
    w.ptr_l = c.take<int64_t>((int64_t)nl + 1);
    w.ptr_r = c.take<int64_t>((int64_t)nr + 1);
    w.len = c.take<uint32_t>(nl);
    w.len_sorted = c.take<uint32_t>(nl);
    w.ids = c.take<int32_t>(nl);
    w.rows = c.take<int32_t>(nl);
    *bytes = c.off;
    return w;
}

// The spare block of model array a, at least `bytes`.  A spare too small goes back to the cache and a block a quarter
// larger replaces it: the stream has drained since the spare's last use (the update's read-back), and a sequence of
// updates reuses the same two blocks per array.
int32_t spare(rs_knn *h, int a, size_t bytes, void **out) {
    rs_knn::UpdArray &u = h->upd[a];
    const int s = u.cur == 0 ? 1 : 0;
    if (u.bytes[s] < bytes) {
        rs_cached_free(h->device, u.p[s], u.bytes[s]);
        u.p[s] = nullptr;
        u.bytes[s] = 0;
        size_t got = 0;
        RS_TRY(rs_cached_malloc(h->device, &u.p[s], bytes + bytes / 4 + 256, &got));
        u.bytes[s] = got;
    }
    *out = u.p[s];
    return RS_OK;
}

template <typename X>
int32_t spare_of(rs_knn *h, int a, int64_t n, X **out) {
    void *p;
    RS_TRY(spare(h, a, (size_t)n * sizeof(X), &p));
    *out = static_cast<X *>(p);
    return RS_OK;
}

}  // namespace

#define RS_UPD_SORT(CALL)                                                                                  \
    do {                                                                                                   \
        void *t_ = nullptr;                                                                                \
        size_t need_ = 0;                                                                                  \
        RS_CUDA(CALL(nullptr, need_));                                                                     \
        RS_TRY(rs_scratch_get(h, RS_SCR_UPD_SORT_TMP, need_ + 256, &t_));                                  \
        RS_CUDA(CALL(t_, need_));                                                                          \
    } while (0)

int32_t rs_update_run(rs_knn *h, const int32_t *d_left, const int32_t *d_right, const double *d_rating, int64_t nd,
                      int32_t nl, int32_t nr, double global_mean) {
    cudaStream_t st = h->stream;
    const int32_t nl0 = h->n_left, nr0 = h->n_right;
    const int64_t nnz0 = h->nnz, nnz = nnz0 + nd;
    const bool int8 = h->rating_class == RS_CLASS_INT8;
    // Fit keeps the dataset-order values only where a statistic is summed in that order (prep.cu)
    const bool dataset_order = !int8 || h->p.knn_type == RS_KNN_ZSCORE;

    // ---- the added ratings, checked and sorted both ways, in scratch ----
    size_t work_bytes = 0;
    carve(nullptr, nd, nl, nr, &work_bytes);
    void *wb;
    RS_TRY(rs_scratch_get(h, RS_SCR_UPD_WORK, work_bytes, &wb));
    const Work w = carve(wb, nd, nl, nr, &work_bytes);
    RS_CUDA(cudaMemsetAsync(w.flags, 0, 16, st));
    if (nd > 0) {
        const int lb = bits_for(nl), rb = bits_for(nr);
        const int n = (int)nd;
        upd_validate_kernel<<<blocks_for(nd), T, 0, st>>>(d_left, d_right, d_rating, nd, nl, nr, w.idx, w.ls, w.rs,
                                                           w.flags);
        // (left, right asc) as Fit sorts: stable by right, then stable by left
        RS_UPD_SORT([&](void *t, size_t &b) {
            return cub::DeviceRadixSort::SortPairs(t, b, w.rs, w.keys_a, w.idx, w.perm_r, n, 0, rb, st);
        });
        gather_keys_kernel<<<blocks_for(nd), T, 0, st>>>(w.ls, w.perm_r, nd, w.keys_b);
        RS_UPD_SORT([&](void *t, size_t &b) {
            return cub::DeviceRadixSort::SortPairs(t, b, w.keys_b, w.keys_l, w.perm_r, w.perm_lr, n, 0, lb, st);
        });
        gather_keys_kernel<<<blocks_for(nd), T, 0, st>>>(w.rs, w.perm_lr, nd, w.col_lr);
        dup_check_kernel<<<blocks_for(nd), T, 0, st>>>(w.keys_l, w.col_lr, nd, w.flags);
        upd_dup_kernel<<<blocks_for(nd), T, 0, st>>>(w.keys_l, w.col_lr, nd, h->l_ptr, h->l_col, nl0, w.flags);
        ptr_from_sorted_kernel<<<blocks_for(nd + 1), T, 0, st>>>(w.keys_l, nd, nl, w.ptr_l);
        // (right, left asc): stable by right of the (left, right) order
        RS_UPD_SORT([&](void *t, size_t &b) {
            return cub::DeviceRadixSort::SortPairs(t, b, w.col_lr, w.keys_r, w.perm_lr, w.perm_rl, n, 0, rb, st);
        });
        gather_keys_kernel<<<blocks_for(nd), T, 0, st>>>(w.ls, w.perm_rl, nd, w.col_rl);
        ptr_from_sorted_kernel<<<blocks_for(nd + 1), T, 0, st>>>(w.keys_r, nd, nr, w.ptr_r);
        // dataset order inside a left row: stable by left of the call order (the sorted keys are keys_l again)
        if (dataset_order)
            RS_UPD_SORT([&](void *t, size_t &b) {
                return cub::DeviceRadixSort::SortPairs(t, b, w.ls, w.keys_a, w.idx, w.perm_l, n, 0, lb, st);
            });
        h->prof.total_launches += 8;
    } else {
        RS_CUDA(cudaMemsetAsync(w.ptr_l, 0, ((size_t)nl + 1) * 8, st));
        RS_CUDA(cudaMemsetAsync(w.ptr_r, 0, ((size_t)nr + 1) * 8, st));
    }
    // the touched rows, longest merged row first (stable: ties by id), and the longest merged right row
    upd_touched_kernel<<<blocks_for(nl), T, 0, st>>>(h->l_ptr, nl0, w.ptr_l, nl, w.len, w.ids, w.flags);
    upd_right_len_kernel<<<blocks_for(nr), T, 0, st>>>(h->r_ptr, nr0, w.ptr_r, nr, w.flags);
    RS_UPD_SORT([&](void *t, size_t &b) {
        return cub::DeviceRadixSort::SortPairsDescending(t, b, w.len, w.len_sorted, w.ids, w.rows, (int)nl, 0, 32, st);
    });
    h->prof.total_launches += 2;
    RS_CUDA(cudaGetLastError());
    int32_t f[3];
    RS_CUDA(cudaMemcpyAsync(f, w.flags, 12, cudaMemcpyDeviceToHost, st));
    RS_CUDA(cudaStreamSynchronize(st));
    if (f[0] & FLAG_BAD_ID) {
        rs_set_error("rs_knn_update: rating rows contain inner ids outside [0,%d) x [0,%d)", nl, nr);
        return RS_ERR_INVALID;
    }
    if (f[0] & FLAG_NAN) {
        rs_set_error("rs_knn_update: NaN ratings are not supported");
        return RS_ERR_UNSUPPORTED;
    }
    if (int8 && (f[0] & FLAG_NOT_INT8)) {
        rs_set_error("rs_knn_update: the model was fitted on integer ratings in [-11,11] and keeps no dataset order "
                     "of them; a rating outside that class needs a refit");
        return RS_ERR_UNSUPPORTED;
    }
    if (f[0] & FLAG_DUP) {
        rs_set_error("rs_knn_update: a (left,right) pair the model holds already, or twice among the added ratings");
        return RS_ERR_DUPLICATE;
    }
    const int64_t n_touched = f[1];
    const int32_t max_right_len = f[2] > h->max_right_len ? f[2] : h->max_right_len;

    // ---- every block the update writes, before the model is written ----
    int64_t *l_ptr, *r_ptr;
    int32_t *l_col, *r_col, *row_cnt = h->row_cnt, *row_sum = h->row_sum;
    double *l_val, *r_val, *ld_val = h->ld_val, *means, *stddevs, *pmeans;
    uint8_t *l_code = h->l_code;
    RS_TRY(spare_of(h, RS_UPD_L_PTR, (int64_t)nl + 1, &l_ptr));
    RS_TRY(spare_of(h, RS_UPD_L_COL, nnz, &l_col));
    RS_TRY(spare_of(h, RS_UPD_L_VAL, nnz, &l_val));
    if (int8) RS_TRY(spare_of(h, RS_UPD_L_CODE, nnz, &l_code));
    if (dataset_order) RS_TRY(spare_of(h, RS_UPD_LD_VAL, nnz, &ld_val));
    RS_TRY(spare_of(h, RS_UPD_R_PTR, (int64_t)nr + 1, &r_ptr));
    RS_TRY(spare_of(h, RS_UPD_R_COL, nnz, &r_col));
    RS_TRY(spare_of(h, RS_UPD_R_VAL, nnz, &r_val));
    RS_TRY(spare_of(h, RS_UPD_MEANS, (int64_t)nl + 1, &means));
    RS_TRY(spare_of(h, RS_UPD_STDDEVS, (int64_t)nl + 1, &stddevs));
    RS_TRY(spare_of(h, RS_UPD_PMEANS, (int64_t)nl + 1, &pmeans));
    if (int8) {
        RS_TRY(spare_of(h, RS_UPD_ROW_CNT, (int64_t)nl + 1, &row_cnt));
        RS_TRY(spare_of(h, RS_UPD_ROW_SUM, (int64_t)nl + 1, &row_sum));
    }
    // the matrix: new rows fit in place while ld_s = ceil(n_left / 16) * 16 keeps its value and the block has the
    // rows; otherwise a block of ld_s rows in the new layout takes the old rows
    const int64_t ld = ((int64_t)nl + 15) / 16 * 16;
    double *sims = h->sims;
    void *grown = nullptr;
    size_t grown_bytes = 0;
    if (nl > nl0 && !(ld == h->ld_s && h->upd_sims && h->upd_sims_bytes >= (size_t)nl * ld * 8)) {
        RS_TRY(rs_cached_malloc(h->device, &grown, (size_t)ld * ld * 8, &grown_bytes));
        sims = static_cast<double *>(grown);
    }
    const int64_t batch = n_touched > 0 ? slab_batch(ld, n_touched) : 0;
    void *slab = nullptr, *counter = nullptr;
    if (n_touched > 0) {
        int32_t rc = rs_scratch_get(h, RS_SCR_UPD_SLAB, (size_t)batch * ld * 8, &slab);
        if (rc == RS_OK) rc = rs_scratch_get(h, RS_SCR_GIVEN_COUNTER, 8, &counter);   // rs_given_sims_launch's
        if (rc != RS_OK) {
            rs_cached_free(h->device, grown, grown_bytes);
            return rc;
        }
    }

    // ---- the merged CSRs, into the spares ----
    upd_ptr_kernel<<<blocks_for((int64_t)nl + 1), T, 0, st>>>(h->l_ptr, nl0, w.ptr_l, nl, l_ptr);
    upd_ptr_kernel<<<blocks_for((int64_t)nr + 1), T, 0, st>>>(h->r_ptr, nr0, w.ptr_r, nr, r_ptr);
    upd_merge_old_kernel<<<blocks_for((int64_t)nl0 * 32), T, 0, st>>>(h->l_ptr, h->l_col, h->l_val, nl0, w.ptr_l,
                                                                       w.col_lr, l_ptr, l_col, l_val,
                                                                       int8 ? l_code : nullptr);
    upd_merge_old_kernel<<<blocks_for((int64_t)nr0 * 32), T, 0, st>>>(h->r_ptr, h->r_col, h->r_val, nr0, w.ptr_r,
                                                                       w.col_rl, r_ptr, r_col, r_val, nullptr);
    if (dataset_order)
        upd_merge_old_kernel<<<blocks_for((int64_t)nl0 * 32), T, 0, st>>>(h->l_ptr, nullptr, h->ld_val, nl0, w.ptr_l,
                                                                           nullptr, l_ptr, nullptr, ld_val, nullptr);
    h->prof.total_launches += dataset_order ? 5 : 4;
    if (nd > 0) {
        upd_merge_new_kernel<<<blocks_for(nd), T, 0, st>>>(w.keys_l, w.col_lr, w.perm_lr, d_rating, nd, h->l_ptr,
                                                            h->l_col, nl0, w.ptr_l, l_ptr, l_col, l_val,
                                                            int8 ? l_code : nullptr);
        upd_merge_new_kernel<<<blocks_for(nd), T, 0, st>>>(w.keys_r, w.col_rl, w.perm_rl, d_rating, nd, h->r_ptr,
                                                            h->r_col, nr0, w.ptr_r, r_ptr, r_col, r_val, nullptr);
        if (dataset_order)
            upd_merge_new_kernel<<<blocks_for(nd), T, 0, st>>>(w.keys_l, nullptr, w.perm_l, d_rating, nd, h->l_ptr,
                                                                nullptr, nl0, w.ptr_l, l_ptr, nullptr, ld_val, nullptr);
        h->prof.total_launches += dataset_order ? 3 : 2;
    }
    if (grown) {
        RS_CUDA(cudaMemcpy2DAsync(sims, (size_t)ld * 8, h->sims, (size_t)h->ld_s * 8, (size_t)nl0 * 8, (size_t)nl0,
                                  cudaMemcpyDeviceToDevice, st));
    }

    // ---- the model: the merged arrays, the statistics, the touched rows and columns ----
    const int arrays[] = {RS_UPD_L_PTR, RS_UPD_L_COL, RS_UPD_L_VAL, RS_UPD_R_PTR, RS_UPD_R_COL, RS_UPD_R_VAL,
                          RS_UPD_MEANS, RS_UPD_STDDEVS, RS_UPD_PMEANS};
    for (int a : arrays) h->upd[a].cur = h->upd[a].cur == 0 ? 1 : 0;
    if (int8)
        for (int a : {RS_UPD_L_CODE, RS_UPD_ROW_CNT, RS_UPD_ROW_SUM}) h->upd[a].cur = h->upd[a].cur == 0 ? 1 : 0;
    if (dataset_order) h->upd[RS_UPD_LD_VAL].cur = h->upd[RS_UPD_LD_VAL].cur == 0 ? 1 : 0;
    h->l_ptr = l_ptr; h->l_col = l_col; h->l_val = l_val; h->l_code = l_code; h->ld_val = ld_val;
    h->r_ptr = r_ptr; h->r_col = r_col; h->r_val = r_val;
    h->means = means; h->stddevs = stddevs; h->pmeans = pmeans; h->row_cnt = row_cnt; h->row_sum = row_sum;
    void *old_sims = nullptr;
    size_t old_sims_bytes = 0;
    if (grown) {
        old_sims = h->upd_sims;                  // null while the matrix is the Fit's, in the arena
        old_sims_bytes = h->upd_sims_bytes;
        h->upd_sims = grown;
        h->upd_sims_bytes = grown_bytes;
        h->sims = sims;
    }
    h->nnz = nnz;
    h->n_left = nl;
    h->n_right = nr;
    h->row_end = nl;
    h->rows_local = nl;
    h->ld_s = ld;
    h->max_right_len = max_right_len;
    h->global_mean = global_mean;
    h->planes = nullptr;                         // rs_knn_cosums rebuilds the int8 planes of the union ...
    h->updated = true;                           // ... into a block of their own (rs_prep_planes)
    RS_TRY(rs_prep_stats(h));
    // the statistics are final when the call returns, as Fit's are: rs_knn_means / rs_knn_stddevs read them on the
    // auxiliary stream, which does not wait for this one
    RS_CUDA(cudaStreamSynchronize(st));
    for (int64_t b0 = 0; b0 < n_touched; b0 += batch) {
        const int64_t nb = n_touched - b0 < batch ? n_touched - b0 : batch;
        RS_TRY(rs_given_sims_launch(h, h->l_ptr, h->l_col, h->l_val, h->pmeans, nb, (double *)slab, ld, w.rows + b0));
        upd_scatter_kernel<<<blocks_for(nb * nl), T, 0, st>>>((const double *)slab, ld, w.rows + b0, nb, nl, sims);
        h->prof.total_launches++;
    }
    RS_CUDA(cudaGetLastError());
    if (old_sims) {                              // the old matrix is free once its copy has run
        RS_CUDA(cudaStreamSynchronize(st));
        rs_cached_free(h->device, old_sims, old_sims_bytes);
    }
    return RS_OK;
}

// The blocks of the updates go back to the cache; the next Fit's arrays are in the arena.  The caller has drained the
// handle's stream.
void rs_update_release(rs_knn *h) {
    for (rs_knn::UpdArray &u : h->upd) {
        for (int s = 0; s < 2; s++) rs_cached_free(h->device, u.p[s], u.bytes[s]);
        u = rs_knn::UpdArray{};
    }
    rs_cached_free(h->device, h->upd_sims, h->upd_sims_bytes);
    h->upd_sims = nullptr;
    h->upd_sims_bytes = 0;
    rs_cached_free(h->device, h->upd_planes, h->upd_planes_bytes);
    h->upd_planes = nullptr;
    h->upd_planes_bytes = 0;
    h->updated = false;
}
