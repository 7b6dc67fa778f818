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
// A cyclic row shard (rs_knn_update_sharded_device) merges the same ratings into its copies of the CSRs and the
// statistics, and recomputes the cells it stores: the full rows of the touched ids it owns, and, for a touched id i that
// another shard owns, the column S[v][i] of each row v it owns (given_sims_kernel<SIM, true>, about N / R cells).
// rs_knn_remove / rs_knn_change (rs_edit_run) edit pairs the model holds: the edited model is the Fit of the remaining
// or changed ratings in their dataset order under the same ids and counts, bit for bit (DESIGN.md §5.3e).  The ids an
// edit names are its touched rows; the CSRs are edited instead of merged (an entry is dropped and the rest of its row
// closes up, or it takes the new rating in place), and the rest is the update's: the statistics of every row, the
// similarity rows of the touched ids, and the cells between untouched rows kept.
// Everything up to the one read-back of the checks goes to scratch; the model's merged or edited arrays go to spare
// blocks (rs_knn::upd), and the model is written only when every check has passed and every block is allocated, so a
// refused call, or one that runs out of memory, leaves the model as it was.
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

// The checks of Fit on the added or changed ratings (ids in range, no NaN, the rating class; a removal has no rating),
// and the ids the sorts use: an id out of range becomes 0, so that every kernel before the read-back stays in bounds.
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
    int f = ok ? 0 : FLAG_BAD_ID;
    if (rating) {
        const double v = rating[e];
        if (v != v) f |= FLAG_NAN;
        if (!(v == rint(v) && fabs(v) <= 11.0)) f |= FLAG_NOT_INT8;
    }
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

// An edited (left, right) pair the fitted left CSR does not hold (the right CSR holds the same pairs).
__global__ void edit_missing_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col, int64_t nd,
                                    const int64_t *__restrict__ l_ptr, const int32_t *__restrict__ l_col,
                                    int32_t *__restrict__ flags) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nd) return;
    const int32_t i = row[e], c = col[e];
    const int64_t b = l_ptr[i], end = l_ptr[i + 1];
    const int64_t p = lower_bound_id(l_col, b, end, c);
    if (!(p < end && l_col[p] == c)) atomicOr(flags, FLAG_MISSING);
}

// The touched left rows, each keyed by its merged or edited length + 1 (0: untouched) and, above that, bit 31 for the
// rows the handle owns (every row unless it is a cyclic shard), for a sort that puts the owned rows first, each group
// longest first; flags[1] counts them, flags[3] the owned ones.  d_ptr: the added or edited ratings' row pointers;
// dsign: what each of them does to its row's length (+1 added, -1 removed, 0 changed).
__global__ void upd_touched_kernel(const int64_t *__restrict__ l_ptr, int32_t nl0, const int64_t *__restrict__ d_ptr,
                                   int32_t nl, int32_t dsign, int32_t cyc_R, int32_t cyc_r, uint32_t *__restrict__ key,
                                   int32_t *__restrict__ ids, int32_t *__restrict__ flags) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nl) return;
    const int64_t dl = d_ptr[i + 1] - d_ptr[i];
    const bool touched = dl > 0 || i >= nl0;
    const bool owned = cyc_R < 2 || rs_cyc_owns(i, cyc_R, cyc_r);
    const int64_t len = (i < nl0 ? l_ptr[i + 1] - l_ptr[i] : 0) + dsign * dl + 1;
    key[i] = touched ? (owned ? 0x80000000u : 0u) | (uint32_t)(len < 0x7fffffff ? len : 0x7fffffff) : 0u;
    ids[i] = i;
    if (touched) atomicAdd(flags + 1, 1);
    if (touched && owned) atomicAdd(flags + 3, 1);
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
// ascending; null: no added entry comes before an old one, the dataset order of ld_val and ld_col).  code: the byte
// codes.  V: the values' type (double; int32_t for ld_col, the right ids in dataset order).
template <typename V>
__global__ void upd_merge_old_kernel(const int64_t *__restrict__ old_ptr, const int32_t *__restrict__ old_col,
                                     const V *__restrict__ old_val, int32_t n0, const int64_t *__restrict__ d_ptr,
                                     const int32_t *__restrict__ d_col, const int64_t *__restrict__ new_ptr,
                                     int32_t *__restrict__ col, V *__restrict__ val, uint8_t *__restrict__ code) {
    const int32_t i = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n0) return;
    const int64_t b = old_ptr[i], e = old_ptr[i + 1], db = d_ptr[i], de = d_ptr[i + 1];
    const int64_t base = new_ptr[i] - b;
    for (int64_t x = b + lane; x < e; x += 32) {
        const V v = old_val[x];
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
// all of them).  V as in upd_merge_old_kernel: `rating` is the added right ids for ld_col.
template <typename V>
__global__ void upd_merge_new_kernel(const int32_t *__restrict__ key, const int32_t *__restrict__ d_col,
                                     const int32_t *__restrict__ perm, const V *__restrict__ rating, int64_t nd,
                                     const int64_t *__restrict__ old_ptr, const int32_t *__restrict__ old_col,
                                     int32_t n0, const int64_t *__restrict__ d_ptr, const int64_t *__restrict__ new_ptr,
                                     int32_t *__restrict__ col, V *__restrict__ val, uint8_t *__restrict__ code) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nd) return;
    const int32_t i = key[e];
    const int64_t b = i < n0 ? old_ptr[i] : 0, end = i < n0 ? old_ptr[i + 1] : 0;
    int64_t pos = new_ptr[i] + (e - d_ptr[i]);
    const V v = rating[perm[e]];
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

// edited row pointers: removal, out[i] = old_ptr[i] - (removals in rows < i); change, the old ones
__global__ void edit_ptr_kernel(const int64_t *__restrict__ old_ptr, const int64_t *__restrict__ d_ptr, int32_t n,
                                bool remove, int64_t *__restrict__ out) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    out[i] = old_ptr[i] - (remove ? d_ptr[i] : 0);
}

// A CSR sorted by id after the edits, one warp per row.  The position p of entry x's id among the row's edited ids
// (d_col[d_ptr[i] .. d_ptr[i+1]), ascending) says whether it is edited and, as every edited id is in the row, how many
// removals come before it.  rating null (removal): an edited entry is dropped and a kept one moves back by p - db;
// otherwise (change) an edited entry takes rating[perm[p]] in place.  code: the byte codes, code_int8_kernel's.
__global__ void edit_sorted_kernel(const int64_t *__restrict__ old_ptr, const int32_t *__restrict__ old_col,
                                   const double *__restrict__ old_val, int32_t n, const int64_t *__restrict__ d_ptr,
                                   const int32_t *__restrict__ d_col, const int32_t *__restrict__ perm,
                                   const double *__restrict__ rating, const int64_t *__restrict__ new_ptr,
                                   int32_t *__restrict__ col, double *__restrict__ val, uint8_t *__restrict__ code) {
    const int32_t i = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n) return;
    const int64_t b = old_ptr[i], e = old_ptr[i + 1], db = d_ptr[i], de = d_ptr[i + 1];
    const int64_t base = new_ptr[i] - b;
    for (int64_t x = b + lane; x < e; x += 32) {
        const int32_t c = old_col[x];
        const int64_t p = lower_bound_id(d_col, db, de, c);
        const bool hit = p < de && d_col[p] == c;
        double v = old_val[x];
        int64_t pos = base + x;
        if (rating) {
            if (hit) v = rating[perm[p]];
        } else {
            if (hit) continue;
            pos -= p - db;
        }
        col[pos] = c;
        val[pos] = v;
        if (code) code[pos] = (uint8_t)((int)v + RS_INT8_BIAS);
    }
}

// The dataset-order arrays of the left rows (ld_col, ld_val) after the edits, one warp per row, 32 entries at a time:
// whether an entry is edited comes from a binary search of its id in the row's edited ids (d_col as above).  rating
// null (removal): the kept entries close up in their order (__ballot_sync, and __popc of the lower lanes for the
// place); otherwise (change) an edited entry takes rating[perm[p]] in place.  A row without edits is copied.
__global__ void edit_dataset_kernel(const int64_t *__restrict__ old_ptr, const int32_t *__restrict__ old_dcol,
                                    const double *__restrict__ old_dval, int32_t n, const int64_t *__restrict__ d_ptr,
                                    const int32_t *__restrict__ d_col, const int32_t *__restrict__ perm,
                                    const double *__restrict__ rating, const int64_t *__restrict__ new_ptr,
                                    int32_t *__restrict__ dcol, double *__restrict__ dval) {
    const int32_t i = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n) return;                          // the whole warp: one row per warp, blocks of whole warps
    const int64_t b = old_ptr[i], e = old_ptr[i + 1], db = d_ptr[i], de = d_ptr[i + 1];
    int64_t out = new_ptr[i];
    for (int64_t x0 = b; x0 < e; x0 += 32) {
        const int64_t x = x0 + lane;
        const bool in = x < e;
        const int32_t c = in ? old_dcol[x] : 0;
        double v = in ? old_dval[x] : 0.0;
        const int64_t p = in ? lower_bound_id(d_col, db, de, c) : de;
        const bool hit = p < de && d_col[p] == c;
        if (rating) {
            if (hit) v = rating[perm[p]];
            if (in) {
                dcol[out + (x - b)] = c;
                dval[out + (x - b)] = v;
            }
        } else {
            const bool keep = in && !hit;
            const unsigned kept = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                const int64_t pos = out + __popc(kept & ((1u << lane) - 1u));
                dcol[pos] = c;
                dval[pos] = v;
            }
            out += __popc(kept);
        }
    }
}

// Row i = rows[b] of the matrix and its column from the recomputed row slab[b]: S[i][v] = S[v][i] = slab[b][v], the
// diagonal NaN as Fit leaves it.  Two touched rows write the same bits into their common cells: Sim(i, j) and
// Sim(j, i) sum the same terms in the same order.  A cyclic shard (cyc_R >= 2) owns row i, stores it at its local row,
// and writes the column into the rows v it owns.
__global__ void upd_scatter_kernel(const double *__restrict__ slab, int64_t ld, const int32_t *__restrict__ rows,
                                   int64_t nb, int32_t n, int32_t cyc_R, int32_t cyc_r, double *__restrict__ sims) {
    const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= nb * n) return;
    const int64_t b = x / n;
    const int32_t v = (int32_t)(x - b * n);
    const int32_t i = rows[b];
    const double s = v == i ? __longlong_as_double(0x7ff8000000000001ll) : slab[b * ld + v];
    if (cyc_R < 2) {
        sims[(int64_t)i * ld + v] = s;
        sims[(int64_t)v * ld + i] = s;
    } else {
        sims[rs_cyc_local(i, cyc_R) * ld + v] = s;
        if (rs_cyc_owns(v, cyc_R, cyc_r)) sims[rs_cyc_local(v, cyc_R) * ld + i] = s;
    }
}

// A cyclic shard's column i = rows[b] of a row another shard owns, from its own-row slab[b] (given_sims_kernel<SIM,
// true>): S[loc][i] = slab[b][loc] for each of its n_own local rows.  Where it meets an owned touched row j, the two
// writes carry the same bits, as above.
__global__ void upd_scatter_own_kernel(const double *__restrict__ slab, int64_t n_own, const int32_t *__restrict__ rows,
                                       int64_t nb, int64_t ld, double *__restrict__ sims) {
    const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= nb * n_own) return;
    const int64_t b = x / n_own, loc = x - b * n_own;
    sims[loc * ld + rows[b]] = slab[b * n_own + loc];
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
    int32_t *flags;           // [0] FLAG_*, [1] touched rows, [2] longest merged right row, [3] touched rows owned
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

#define RS_UPD_SORT(CALL)                                                                                  \
    do {                                                                                                   \
        void *t_ = nullptr;                                                                                \
        size_t need_ = 0;                                                                                  \
        RS_CUDA(CALL(nullptr, need_));                                                                     \
        RS_TRY(rs_scratch_get(h, RS_SCR_UPD_SORT_TMP, need_ + 256, &t_));                                  \
        RS_CUDA(CALL(t_, need_));                                                                          \
    } while (0)

enum Mode { UPD_ADD, UPD_REMOVE, UPD_CHANGE };

// The first half of an update or an edit, in scratch: the ratings checked and sorted by (left, right) and by (right,
// left), their row pointers, the duplicate check (ADD: and the pairs the model holds; REMOVE / CHANGE: the pairs it does
// not hold), the touched rows sorted owned first, each group longest first, and the one read-back, f[0..3] (upd.flags).
// Refusals return here, before anything of the model is written.
int32_t upd_prepare(rs_knn *h, const char *who, Mode mode, const int32_t *d_left, const int32_t *d_right,
                    const double *d_rating, int64_t nd, int32_t nl, int32_t nr, Work *out, int32_t f[4]) {
    cudaStream_t st = h->stream;
    const int32_t nl0 = h->n_left, nr0 = h->n_right;
    const bool int8 = h->rating_class == RS_CLASS_INT8;
    const bool add = mode == UPD_ADD;
    const int32_t cyc_R = h->cyc_R > 1 ? h->cyc_R : 0, cyc_r = h->cyc_r;
    // Fit keeps the dataset-order values only where a statistic is summed in that order (prep.cu)
    const bool dataset_order = !int8 || h->p.knn_type == RS_KNN_ZSCORE;

    size_t work_bytes = 0;
    carve(nullptr, nd, nl, nr, &work_bytes);
    void *wb;
    RS_TRY(rs_scratch_get(h, RS_SCR_UPD_WORK, work_bytes, &wb));
    const Work w = carve(wb, nd, nl, nr, &work_bytes);
    *out = w;
    RS_CUDA(cudaMemsetAsync(w.flags, 0, 16, st));
    if (nd > 0) {
        const int lb = bits_for(nl), rb = bits_for(nr);
        const int n = (int)nd;
        upd_validate_kernel<<<blocks_for(nd), T, 0, st>>>(d_left, d_right, mode == UPD_REMOVE ? nullptr : d_rating, nd,
                                                           nl, nr, w.idx, w.ls, w.rs, w.flags);
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
        if (add)
            upd_dup_kernel<<<blocks_for(nd), T, 0, st>>>(w.keys_l, w.col_lr, nd, h->l_ptr, h->l_col, nl0, w.flags);
        else
            edit_missing_kernel<<<blocks_for(nd), T, 0, st>>>(w.keys_l, w.col_lr, nd, h->l_ptr, h->l_col, w.flags);
        ptr_from_sorted_kernel<<<blocks_for(nd + 1), T, 0, st>>>(w.keys_l, nd, nl, w.ptr_l);
        // (right, left asc): stable by right of the (left, right) order
        RS_UPD_SORT([&](void *t, size_t &b) {
            return cub::DeviceRadixSort::SortPairs(t, b, w.col_lr, w.keys_r, w.perm_lr, w.perm_rl, n, 0, rb, st);
        });
        gather_keys_kernel<<<blocks_for(nd), T, 0, st>>>(w.ls, w.perm_rl, nd, w.col_rl);
        ptr_from_sorted_kernel<<<blocks_for(nd + 1), T, 0, st>>>(w.keys_r, nd, nr, w.ptr_r);
        // dataset order inside a left row: stable by left of the call order (the sorted keys are keys_l again); an
        // edit finds its entry in that order by its right id instead
        if (add && dataset_order)
            RS_UPD_SORT([&](void *t, size_t &b) {
                return cub::DeviceRadixSort::SortPairs(t, b, w.ls, w.keys_a, w.idx, w.perm_l, n, 0, lb, st);
            });
        h->prof.total_launches += 8;
    } else {
        RS_CUDA(cudaMemsetAsync(w.ptr_l, 0, ((size_t)nl + 1) * 8, st));
        RS_CUDA(cudaMemsetAsync(w.ptr_r, 0, ((size_t)nr + 1) * 8, st));
    }
    // the touched rows, owned first, each group longest merged or edited row first (stable: ties by id), and the
    // longest merged right row (an edit keeps max_right_len: a bound on the candidates, which no removal raises)
    upd_touched_kernel<<<blocks_for(nl), T, 0, st>>>(h->l_ptr, nl0, w.ptr_l, nl,
                                                      mode == UPD_ADD ? 1 : mode == UPD_REMOVE ? -1 : 0, cyc_R, cyc_r,
                                                      w.len, w.ids, w.flags);
    if (add) upd_right_len_kernel<<<blocks_for(nr), T, 0, st>>>(h->r_ptr, nr0, w.ptr_r, nr, w.flags);
    RS_UPD_SORT([&](void *t, size_t &b) {
        return cub::DeviceRadixSort::SortPairsDescending(t, b, w.len, w.len_sorted, w.ids, w.rows, (int)nl, 0, 32, st);
    });
    h->prof.total_launches += add ? 2 : 1;
    RS_CUDA(cudaGetLastError());
    RS_CUDA(cudaMemcpyAsync(f, w.flags, 16, cudaMemcpyDeviceToHost, st));
    RS_CUDA(cudaStreamSynchronize(st));
    if (f[0] & FLAG_BAD_ID) {
        rs_set_error("%s: rating rows contain inner ids outside [0,%d) x [0,%d)", who, nl, nr);
        return RS_ERR_INVALID;
    }
    if (f[0] & FLAG_MISSING) {
        rs_set_error("%s: a (left,right) pair the model does not hold", who);
        return RS_ERR_INVALID;
    }
    if (f[0] & FLAG_NAN) {
        rs_set_error("%s: NaN ratings are not supported", who);
        return RS_ERR_UNSUPPORTED;
    }
    if (int8 && (f[0] & FLAG_NOT_INT8)) {
        rs_set_error("%s: the model was fitted on integer ratings in [-11,11] and keeps no dataset order of them; a "
                     "rating outside that class needs a refit", who);
        return RS_ERR_UNSUPPORTED;
    }
    if (f[0] & FLAG_DUP) {
        rs_set_error(add ? "%s: a (left,right) pair the model holds already, or twice among the added ratings"
                         : "%s: a (left,right) pair named twice", who);
        return RS_ERR_DUPLICATE;
    }
    return RS_OK;
}

// The model array a's spare becomes the model's.
void upd_swap(rs_knn *h, int a) { h->upd[a].cur = h->upd[a].cur == 0 ? 1 : 0; }

// The scratch of the recompute, allocated before the model is written: the slab of a batch of recomputed rows (owned
// rows: full rows of ld; other shards' rows: columns of the handle's rows) and the counter of rs_given_sims_launch.
struct Slab {
    int64_t batch = 0, batch_own = 0;
    double *p = nullptr;
};

int32_t upd_slab(rs_knn *h, int64_t n_owned, int64_t n_foreign, int64_t ld, int64_t rows, Slab *s) {
    s->batch = n_owned > 0 ? slab_batch(ld, n_owned) : 0;
    s->batch_own = n_foreign > 0 ? slab_batch(rows, n_foreign) : 0;
    const size_t slab_bytes = (size_t)(s->batch * ld > s->batch_own * rows ? s->batch * ld : s->batch_own * rows) * 8;
    if (n_owned + n_foreign == 0) return RS_OK;
    void *slab = nullptr, *counter = nullptr;
    RS_TRY(rs_scratch_get(h, RS_SCR_UPD_SLAB, slab_bytes, &slab));
    RS_TRY(rs_scratch_get(h, RS_SCR_GIVEN_COUNTER, 8, &counter));
    s->p = static_cast<double *>(slab);
    return RS_OK;
}

// The second half, on the model as it now stands (its CSRs merged or edited, its counts and ld_s final): the
// statistics of every row with Fit's kernels, the int8 planes dropped, and the similarity rows of the touched ids
// (touched[0 .. n_owned): rows the handle owns, then n_foreign rows of other shards), longest first in batches,
// written into their rows and columns of the matrix.
int32_t upd_recompute(rs_knn *h, const int32_t *touched, int64_t n_owned, int64_t n_foreign, const Slab &s) {
    cudaStream_t st = h->stream;
    const int32_t nl = h->n_left;
    const int32_t cyc_R = h->cyc_R > 1 ? h->cyc_R : 0, cyc_r = h->cyc_r;
    const int64_t ld = h->ld_s, rows = h->rows_local;
    double *sims = h->sims;
    h->planes = nullptr;                         // rs_knn_cosums rebuilds the int8 planes of the new ratings ...
    h->updated = true;                           // ... into a block of their own (rs_prep_planes)
    // the tensor path's limits of the new ratings (rs_knn_cosums), read back with the synchronisation below
    int32_t fl[16];
    RS_CUDA(cudaMemsetAsync(h->d_flags + RS_FL_ABS_MAX, 0, 4, st));
    RS_CUDA(cudaMemsetAsync(h->d_flags + RS_FL_LEN_TOP2, 0, 8, st));
    RS_TRY(rs_prep_stats(h));
    RS_CUDA(cudaMemcpyAsync(fl, h->d_flags, sizeof(fl), cudaMemcpyDeviceToHost, st));
    // the statistics are final when the call returns, as Fit's are: rs_knn_means / rs_knn_stddevs read them on the
    // auxiliary stream, which does not wait for this one
    RS_CUDA(cudaStreamSynchronize(st));
    rs_tensor_limits_read(h, fl);
    for (int64_t b0 = 0; b0 < n_owned; b0 += s.batch) {
        const int64_t nb = n_owned - b0 < s.batch ? n_owned - b0 : s.batch;
        RS_TRY(rs_given_sims_launch(h, h->l_ptr, h->l_col, h->l_val, h->pmeans, nb, s.p, ld, touched + b0));
        upd_scatter_kernel<<<blocks_for(nb * nl), T, 0, st>>>(s.p, ld, touched + b0, nb, nl, cyc_R, cyc_r, sims);
        h->prof.total_launches++;
    }
    const int32_t *foreign = touched + n_owned;
    for (int64_t b0 = 0; b0 < n_foreign; b0 += s.batch_own) {
        const int64_t nb = n_foreign - b0 < s.batch_own ? n_foreign - b0 : s.batch_own;
        RS_TRY(rs_given_sims_launch(h, h->l_ptr, h->l_col, h->l_val, h->pmeans, nb, s.p, rows, foreign + b0, true));
        upd_scatter_own_kernel<<<blocks_for(nb * rows), T, 0, st>>>(s.p, rows, foreign + b0, nb, ld, sims);
        h->prof.total_launches++;
    }
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

}  // namespace

int32_t rs_update_run(rs_knn *h, const int32_t *d_left, const int32_t *d_right, const double *d_rating, int64_t nd,
                      int32_t nl, int32_t nr, double global_mean) {
    cudaStream_t st = h->stream;
    const int32_t nl0 = h->n_left, nr0 = h->n_right;
    const int64_t nnz0 = h->nnz, nnz = nnz0 + nd;
    const bool int8 = h->rating_class == RS_CLASS_INT8;
    const int32_t cyc_R = h->cyc_R > 1 ? h->cyc_R : 0, cyc_r = h->cyc_r;
    const int64_t rows0 = h->rows_local, rows = cyc_R ? rs_cyc_rows(nl, cyc_R, cyc_r) : nl;   // the matrix's rows
    const bool dataset_order = !int8 || h->p.knn_type == RS_KNN_ZSCORE;

    // ---- the added ratings, checked and sorted both ways, in scratch ----
    Work w;
    int32_t f[4];
    RS_TRY(upd_prepare(h, h->cyc_R > 1 ? "rs_knn_update_sharded" : "rs_knn_update", UPD_ADD, d_left, d_right,
                       d_rating, nd, nl, nr, &w, f));
    const int64_t n_touched = f[1], n_owned = f[3];
    const int64_t n_foreign = rows > 0 ? n_touched - n_owned : 0;   // the touched rows of other shards
    const int32_t max_right_len = f[2] > h->max_right_len ? f[2] : h->max_right_len;

    // ---- every block the update writes, before the model is written ----
    int64_t *l_ptr, *r_ptr;
    int32_t *l_col, *r_col, *ld_col = h->ld_col, *row_cnt = h->row_cnt, *row_sum = h->row_sum;
    double *l_val, *r_val, *ld_val = h->ld_val, *means, *stddevs, *pmeans;
    uint8_t *l_code = h->l_code;
    RS_TRY(spare_of(h, RS_UPD_L_PTR, (int64_t)nl + 1, &l_ptr));
    RS_TRY(spare_of(h, RS_UPD_L_COL, nnz, &l_col));
    RS_TRY(spare_of(h, RS_UPD_L_VAL, nnz, &l_val));
    if (int8) RS_TRY(spare_of(h, RS_UPD_L_CODE, nnz, &l_code));
    if (dataset_order) {
        RS_TRY(spare_of(h, RS_UPD_LD_VAL, nnz, &ld_val));
        RS_TRY(spare_of(h, RS_UPD_LD_COL, nnz, &ld_col));
    }
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
    // rows; otherwise a block of the rows the handle holds at n_left = ld_s, in the new layout, takes the old rows
    const int64_t ld = ((int64_t)nl + 15) / 16 * 16;
    double *sims = h->sims;
    void *grown = nullptr;
    size_t grown_bytes = 0;
    if ((rows > rows0 || ld != h->ld_s) &&
        !(ld == h->ld_s && h->upd_sims && h->upd_sims_bytes >= (size_t)rows * ld * 8)) {
        const int64_t cap = cyc_R ? rs_cyc_rows(ld, cyc_R, cyc_r) : ld;
        RS_TRY(rs_cached_malloc(h->device, &grown, cap > 0 ? (size_t)cap * ld * 8 : 256, &grown_bytes));
        sims = static_cast<double *>(grown);
    }
    Slab slab;
    if (int32_t rc = upd_slab(h, n_owned, n_foreign, ld, rows, &slab)) {
        rs_cached_free(h->device, grown, grown_bytes);
        return rc;
    }

    // ---- the merged CSRs, into the spares ----
    upd_ptr_kernel<<<blocks_for((int64_t)nl + 1), T, 0, st>>>(h->l_ptr, nl0, w.ptr_l, nl, l_ptr);
    upd_ptr_kernel<<<blocks_for((int64_t)nr + 1), T, 0, st>>>(h->r_ptr, nr0, w.ptr_r, nr, r_ptr);
    upd_merge_old_kernel<<<blocks_for((int64_t)nl0 * 32), T, 0, st>>>(h->l_ptr, h->l_col, h->l_val, nl0, w.ptr_l,
                                                                       w.col_lr, l_ptr, l_col, l_val,
                                                                       int8 ? l_code : nullptr);
    upd_merge_old_kernel<<<blocks_for((int64_t)nr0 * 32), T, 0, st>>>(h->r_ptr, h->r_col, h->r_val, nr0, w.ptr_r,
                                                                       w.col_rl, r_ptr, r_col, r_val, nullptr);
    if (dataset_order) {
        upd_merge_old_kernel<<<blocks_for((int64_t)nl0 * 32), T, 0, st>>>(h->l_ptr, nullptr, h->ld_val, nl0, w.ptr_l,
                                                                           nullptr, l_ptr, nullptr, ld_val, nullptr);
        upd_merge_old_kernel<<<blocks_for((int64_t)nl0 * 32), T, 0, st>>>(h->l_ptr, nullptr, h->ld_col, nl0, w.ptr_l,
                                                                           nullptr, l_ptr, nullptr, ld_col, nullptr);
    }
    h->prof.total_launches += dataset_order ? 6 : 4;
    if (nd > 0) {
        upd_merge_new_kernel<<<blocks_for(nd), T, 0, st>>>(w.keys_l, w.col_lr, w.perm_lr, d_rating, nd, h->l_ptr,
                                                            h->l_col, nl0, w.ptr_l, l_ptr, l_col, l_val,
                                                            int8 ? l_code : nullptr);
        upd_merge_new_kernel<<<blocks_for(nd), T, 0, st>>>(w.keys_r, w.col_rl, w.perm_rl, d_rating, nd, h->r_ptr,
                                                            h->r_col, nr0, w.ptr_r, r_ptr, r_col, r_val, nullptr);
        if (dataset_order) {
            upd_merge_new_kernel<<<blocks_for(nd), T, 0, st>>>(w.keys_l, nullptr, w.perm_l, d_rating, nd, h->l_ptr,
                                                                nullptr, nl0, w.ptr_l, l_ptr, nullptr, ld_val, nullptr);
            upd_merge_new_kernel<<<blocks_for(nd), T, 0, st>>>(w.keys_l, nullptr, w.perm_l, d_right, nd, h->l_ptr,
                                                                nullptr, nl0, w.ptr_l, l_ptr, nullptr, ld_col, nullptr);
        }
        h->prof.total_launches += dataset_order ? 4 : 2;
    }
    if (grown && rows0 > 0) {
        RS_CUDA(cudaMemcpy2DAsync(sims, (size_t)ld * 8, h->sims, (size_t)h->ld_s * 8, (size_t)nl0 * 8, (size_t)rows0,
                                  cudaMemcpyDeviceToDevice, st));
    }

    // ---- the model: the merged arrays, the statistics, the touched rows and columns ----
    for (int a : {RS_UPD_L_PTR, RS_UPD_L_COL, RS_UPD_L_VAL, RS_UPD_R_PTR, RS_UPD_R_COL, RS_UPD_R_VAL, RS_UPD_MEANS,
                  RS_UPD_STDDEVS, RS_UPD_PMEANS})
        upd_swap(h, a);
    if (int8)
        for (int a : {RS_UPD_L_CODE, RS_UPD_ROW_CNT, RS_UPD_ROW_SUM}) upd_swap(h, a);
    if (dataset_order)
        for (int a : {RS_UPD_LD_VAL, RS_UPD_LD_COL}) upd_swap(h, a);
    h->l_ptr = l_ptr; h->l_col = l_col; h->l_val = l_val; h->l_code = l_code; h->ld_val = ld_val; h->ld_col = ld_col;
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
    h->rows_local = rows;
    h->ld_s = ld;
    h->max_right_len = max_right_len;
    h->global_mean = global_mean;
    RS_TRY(upd_recompute(h, w.rows, n_owned, n_foreign, slab));
    if (old_sims) {                              // the old matrix is free once its copy has run
        RS_CUDA(cudaStreamSynchronize(st));
        rs_cached_free(h->device, old_sims, old_sims_bytes);
    }
    return RS_OK;
}

int32_t rs_edit_run(rs_knn *h, bool remove, const int32_t *d_left, const int32_t *d_right, const double *d_rating,
                    int64_t nd, double global_mean) {
    const char *who = remove ? "rs_knn_remove" : "rs_knn_change";
    cudaStream_t st = h->stream;
    const int32_t nl = h->n_left, nr = h->n_right;
    const bool int8 = h->rating_class == RS_CLASS_INT8;
    const bool dataset_order = !int8 || h->p.knn_type == RS_KNN_ZSCORE;
    const double *rating = remove ? nullptr : d_rating;

    // ---- the edited pairs, checked, located and sorted both ways, in scratch ----
    Work w;
    int32_t f[4];
    RS_TRY(upd_prepare(h, who, remove ? UPD_REMOVE : UPD_CHANGE, d_left, d_right, d_rating, nd, nl, nr, &w, f));
    // every pair is held and named once: a removal of nnz of them leaves none
    const int64_t nnz = remove ? h->nnz - nd : h->nnz;
    if (nnz == 0) {
        rs_set_error("%s: the removal would leave no rating (a Fit needs at least one)", who);
        return RS_ERR_INVALID;
    }
    const int64_t n_touched = f[1];

    // ---- every block the edit writes, before the model is written ----
    int64_t *l_ptr, *r_ptr;
    int32_t *l_col, *r_col, *ld_col = h->ld_col, *row_cnt = h->row_cnt, *row_sum = h->row_sum;
    double *l_val, *r_val, *ld_val = h->ld_val, *means, *stddevs, *pmeans;
    uint8_t *l_code = h->l_code;
    RS_TRY(spare_of(h, RS_UPD_L_PTR, (int64_t)nl + 1, &l_ptr));
    RS_TRY(spare_of(h, RS_UPD_L_COL, nnz, &l_col));
    RS_TRY(spare_of(h, RS_UPD_L_VAL, nnz, &l_val));
    if (int8) RS_TRY(spare_of(h, RS_UPD_L_CODE, nnz, &l_code));
    if (dataset_order) {
        RS_TRY(spare_of(h, RS_UPD_LD_VAL, nnz, &ld_val));
        RS_TRY(spare_of(h, RS_UPD_LD_COL, nnz, &ld_col));
    }
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
    Slab slab;                                   // the counts do not change: the matrix keeps its block and layout
    RS_TRY(upd_slab(h, n_touched, 0, h->ld_s, h->rows_local, &slab));

    // ---- the edited CSRs, into the spares ----
    edit_ptr_kernel<<<blocks_for((int64_t)nl + 1), T, 0, st>>>(h->l_ptr, w.ptr_l, nl, remove, l_ptr);
    edit_ptr_kernel<<<blocks_for((int64_t)nr + 1), T, 0, st>>>(h->r_ptr, w.ptr_r, nr, remove, r_ptr);
    edit_sorted_kernel<<<blocks_for((int64_t)nl * 32), T, 0, st>>>(h->l_ptr, h->l_col, h->l_val, nl, w.ptr_l, w.col_lr,
                                                                    w.perm_lr, rating, l_ptr, l_col, l_val,
                                                                    int8 ? l_code : nullptr);
    edit_sorted_kernel<<<blocks_for((int64_t)nr * 32), T, 0, st>>>(h->r_ptr, h->r_col, h->r_val, nr, w.ptr_r, w.col_rl,
                                                                    w.perm_rl, rating, r_ptr, r_col, r_val, nullptr);
    if (dataset_order)
        edit_dataset_kernel<<<blocks_for((int64_t)nl * 32), T, 0, st>>>(h->l_ptr, h->ld_col, h->ld_val, nl, w.ptr_l,
                                                                         w.col_lr, w.perm_lr, rating, l_ptr, ld_col,
                                                                         ld_val);
    h->prof.total_launches += dataset_order ? 5 : 4;

    // ---- the model: the edited arrays, the statistics, the touched rows and columns ----
    for (int a : {RS_UPD_L_PTR, RS_UPD_L_COL, RS_UPD_L_VAL, RS_UPD_R_PTR, RS_UPD_R_COL, RS_UPD_R_VAL, RS_UPD_MEANS,
                  RS_UPD_STDDEVS, RS_UPD_PMEANS})
        upd_swap(h, a);
    if (int8)
        for (int a : {RS_UPD_L_CODE, RS_UPD_ROW_CNT, RS_UPD_ROW_SUM}) upd_swap(h, a);
    if (dataset_order)
        for (int a : {RS_UPD_LD_VAL, RS_UPD_LD_COL}) upd_swap(h, a);
    h->l_ptr = l_ptr; h->l_col = l_col; h->l_val = l_val; h->l_code = l_code; h->ld_val = ld_val; h->ld_col = ld_col;
    h->r_ptr = r_ptr; h->r_col = r_col; h->r_val = r_val;
    h->means = means; h->stddevs = stddevs; h->pmeans = pmeans; h->row_cnt = row_cnt; h->row_sum = row_sum;
    h->nnz = nnz;
    h->global_mean = global_mean;
    return upd_recompute(h, w.rows, n_touched, 0, slab);
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
