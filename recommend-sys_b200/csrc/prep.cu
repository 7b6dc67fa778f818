// prep.cu — device-side preparation for Fit: CSR construction from the inner-id COO,
// rating classification, row statistics, and the dense byte/int8 layouts the similarity
// kernels consume.  Follows the data-model contract of the reference:
//   core/data.go:185-216  adjacency lists are appended in dataset order
//   core/data.go:236-243  left rows are then sorted by id (unique keys)
//   core/data.go:222-235  means = sequential sum / count over the dataset-order row
//   core/knn.go:167-177   StdDevs[i] = sqrt(sum((x-mean)^2)/n) + 1e-5, dataset order
//   core/sim.go:49-62     Pearson recomputes sum/count over the id-sorted row
// CUB (ships with the CUDA toolkit) is used for the radix sorts and scans only.
#include <cub/cub.cuh>

#include <cstdlib>
#include <cstring>

#include "common.cuh"

int32_t rs_dev_alloc(rs_knn *h, void **out, size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    if (bytes == 0) bytes = 256;
    while (h->cur_chunk < h->chunks.size()) {
        rs_knn::Chunk &c = h->chunks[h->cur_chunk];
        if (h->cur_off + bytes <= c.bytes) {
            *out = c.p + h->cur_off;
            h->cur_off += bytes;
            return RS_OK;
        }
        h->cur_chunk++;
        h->cur_off = 0;
    }
    const size_t min_chunk = (size_t)64 << 20;
    const size_t want = bytes > min_chunk ? bytes : min_chunk;
    void *p = nullptr;
    size_t got = 0;
    RS_TRY(rs_cached_malloc(h->device, &p, want, &got));
    h->chunks.push_back({(char *)p, got});
    h->cur_chunk = h->chunks.size() - 1;
    h->cur_off = bytes;
    *out = p;
    return RS_OK;
}

namespace {

constexpr int T = 256;
inline unsigned blocks_for(int64_t n, int t = T) { return (unsigned)((n + t - 1) / t); }

// (the per-row counts are NOT taken here: 40 M atomic increments were the largest kernel of the ML-20M prep,
// 1.0 ms; the row pointers come out of the sorted key sequences instead, ptr_from_sorted_kernel)
__global__ void iota_validate_kernel(const int32_t *__restrict__ left, const int32_t *__restrict__ right,
                                     const double *__restrict__ rating, int64_t nnz, int32_t n_left,
                                     int32_t n_right, int32_t *__restrict__ idx, int32_t *__restrict__ flags) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nnz) return;
    idx[i] = (int32_t)i;
    int32_t l = left[i], r = right[i];
    int f = 0;
    if (l < 0 || l >= n_left || r < 0 || r >= n_right) f |= FLAG_BAD_ID;
    double v = rating[i];
    if (v != v) f |= FLAG_NAN;
    if (!(v == rint(v) && fabs(v) <= 11.0)) f |= FLAG_NOT_INT8;
    if (f) atomicOr(flags, f);
}

}  // namespace

// CSR row pointers from the ascending key sequence of a sort: ptr[k] = first position whose key is >= k
// (k = 0 .. n_rows; empty rows included).  The entry that opens a new key closes every pointer in between.
__global__ void ptr_from_sorted_kernel(const int32_t *__restrict__ keys, int64_t nnz, int32_t n_rows,
                                       int64_t *__restrict__ ptr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > nnz) return;
    const int32_t cur = i < nnz ? keys[i] : n_rows;           // sentinel after the last entry
    const int32_t prev = i > 0 ? keys[i - 1] : -1;
    for (int32_t k = prev + 1; k <= cur; k++) ptr[k] = i;
}

__global__ void gather_keys_kernel(const int32_t *__restrict__ src, const int32_t *__restrict__ perm, int64_t n,
                                   int32_t *__restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = src[perm[i]];
}

// entries of the (major, minor)-sorted permutation -> CSR column / value arrays
__global__ void gather_csr_kernel(const int32_t *__restrict__ perm, const int32_t *__restrict__ minor,
                                  const double *__restrict__ rating, int64_t nnz, int32_t *__restrict__ col,
                                  double *__restrict__ val) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nnz) return;
    int32_t p = perm[i];
    col[i] = minor[p];
    val[i] = rating[p];
}

// duplicate (left, right) pairs are adjacent in a CSR: `row` = the sorted major keys the last sort left behind,
// `col` = the gathered minor ids (both read coalesced; the check used to re-gather three ids per entry)
__global__ void dup_check_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col, int64_t nnz,
                                 int32_t *__restrict__ flags) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0 || i >= nnz) return;
    if (row[i] == row[i - 1] && col[i] == col[i - 1]) atomicOr(flags, FLAG_DUP);
}

namespace {

__global__ void gather_val_kernel(const int32_t *__restrict__ perm, const double *__restrict__ rating, int64_t nnz,
                                  double *__restrict__ val) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) val[i] = rating[perm[i]];
}

__global__ void code_int8_kernel(const double *__restrict__ val, int64_t nnz, uint8_t *__restrict__ code) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) code[i] = (uint8_t)((int)val[i] + RS_INT8_BIAS);
}

__global__ void row_isum_kernel(const int64_t *__restrict__ l_ptr, const uint8_t *__restrict__ l_code,
                                int32_t n_left, int32_t *__restrict__ row_cnt, int32_t *__restrict__ row_sum) {
    int32_t row = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    int lane = threadIdx.x & 31;
    if (row >= n_left) return;
    int s = 0;
    for (int64_t x = l_ptr[row] + lane; x < l_ptr[row + 1]; x += 32) s += (int)l_code[x] - RS_INT8_BIAS;
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
        row_cnt[row] = (int32_t)(l_ptr[row + 1] - l_ptr[row]);
        row_sum[row] = s;
    }
}

// Row statistics in the reference's order.  One warp per left row: the lanes load 32 entries
// at a time (coalesced) and the additions are then applied one after the other through
// shuffles, so every sum sees exactly the reference's sequence of IEEE additions:
//   means   core/data.go:226-232   (dataset order)
//   stddevs core/knn.go:170-175    (dataset order)
//   pmeans  core/sim.go:49-54      (ascending id order, the row after `sorts`)
__device__ __forceinline__ double ordered_sum(const double *__restrict__ v, int64_t b, int64_t e, int lane,
                                              double mean, bool squared_dev) {
    double sum = 0.0;
    for (int64_t base = b; base < e; base += 32) {
        double x = (base + lane < e) ? v[base + lane] : 0.0;
        if (squared_dev) x = (x - mean) * (x - mean);
        const int lim = (e - base) < 32 ? (int)(e - base) : 32;
        for (int q = 0; q < lim; q++) sum += __shfl_sync(0xffffffffu, x, q);
    }
    return sum;
}

__global__ void row_stats_ordered_kernel(const int64_t *__restrict__ l_ptr, const double *__restrict__ ld_val,
                                         const double *__restrict__ l_val, int32_t n_left, int want_mean,
                                         int want_std, double *__restrict__ means, double *__restrict__ stddevs,
                                         double *__restrict__ pmeans) {
    const int32_t i = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n_left) return;
    const int64_t b = l_ptr[i], e = l_ptr[i + 1];
    const double count = (double)(e - b);
    double mean = means[i];
    if (want_mean) {
        mean = ordered_sum(ld_val, b, e, lane, 0.0, false) / count;
        const double pm = ordered_sum(l_val, b, e, lane, 0.0, false) / count;
        if (lane == 0) { means[i] = mean; pmeans[i] = pm; }
    }
    if (want_std) {
        const double s2 = ordered_sum(ld_val, b, e, lane, mean, true);
        if (lane == 0) stddevs[i] = sqrt(s2 / count) + 1e-5;
    }
}

// Integer ratings: every partial sum is an exact integer < 2^53, so sum/count is the same
// double in any order — computed from the exact integer row sum.
__global__ void means_from_isum_kernel(const int32_t *__restrict__ row_cnt, const int32_t *__restrict__ row_sum,
                                       int32_t n_left, double *__restrict__ means, double *__restrict__ pmeans) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_left) return;
    const double m = (double)row_sum[i] / (double)row_cnt[i];
    means[i] = m;
    pmeans[i] = m;
}

// b-side term of every right-CSR entry (c, j): the value the reference combines with the a-side
// term, computed once with the same IEEE operations (core/sim.go:74 `ratingB := jr.Rating - meanB`).
__global__ void build_rdev_kernel(const int64_t *__restrict__ r_ptr, const int32_t *__restrict__ r_col,
                                  const double *__restrict__ r_val, int32_t n_right, int sim,
                                  const double *__restrict__ pmeans, const double *__restrict__ left_bias,
                                  const double *__restrict__ right_bias, double global_bias,
                                  double *__restrict__ r_dev) {
    const int32_t c = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (c >= n_right) return;
    for (int64_t x = r_ptr[c] + lane; x < r_ptr[c + 1]; x += 32) {
        const int32_t j = r_col[x];
        const double y = r_val[x];
        double t;
        if (sim == RS_SIM_PEARSON) t = y - pmeans[j];
        else if (sim == RS_SIM_PEARSON_BASELINE) { const double base = global_bias + left_bias[j]; const double bb = base + right_bias[c]; t = y - bb; }
        else t = y;
        r_dev[x] = t;
    }
}

__global__ void row_len_kernel(const int64_t *__restrict__ l_ptr, int32_t n_left, int32_t *__restrict__ len,
                               int32_t *__restrict__ ids) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_left) return;
    len[i] = (int32_t)(l_ptr[i + 1] - l_ptr[i]);
    ids[i] = i;
}

// cp[c][q] = number of entries of right row c with left id < (q0 + q) * jc, for q = 0 .. n_q (the chunk
// boundaries inside every right row).  One warp per right row walks the row once: an entry whose chunk
// differs from its predecessor's closes the boundaries in between (no binary searches: 14.6 M of them, 7
// dependent loads each, were the largest kernel of the ML-20M prep).
__global__ void build_cp_kernel(const int64_t *__restrict__ r_ptr, const int32_t *__restrict__ r_col,
                                int32_t n_right, int32_t q0, int32_t n_q, int32_t jc, int32_t *__restrict__ cp) {
    const int32_t c = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (c >= n_right) return;
    const int64_t b = r_ptr[c], e = r_ptr[c + 1];
    int32_t *out = cp + (int64_t)c * (n_q + 1);
    // boundary q is closed by the first entry whose chunk index (relative to q0, clamped) is >= q
    auto rel = [&](int32_t col) {
        const int32_t q = col / jc - q0;
        return q < 0 ? -1 : (q >= n_q ? n_q : q);            // -1: before the window, n_q: beyond it
    };
    for (int64_t x0 = b; x0 <= e; x0 += 32) {                 // x == e is the sentinel that closes the tail
        const int64_t x = x0 + lane;
        if (x > e) continue;
        const int32_t cur = x < e ? rel(r_col[x]) : n_q;      // sentinel after the last entry
        const int32_t prev = x > b ? rel(r_col[x - 1]) : -1;
        for (int32_t q = prev + 1; q <= cur; q++) out[q] = (int32_t)(x - b);
    }
}

// l2r[e] for the left-CSR entry e = (i, c): position of (c, i) in the right CSR.  Both CSRs are
// permutations of the input rows (perm_lr[e] / perm_rl[x] = original row index), so
// l2r = inverse(perm_rl) o perm_lr: one scatter and one gather, no search.
__global__ void invert_perm_kernel(const int32_t *__restrict__ perm, int64_t n, int32_t *__restrict__ inv) {
    const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (x < n) inv[perm[x]] = (int32_t)x;
}
__global__ void compose_l2r_kernel(const int32_t *__restrict__ perm_lr, const int32_t *__restrict__ inv_rl, int64_t n,
                                   int64_t *__restrict__ l2r) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n) l2r[e] = inv_rl[perm_lr[e]];
}

// ---- popular columns (sim_stream.cu: sim_pop_kernel) ----
// n_pop = rows of at least min_len entries (len_sorted is descending), at most cap
__global__ void pop_count_kernel(const int32_t *__restrict__ len_sorted, int32_t n, int64_t min_len, int32_t cap,
                                 int32_t *__restrict__ out) {
    int32_t lo = 0, hi = n;                                   // first position whose length is < min_len
    while (lo < hi) {
        const int32_t mid = (lo + hi) >> 1;
        if ((int64_t)len_sorted[mid] >= min_len) lo = mid + 1; else hi = mid;
    }
    *out = lo < cap ? lo : cap;
}
// pop_items = the popular list, -1 beyond it
__global__ void pop_items_kernel(const int32_t *__restrict__ sorted, int32_t n_pop, int32_t pop_ld,
                                 int32_t *__restrict__ pop_items) {
    const int32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < pop_ld) pop_items[p] = p < n_pop ? sorted[p] : -1;
}
// One warp per right row: its popular ratings go into the dense table (preset to "no rating").
template <typename DT>
__global__ void pop_scatter_kernel(const int64_t *__restrict__ r_ptr, const int32_t *__restrict__ r_col,
                                   const double *__restrict__ r_val, const double *__restrict__ r_dev,
                                   int32_t n_right, const int32_t *__restrict__ rank, int32_t n_pop, int32_t pop_ld,
                                   DT *__restrict__ dense) {
    const int32_t c = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (c >= n_right) return;
    for (int64_t x = r_ptr[c] + lane; x < r_ptr[c + 1]; x += 32) {
        const int32_t p = rank[r_col[x]];
        if (p >= n_pop) continue;
        if (sizeof(DT) == 1) dense[(int64_t)c * pop_ld + p] = (DT)((int)r_val[x] + RS_INT8_BIAS);            // the byte code of code_int8_kernel
        else dense[(int64_t)c * pop_ld + p] = (DT)r_dev[x];
    }
}
// The walk CSR is the transpose of the walked rows taken in label order: one warp per rank lays out the entries of
// the walked rows as (right id, left-CSR entry) pairs at the row's offset in label order (w_off), and notes the
// entry's label; a stable sort by right id then leaves every right row's entries in ascending label.  The entries
// of the popular rows are never walked: l2r = -1.
__global__ void walk_seq_kernel(const int32_t *__restrict__ sorted, int32_t n_left, int32_t n_pop,
                                const int64_t *__restrict__ l_ptr, const int32_t *__restrict__ l_col,
                                const int64_t *__restrict__ w_off, int32_t *__restrict__ key, int32_t *__restrict__ ent,
                                int32_t *__restrict__ ent_lab, int64_t *__restrict__ l2r) {
    const int32_t p = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= n_left) return;
    const int32_t i = sorted[p];
    const int64_t b = l_ptr[i], e = l_ptr[i + 1];
    if (p < n_pop) {
        for (int64_t x = b + lane; x < e; x += 32) l2r[x] = -1;
        return;
    }
    const int32_t lab = p - n_pop;
    const int64_t o = w_off[lab] - b;
#pragma unroll 4
    for (int64_t x = b + lane; x < e; x += 32) {
        key[o + x] = l_col[x];
        ent[o + x] = (int32_t)x;
        ent_lab[x] = lab;
    }
}
// walk CSR position o <- left-CSR entry x = ent[o]: its label, its b-side term, and l2r[x] = o
__global__ void walk_gather_kernel(const int32_t *__restrict__ ent, const int32_t *__restrict__ ent_lab,
                                   const double *__restrict__ r_dev, int64_t n, int32_t *__restrict__ w_col,
                                   double *__restrict__ w_dev, int64_t *__restrict__ l2r) {
    const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n) return;
    const int32_t x = ent[o];
    w_col[o] = ent_lab[x];
    w_dev[o] = r_dev[l2r[x]];
    l2r[x] = o;
}
struct PopLight {
    const int32_t *rank;
    int32_t n_pop;
    __host__ __device__ bool operator()(const int32_t &i) const { return rank[i] >= n_pop; }
};


// planes[p][col / kblk][row][col % kblk]: p=0 rating^2, p=1 mask, p=2 rating (the order the MMAs of
// sim_tensor.cu rely on: B planes adjacent in shared memory as X2 | M | X); int8, K-blocked so that
// the TMA box of one (plane, K block, row range) is one contiguous run of bytes
__global__ void scatter_planes_kernel(const int64_t *__restrict__ l_ptr, const int32_t *__restrict__ l_col,
                                      const uint8_t *__restrict__ l_code, int32_t n_left, int64_t npad,
                                      int64_t kpad, int32_t kblk, int8_t *__restrict__ planes) {
    int32_t row = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    int lane = threadIdx.x & 31;
    if (row >= n_left) return;
    int64_t plane = npad * kpad;
    for (int64_t x = l_ptr[row] + lane; x < l_ptr[row + 1]; x += 32) {
        int v = (int)l_code[x] - RS_INT8_BIAS;
        const int32_t col = l_col[x];
        int64_t o = ((int64_t)(col / kblk) * npad + row) * kblk + (col % kblk);
        planes[o] = (int8_t)(v * v);
        planes[plane + o] = 1;
        planes[2 * plane + o] = (int8_t)v;
    }
}

struct CycOwned {
    int count, index;
    __host__ __device__ bool operator()(const int32_t &i) const { return rs_cyc_owns(i, count, index); }
};

struct SortTmp {
    void *p = nullptr;
    size_t bytes = 0;
};

int bits_for(int32_t n) {
    int b = 1;
    while ((1ll << b) < (long long)n) b++;
    return b;
}

}  // namespace

// The statistics of every left row from the left CSR, into the buffers h points to: means, stddevs (z-score) and
// pmeans, and for integer ratings row_cnt / row_sum.  Fit's, and rs_knn_update's for the merged rows.
int32_t rs_prep_stats(rs_knn *h) {
    cudaStream_t st = h->stream;
    const int32_t nl = h->n_left;
    const int want_std = h->p.knn_type == RS_KNN_ZSCORE;
    if (h->rating_class == RS_CLASS_INT8) {
        row_isum_kernel<<<blocks_for((int64_t)nl * 32), T, 0, st>>>(h->l_ptr, h->l_code, nl, h->row_cnt, h->row_sum);
        means_from_isum_kernel<<<blocks_for(nl), T, 0, st>>>(h->row_cnt, h->row_sum, nl, h->means, h->pmeans);
        h->prof.total_launches += 2;
    }
    if (h->rating_class != RS_CLASS_INT8 || want_std) {
        row_stats_ordered_kernel<<<blocks_for((int64_t)nl * 32), T, 0, st>>>(
            h->l_ptr, h->ld_val, h->l_val, nl, h->rating_class != RS_CLASS_INT8, want_std, h->means, h->stddevs,
            h->pmeans);
        h->prof.total_launches++;
    }
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

// Row statistics of `n` rows given as a CSR: the entries of row i are ptr[i] .. ptr[i+1) of ld_val (dataset order:
// means, stddevs) and of l_val (ascending id: pmeans).  Fit's statistics, for the rating lists of rs_knn_*_given.
int32_t rs_row_stats_launch(rs_knn *h, const int64_t *ptr, const double *ld_val, const double *l_val, int64_t n,
                            int want_std, double *means, double *stddevs, double *pmeans) {
    if (n <= 0) return RS_OK;
    row_stats_ordered_kernel<<<blocks_for(n * 32), T, 0, h->stream>>>(ptr, ld_val, l_val, (int32_t)n, 1, want_std,
                                                                      means, stddevs, pmeans);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

#define RS_SORT_PAIRS(keys_in, keys_out, vals_in, vals_out, n, end_bit)                                      \
    do {                                                                                                     \
        size_t need_ = 0;                                                                                    \
        RS_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, need_, keys_in, keys_out, vals_in, vals_out, (int)(n), \
                                                0, end_bit, st));                                            \
        if (need_ > tmp.bytes) {                                                                             \
            RS_TRY(rs_dev_alloc(h, &tmp.p, need_));                                                          \
            tmp.bytes = need_;                                                                               \
        }                                                                                                    \
        RS_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp.bytes, keys_in, keys_out, vals_in, vals_out,      \
                                                (int)(n), 0, end_bit, st));                                  \
    } while (0)

// sum over right rows of cnt*(cnt-1)/2 = co-rated triples (i < j, common right id): the work of the
// stream path, used by the Fit path model (api.cu)
__global__ void triples_kernel(const int64_t *__restrict__ r_ptr, int32_t nr, unsigned long long *out,
                               int32_t *max_len) {
    unsigned long long acc = 0;
    int32_t mx = 0;
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < nr; c += (int64_t)gridDim.x * blockDim.x) {
        const int32_t cnt = (int32_t)(r_ptr[c + 1] - r_ptr[c]);
        const unsigned long long n = (unsigned long long)cnt;
        acc += n * (n - (n ? 1 : 0)) / 2;
        mx = cnt > mx ? cnt : mx;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const int32_t v = __shfl_xor_sync(0xffffffffu, mx, o); mx = v > mx ? v : mx; }
    if ((threadIdx.x & 31) == 0 && mx) atomicMax(max_len, mx);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

// (entry, chunk) lookups the stream kernel performs when it computes the upper (j > i) or the lower
// (j < i) triangle: row i pays one lookup per entry and per column chunk it visits.  Row i's length is
// len[i], or taken from l_ptr when len is null.
__global__ void incidence_kernel(const int64_t *__restrict__ l_ptr, const int32_t *__restrict__ len, int32_t nl,
                                 int32_t jc, unsigned long long *out) {
    unsigned long long up = 0, lo = 0;
    const long long q_all = (nl + jc - 1) / jc;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nl; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long d = (unsigned long long)(len ? (int64_t)len[i] : l_ptr[i + 1] - l_ptr[i]);
        const long long q = i / jc;
        up += d * (unsigned long long)(q_all - q);
        lo += d * (unsigned long long)(q + 1);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        up += __shfl_xor_sync(0xffffffffu, up, o);
        lo += __shfl_xor_sync(0xffffffffu, lo, o);
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(out, up); atomicAdd(out + 1, lo); }
}

// Slope One: mean of every right row (user).  Integer ratings: the sum is exact in any order, so
// one correctly rounded division reproduces core/data.go:222-235 whatever the order.
__global__ void right_means_kernel(const int64_t *__restrict__ r_ptr, const double *__restrict__ r_val, int32_t nr,
                                   double *__restrict__ out) {
    const int32_t c = (int32_t)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (c >= nr) return;
    double s = 0.0;
    for (int64_t x = r_ptr[c] + lane; x < r_ptr[c + 1]; x += 32) s += r_val[x];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[c] = s / (double)(r_ptr[c + 1] - r_ptr[c]);
}

// the cheaper triangle by the lookup counts inc_upper / inc_lower
static void pick_triangle(rs_knn *h) {
    h->stream_lower = h->inc_lower < h->inc_upper;
    if (const char *e = getenv("RS_KNN_STREAM_TRI")) h->stream_lower = !strcmp(e, "lower");   // tests: force a triangle
}

static int32_t rs_stream_jc(int32_t n_left) {
    int32_t jc = n_left < 8192 ? 128 : 256;
    // the stream kernel is instantiated for 128 and 256 columns only (launch_stream_sym): anything else takes 256
    if (const char *e = getenv("RS_KNN_STREAM_JC")) jc = atoi(e) == 128 ? 128 : 256;
    return jc;
}

int32_t rs_prep_build(rs_knn *h, const int32_t *d_left, const int32_t *d_right, const double *d_rating,
                      const double *d_left_bias, const double *d_right_bias) {
    cudaStream_t st = h->stream;
    const int64_t nnz = h->nnz;
    const int32_t nl = h->n_left, nr = h->n_right;
    if (nnz >= (1ll << 31)) {
        rs_set_error("nnz %lld exceeds the 2^31-1 entries supported", (long long)nnz);
        return RS_ERR_UNSUPPORTED;
    }
    SortTmp tmp;
    int32_t *idx, *keys_a, *keys_b, *perm_l, *perm_r, *perm_lr, *perm_rl;
    RS_TRY(rs_alloc(h, &idx, nnz));
    RS_TRY(rs_alloc(h, &keys_a, nnz));
    RS_TRY(rs_alloc(h, &keys_b, nnz));
    RS_TRY(rs_alloc(h, &perm_l, nnz));
    RS_TRY(rs_alloc(h, &perm_r, nnz));
    RS_TRY(rs_alloc(h, &perm_lr, nnz));
    RS_TRY(rs_alloc(h, &perm_rl, nnz));
    RS_TRY(rs_alloc(h, &h->d_flags, 16));
    RS_TRY(rs_alloc(h, &h->l_ptr, (size_t)nl + 1));
    RS_TRY(rs_alloc(h, &h->r_ptr, (size_t)nr + 1));
    RS_CUDA(cudaMemsetAsync(h->d_flags, 0, 64, st));

    iota_validate_kernel<<<blocks_for(nnz), T, 0, st>>>(d_left, d_right, d_rating, nnz, nl, nr, idx, h->d_flags);
    h->stream_jc = rs_stream_jc(nl);
    h->prof.total_launches += 1;
    int32_t flags = 0;
    RS_CUDA(cudaMemcpyAsync(&flags, h->d_flags, 4, cudaMemcpyDeviceToHost, st));
    RS_CUDA(cudaStreamSynchronize(st));
    if (flags & FLAG_BAD_ID) {
        rs_set_error("rating rows contain inner ids outside [0,n_left) x [0,n_right)");
        return RS_ERR_INVALID;
    }
    if (flags & FLAG_NAN) {
        rs_set_error("NaN ratings are not supported");
        return RS_ERR_UNSUPPORTED;
    }
    h->rating_class = (flags & FLAG_NOT_INT8) ? RS_CLASS_TABLE : RS_CLASS_INT8;

    const int lb = bits_for(nl), rb = bits_for(nr);
    // stable LSD sorts: perm_l = by left (dataset order inside a row) — only needed when row
    // statistics must be summed in dataset order (non-integer ratings, or z-score's stddevs; integer
    // means are exact in any order) —, perm_r = by right
    const bool need_dataset_order = h->rating_class != RS_CLASS_INT8 || h->p.knn_type == RS_KNN_ZSCORE;
    if (need_dataset_order) RS_SORT_PAIRS(d_left, keys_a, idx, perm_l, nnz, lb);
    RS_SORT_PAIRS(d_right, keys_a, idx, perm_r, nnz, rb);
    // keys_a = the right ids in ascending order: the right CSR's row pointers, and from them the co-rated
    // triples and the longest right row (read back with the duplicate flag at the end)
    ptr_from_sorted_kernel<<<blocks_for(nnz + 1), T, 0, st>>>(keys_a, nnz, nr, h->r_ptr);
    triples_kernel<<<148, T, 0, st>>>(h->r_ptr, nr, reinterpret_cast<unsigned long long *>(h->d_flags + 6), h->d_flags + 15);
    // (left, right asc): stable sort by left of the right-sorted sequence
    gather_keys_kernel<<<blocks_for(nnz), T, 0, st>>>(d_left, perm_r, nnz, keys_a);
    RS_SORT_PAIRS(keys_a, keys_b, perm_r, perm_lr, nnz, lb);
    // keys_b = the left ids in ascending order: the left CSR's row pointers, and the (entry, chunk) lookups of
    // the two triangles of a stream Fit
    ptr_from_sorted_kernel<<<blocks_for(nnz + 1), T, 0, st>>>(keys_b, nnz, nl, h->l_ptr);
    incidence_kernel<<<148, T, 0, st>>>(h->l_ptr, nullptr, nl, h->stream_jc, reinterpret_cast<unsigned long long *>(h->d_flags + 8));
    h->prof.total_launches += 4;
    // (right, left asc): stable sort by right of the (left, right asc) sequence
    gather_keys_kernel<<<blocks_for(nnz), T, 0, st>>>(d_right, perm_lr, nnz, keys_a);
    RS_SORT_PAIRS(keys_a, keys_b, perm_lr, perm_rl, nnz, rb);
    h->prof.total_launches += 2;  // own kernels only; CUB's sort/scan kernels are not counted
    if (h->p.sim == RS_SIM_SLOPE_ONE) {
        // SlopeOne.Predict sums dev[item][.] over the user's ratings in DATASET order
        // (core/slope_one.go:35-38): perm_r is the stable sort by right id of the input rows
        RS_TRY(rs_alloc(h, &h->rd_col, nnz));
        gather_keys_kernel<<<blocks_for(nnz), T, 0, st>>>(d_left, perm_r, nnz, h->rd_col);
        h->prof.total_launches++;
    }
    h->perm_lr = perm_lr;         // kept for the stream tables (rs_prep_rt); keys_b is free from here on
    h->perm_rl = perm_rl;
    h->perm_tmp = keys_b;

    RS_TRY(rs_alloc(h, &h->l_col, nnz));
    RS_TRY(rs_alloc(h, &h->l_val, nnz));
    RS_TRY(rs_alloc(h, &h->ld_val, nnz));
    RS_TRY(rs_alloc(h, &h->r_col, nnz));
    RS_TRY(rs_alloc(h, &h->r_val, nnz));
    gather_csr_kernel<<<blocks_for(nnz), T, 0, st>>>(perm_lr, d_right, d_rating, nnz, h->l_col, h->l_val);
    gather_csr_kernel<<<blocks_for(nnz), T, 0, st>>>(perm_rl, d_left, d_rating, nnz, h->r_col, h->r_val);
    dup_check_kernel<<<blocks_for(nnz), T, 0, st>>>(keys_b, h->r_col, nnz, h->d_flags);   // keys_b: the right ids, sorted
    if (need_dataset_order) gather_val_kernel<<<blocks_for(nnz), T, 0, st>>>(perm_l, d_rating, nnz, h->ld_val);
    h->prof.total_launches += need_dataset_order ? 4 : 3;

    // byte codes (rating + 12) of the integer class: operands of the tensor path and of the exact
    // integer row sums.  Any other float64 rating set runs on the stream path, which reads the
    // values themselves (l_val / r_dev) — no code table, no limit on the number of distinct values.
    if (h->rating_class == RS_CLASS_INT8) {
        RS_TRY(rs_alloc(h, &h->l_code, nnz));
        code_int8_kernel<<<blocks_for(nnz), T, 0, st>>>(h->l_val, nnz, h->l_code);
        h->prof.total_launches += 1;
    }

    // row statistics
    RS_TRY(rs_alloc(h, &h->means, (size_t)nl + 1));
    RS_TRY(rs_alloc(h, &h->stddevs, (size_t)nl + 1));
    RS_TRY(rs_alloc(h, &h->pmeans, (size_t)nl + 1));
    if (h->rating_class == RS_CLASS_INT8) {
        RS_TRY(rs_alloc(h, &h->row_cnt, (size_t)nl + 1));
        RS_TRY(rs_alloc(h, &h->row_sum, (size_t)nl + 1));
    }
    RS_TRY(rs_prep_stats(h));

    if (h->p.sim == RS_SIM_SLOPE_ONE) {
        RS_TRY(rs_alloc(h, &h->right_means, (size_t)nr + 1));
        right_means_kernel<<<blocks_for((int64_t)nr * 32), T, 0, st>>>(h->r_ptr, h->r_val, nr, h->right_means);
        h->prof.total_launches++;
    }
    if (d_left_bias) {
        RS_TRY(rs_alloc(h, &h->left_bias, (size_t)nl + 1));
        RS_CUDA(cudaMemcpyAsync(h->left_bias, d_left_bias, (size_t)nl * 8, cudaMemcpyDeviceToDevice, st));
    }
    if (d_right_bias) {
        RS_TRY(rs_alloc(h, &h->right_bias, (size_t)nr + 1));
        RS_CUDA(cudaMemcpyAsync(h->right_bias, d_right_bias, (size_t)nr * 8, cudaMemcpyDeviceToDevice, st));
    }

    int32_t fl8[16] = {0};
    RS_CUDA(cudaMemcpyAsync(fl8, h->d_flags, 64, cudaMemcpyDeviceToHost, st));
    RS_CUDA(cudaStreamSynchronize(st));
    flags = fl8[0];
    { unsigned long long t; memcpy(&t, fl8 + 6, 8); h->triples = (double)t; }
    h->max_right_len = fl8[15];
    { unsigned long long t[2]; memcpy(t, fl8 + 8, 16); h->inc_upper = (double)t[0]; h->inc_lower = (double)t[1]; }
    pick_triangle(h);
    if (flags & FLAG_DUP) {
        rs_set_error("duplicate (left,right) rating pairs are not supported (the reference's merge-join "
                     "double-counts them)");
        return RS_ERR_DUPLICATE;
    }
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

// Heavy rows (sim_stream.cu: sim_stream_heavy_kernel): rows of >= min_len entries are split off the
// longest-first order and processed by producer / consumer CTAs.  `order`: the rows to process, longest
// first.  Writes h->row_order (the other rows, same order), h->row_heavy and the counts.
struct HeavyPred {
    const int64_t *l_ptr;
    int64_t min_len;
    bool negate;
    __host__ __device__ bool operator()(const int32_t &i) const { return ((l_ptr[i + 1] - l_ptr[i]) >= min_len) != negate; }
};

static int32_t split_heavy_rows(rs_knn *h, int32_t *order, int64_t n_rows, bool allow) {
    cudaStream_t st = h->stream;
    // On ONE GPU the serial walk of a blockbuster row hides under the other rows' work; under cyclic sharding the
    // per-GPU work shrinks and that walk becomes the critical path (profiles/r02_stream_notes.md).
    int64_t min_len = h->cyc_R > 1 ? 8192 : -1;
    if (const char *e = getenv("RS_KNN_HEAVY_MIN")) min_len = atoll(e);      // tests: 0 = every row
    h->n_heavy = 0;
    h->row_heavy = nullptr;
    h->row_order = order;
    h->n_work_rows = n_rows;
    if (n_rows <= 0 || !allow || min_len < 0 || h->stream_jc != 256) return RS_OK;
    int32_t *rest, *d_num;
    RS_TRY(rs_alloc(h, &h->row_heavy, (size_t)n_rows));
    RS_TRY(rs_alloc(h, &rest, (size_t)n_rows));
    RS_TRY(rs_alloc(h, &d_num, 4));
    HeavyPred yes{h->l_ptr, min_len, false}, no{h->l_ptr, min_len, true};
    size_t need = 0;
    RS_CUDA(cub::DeviceSelect::If(nullptr, need, order, h->row_heavy, d_num, (int)n_rows, yes, st));
    void *tmp;
    RS_TRY(rs_dev_alloc(h, &tmp, need + 256));
    RS_CUDA(cub::DeviceSelect::If(tmp, need, order, h->row_heavy, d_num, (int)n_rows, yes, st));
    RS_CUDA(cub::DeviceSelect::If(tmp, need, order, rest, d_num + 1, (int)n_rows, no, st));
    int32_t cnt = 0;
    RS_CUDA(cudaMemcpyAsync(&cnt, d_num, 4, cudaMemcpyDeviceToHost, st));
    RS_CUDA(cudaStreamSynchronize(st));
    h->n_heavy = cnt;
    h->row_order = rest;
    h->n_work_rows = n_rows - cnt;
    return RS_OK;
}

// Popular columns: the rows of >= min_len entries (at most RS_POP_MAX, the longest).  `sorted`: ALL rows, longest
// first (stable: ties by id), so a row's position in it is its rank; `len_sorted`: their lengths; `order` / n_rows:
// the rows of this shard, longest first.  Splits the popular rows' ratings off the right CSR into the dense table,
// builds the walk CSR over the other rows' labels (see rs_knn::rank) and re-targets `l2r` to it, picks the triangle
// by the lookups in label space, and leaves the rows the column walk visits (the others, same order) in
// h->row_order.  `cp` is built by the caller over the labels.
constexpr int RS_POP_MAX = 512;

static int32_t split_popular(rs_knn *h, const int32_t *sorted, const int32_t *len_sorted, int32_t *order, int64_t n_rows,
                             int64_t min_len) {
    cudaStream_t st = h->stream;
    int32_t *d_num;
    RS_TRY(rs_alloc(h, &d_num, 4));
    int32_t cap = RS_POP_MAX;
    if (const char *e = getenv("RS_KNN_POP_MAX")) { cap = atoi(e); cap = cap < 2 ? 2 : (cap > 2048 ? 2048 : cap); }   // experiments
    pop_count_kernel<<<1, 1, 0, st>>>(len_sorted, h->n_left, min_len, cap, d_num);
    int32_t n_pop = 0;
    RS_CUDA(cudaMemcpyAsync(&n_pop, d_num, 4, cudaMemcpyDeviceToHost, st));
    RS_CUDA(cudaStreamSynchronize(st));
    h->prof.total_launches++;
    if (n_pop < 2) return RS_OK;                              // nothing to split off
    const int32_t nr = h->n_right, nl = h->n_left, n_walk = nl - n_pop;
    h->n_pop = n_pop;
    h->pop_ld = (n_pop + 31) / 32 * 32;
    h->pop_u8 = h->rating_class == RS_CLASS_INT8;
    h->lab_row = const_cast<int32_t *>(sorted) + n_pop;
    RS_TRY(rs_alloc(h, &h->rank, (size_t)nl));
    RS_TRY(rs_alloc(h, &h->pop_items, (size_t)h->pop_ld));
    invert_perm_kernel<<<blocks_for(nl), T, 0, st>>>(sorted, nl, h->rank);
    pop_items_kernel<<<blocks_for(h->pop_ld), T, 0, st>>>(sorted, n_pop, h->pop_ld, h->pop_items);
    // dense table
    const size_t cell = h->pop_u8 ? 1 : 8;
    RS_TRY(rs_dev_alloc(h, &h->pop_dense, (size_t)nr * h->pop_ld * cell));
    RS_CUDA(cudaMemsetAsync(h->pop_dense, h->pop_u8 ? 0 : 0xFF, (size_t)nr * h->pop_ld * cell, st));   // 0 / NaN = no rating
    if (h->pop_u8)
        pop_scatter_kernel<uint8_t><<<blocks_for((int64_t)nr * 32), T, 0, st>>>(
            h->r_ptr, h->r_col, h->r_val, h->r_dev, nr, h->rank, n_pop, h->pop_ld, static_cast<uint8_t *>(h->pop_dense));
    else
        pop_scatter_kernel<double><<<blocks_for((int64_t)nr * 32), T, 0, st>>>(
            h->r_ptr, h->r_col, h->r_val, h->r_dev, nr, h->rank, n_pop, h->pop_ld, static_cast<double *>(h->pop_dense));
    h->prof.total_launches += 3;
    // offsets of the walked rows in label order, and the (entry, chunk) lookups of both triangles over the labels
    int64_t *w_off;
    unsigned long long *d_inc;
    RS_TRY(rs_alloc(h, &w_off, (size_t)n_walk + 1));
    RS_TRY(rs_alloc(h, &d_inc, 2));
    RS_CUDA(cudaMemsetAsync(w_off, 0, 8, st));
    RS_CUDA(cudaMemsetAsync(d_inc, 0, 16, st));
    if (n_walk > 0) {
        size_t need = 0;
        RS_CUDA(cub::DeviceScan::InclusiveSum(nullptr, need, len_sorted + n_pop, w_off + 1, n_walk, st));
        void *tmp;
        RS_TRY(rs_dev_alloc(h, &tmp, need + 256));
        RS_CUDA(cub::DeviceScan::InclusiveSum(tmp, need, len_sorted + n_pop, w_off + 1, n_walk, st));
    }
    incidence_kernel<<<148, T, 0, st>>>(nullptr, len_sorted + n_pop, n_walk, h->stream_jc, d_inc);
    h->prof.total_launches++;
    // the rows the column walk visits: the shard's rows that are not popular
    h->row_all = order;
    h->n_all_rows = n_rows;
    int32_t *rest;
    RS_TRY(rs_alloc(h, &rest, (size_t)(n_rows > 0 ? n_rows : 1)));
    h->row_order = rest;
    int32_t cnt = 0;
    if (n_rows > 0) {
        PopLight light{h->rank, n_pop};
        size_t need2 = 0;
        RS_CUDA(cub::DeviceSelect::If(nullptr, need2, order, rest, d_num, (int)n_rows, light, st));
        void *tmp2;
        RS_TRY(rs_dev_alloc(h, &tmp2, need2 + 256));
        RS_CUDA(cub::DeviceSelect::If(tmp2, need2, order, rest, d_num, (int)n_rows, light, st));
        RS_CUDA(cudaMemcpyAsync(&cnt, d_num, 4, cudaMemcpyDeviceToHost, st));
    }
    int64_t nnz_w = 0;
    unsigned long long inc[2] = {0, 0};
    RS_CUDA(cudaMemcpyAsync(&nnz_w, w_off + n_walk, 8, cudaMemcpyDeviceToHost, st));
    RS_CUDA(cudaMemcpyAsync(inc, d_inc, 16, cudaMemcpyDeviceToHost, st));
    RS_CUDA(cudaStreamSynchronize(st));
    h->n_work_rows = cnt;
    h->inc_upper = (double)inc[0];
    h->inc_lower = (double)inc[1];
    pick_triangle(h);
    h->n_chunks = (int32_t)(((int64_t)n_walk + h->stream_jc - 1) / h->stream_jc);
    // walk CSR: the walked entries in label order, stably sorted by right id
    int32_t *key, *ent, *key_s, *ent_s, *ent_lab;
    RS_TRY(rs_alloc(h, &h->w_ptr, (size_t)nr + 1));
    RS_TRY(rs_alloc(h, &h->w_col, (size_t)nnz_w));
    RS_TRY(rs_alloc(h, &h->w_dev, (size_t)nnz_w));
    RS_TRY(rs_alloc(h, &key, (size_t)nnz_w));
    RS_TRY(rs_alloc(h, &ent, (size_t)nnz_w));
    RS_TRY(rs_alloc(h, &key_s, (size_t)nnz_w));
    RS_TRY(rs_alloc(h, &ent_s, (size_t)nnz_w));
    RS_TRY(rs_alloc(h, &ent_lab, (size_t)h->nnz));
    walk_seq_kernel<<<blocks_for((int64_t)nl * 32), T, 0, st>>>(sorted, nl, n_pop, h->l_ptr, h->l_col, w_off, key, ent,
                                                                ent_lab, h->l2r);
    h->prof.total_launches++;
    if (nnz_w > 0) {
        SortTmp tmp;
        RS_SORT_PAIRS(key, key_s, ent, ent_s, nnz_w, bits_for(nr));
        walk_gather_kernel<<<blocks_for(nnz_w), T, 0, st>>>(ent_s, ent_lab, h->r_dev, nnz_w, h->w_col, h->w_dev, h->l2r);
        h->prof.total_launches++;
    }
    ptr_from_sorted_kernel<<<blocks_for(nnz_w + 1), T, 0, st>>>(key_s, nnz_w, nr, h->w_ptr);
    h->prof.total_launches++;
    return RS_OK;
}

int32_t rs_prep_rt(rs_knn *h) {
    cudaStream_t st = h->stream;
    h->n_chunks = (int32_t)(((int64_t)h->n_left + h->stream_jc - 1) / h->stream_jc);
    h->n_pop = 0;
    RS_TRY(rs_alloc(h, &h->r_dev, (size_t)h->nnz));
    RS_TRY(rs_alloc(h, &h->l2r, (size_t)h->nnz));
    RS_TRY(rs_alloc(h, &h->cp, (size_t)h->n_right * ((size_t)h->n_chunks + 1)));
    build_rdev_kernel<<<blocks_for((int64_t)h->n_right * 32), T, 0, st>>>(
        h->r_ptr, h->r_col, h->r_val, h->n_right, h->p.sim, h->pmeans, h->left_bias, h->right_bias, h->global_bias,
        h->r_dev);
    invert_perm_kernel<<<blocks_for(h->nnz), T, 0, st>>>(h->perm_rl, h->nnz, h->perm_tmp);
    compose_l2r_kernel<<<blocks_for(h->nnz), T, 0, st>>>(h->perm_lr, h->perm_tmp, h->nnz, h->l2r);
    h->prof.total_launches += 4;
    // chunk pointers of the CSR the column walk reads: the right CSR, or the walk CSR once popular columns are split off
    auto build_cp = [&]() {
        build_cp_kernel<<<blocks_for((int64_t)h->n_right * 32), T, 0, st>>>(
            h->n_pop ? h->w_ptr : h->r_ptr, h->n_pop ? h->w_col : h->r_col, h->n_right, 0, h->n_chunks, h->stream_jc, h->cp);
    };
    // rows of the shard ordered longest first (a stable descending sort of the row lengths keeps the
    // order deterministic): the longest work items start first
    {
        const int64_t rb = h->row_begin, rows = h->row_end - h->row_begin;
        int32_t *len, *len_sorted, *ids, *sorted;
        RS_TRY(rs_alloc(h, &len, (size_t)h->n_left));
        RS_TRY(rs_alloc(h, &len_sorted, (size_t)h->n_left));
        RS_TRY(rs_alloc(h, &ids, (size_t)h->n_left));
        RS_TRY(rs_alloc(h, &sorted, (size_t)h->n_left));
        row_len_kernel<<<blocks_for(h->n_left), T, 0, st>>>(h->l_ptr, h->n_left, len, ids);
        h->prof.total_launches++;
        if (h->p.store == RS_STORE_TOPK) {
            // rows are produced slab by slab into a slab-sized buffer: keep the natural order
            h->row_order = ids;
            h->n_work_rows = -1;                 // the launcher takes [row_begin, row_end) of the natural order
            build_cp();
            RS_CUDA(cudaGetLastError());
            return RS_OK;
        }
        size_t need = 0;
        RS_CUDA(cub::DeviceRadixSort::SortPairsDescending(nullptr, need, len + rb, len_sorted + rb, ids + rb,
                                                          sorted, (int)rows, 0, 32, st));
        void *tmp;
        RS_TRY(rs_dev_alloc(h, &tmp, need));
        RS_CUDA(cub::DeviceRadixSort::SortPairsDescending(tmp, need, len + rb, len_sorted + rb, ids + rb,
                                                          sorted, (int)rows, 0, 32, st));
        // Full-matrix Fits (one GPU, or cyclic shards) compute one triangle and mirror the other: there the longest
        // rows can be taken out of the column walk.  RS_KNN_POP=0 keeps them in it (under cyclic sharding as
        // producer / consumer CTAs: split_heavy_rows); RS_KNN_HEAVY_MIN sets the length threshold (tests).
        const bool full = h->row_begin == 0 && h->row_end == h->n_left;
        int64_t min_len = 8192;
        if (const char *e = getenv("RS_KNN_HEAVY_MIN")) min_len = atoll(e);
        bool pop = full && min_len >= 0;
        if (const char *e = getenv("RS_KNN_POP")) pop = pop && atoi(e) != 0;
        int32_t *order = sorted;
        int64_t n_order = rows;
        if (h->cyc_R > 1) {
            // cyclic shards: the owned rows picked out of the longest-first order
            int32_t *owned, *d_num;
            RS_TRY(rs_alloc(h, &owned, (size_t)h->n_left));
            RS_TRY(rs_alloc(h, &d_num, 4));
            size_t need2 = 0;
            CycOwned pred{h->cyc_R, h->cyc_r};
            RS_CUDA(cub::DeviceSelect::If(nullptr, need2, sorted, owned, d_num, (int)h->n_left, pred, st));
            void *tmp2;
            RS_TRY(rs_dev_alloc(h, &tmp2, need2 + 256));
            RS_CUDA(cub::DeviceSelect::If(tmp2, need2, sorted, owned, d_num, (int)h->n_left, pred, st));
            order = owned;
            n_order = h->rows_local;
        }
        h->n_heavy = 0;
        h->row_heavy = nullptr;
        h->row_order = order;
        h->n_work_rows = n_order;
        if (pop) RS_TRY(split_popular(h, sorted, len_sorted, order, n_order, min_len));
        else RS_TRY(split_heavy_rows(h, order, n_order, full));
        build_cp();
    }
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

int32_t rs_prep_planes(rs_knn *h) {
    cudaStream_t st = h->stream;
    const int32_t kblk = RS_TC_KBLK;
    h->tc_npad = ((int64_t)h->n_left + RS_TC_BM - 1) / RS_TC_BM * RS_TC_BM;
    h->tc_kpad = ((int64_t)h->n_right + RS_TC_KBLK - 1) / RS_TC_KBLK * RS_TC_KBLK;
    size_t bytes = 3 * (size_t)h->tc_npad * (size_t)h->tc_kpad;
    if (h->updated) {
        // after rs_knn_update: a block of their own, reused while it is large enough, so that updates alternating with
        // rs_knn_cosums do not grow the arena.  The stream has drained since the block's last use (rs_knn_cosums ends
        // with a synchronisation).
        if (h->upd_planes_bytes < bytes) {
            rs_cached_free(h->device, h->upd_planes, h->upd_planes_bytes);
            h->upd_planes = nullptr;
            h->upd_planes_bytes = 0;
            RS_TRY(rs_cached_malloc(h->device, &h->upd_planes, bytes + bytes / 4 + 256, &h->upd_planes_bytes));
        }
        h->planes = static_cast<int8_t *>(h->upd_planes);
    } else {
        RS_TRY(rs_alloc(h, &h->planes, bytes));
    }
    RS_CUDA(cudaMemsetAsync(h->planes, 0, bytes, st));
    scatter_planes_kernel<<<blocks_for((int64_t)h->n_left * 32), T, 0, st>>>(h->l_ptr, h->l_col, h->l_code,
                                                                            h->n_left, h->tc_npad, h->tc_kpad,
                                                                            kblk, h->planes);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}
