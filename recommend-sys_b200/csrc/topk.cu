// topk.cu — neighbour lists: the k best entries of a row under (similarity desc, id asc).  rs_knn_topk on a matrix,
// the lists of an RS_STORE_TOPK Fit (rs_fit_lists) and the lists of top-N recommendation (recommend.cu) are all
// selected here, by one block per row over one shared-memory candidate buffer.
#include <cstdlib>

#include "common.cuh"
#include "select.cuh"

namespace {

// +-0 share one key: they tie and are ordered by id, as the reference's float comparison does.  The lists carry the
// sign of a zero in bit 31 of the id word, so that a list reports the exact similarity (-0.0 included) while the
// order stays that of (key, id).
constexpr uint32_t NEG0 = 0x80000000u;
__device__ __forceinline__ uint32_t neg0_bit(double s) {
    return (unsigned long long)__double_as_longlong(s) == 0x8000000000000000ull ? NEG0 : 0u;
}
__device__ __forceinline__ bool ent_before(uint64_t ka, uint32_t pa, uint64_t kb, uint32_t pb) {
    return rec_before(ka, pa & ~NEG0, kb, pb & ~NEG0);
}
__device__ __forceinline__ double ent_sim(uint64_t k, uint32_t p) { return (p & NEG0) ? -0.0 : rs_key_sim(k); }

constexpr int TOPK_THREADS = 256;
constexpr int TOPK_CAP = 2048;

__device__ void block_bitonic(uint64_t *keys, uint32_t *pos, int n_pad) {
    for (int size = 2; size <= n_pad; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int t = threadIdx.x; t < (n_pad >> 1); t += blockDim.x) {
                int lo = 2 * t - (t & (stride - 1));
                int hi = lo + stride;
                bool up = ((lo & size) == 0);
                uint64_t ka = keys[lo], kb = keys[hi];
                uint32_t pa = pos[lo], pb = pos[hi];
                bool swap = up ? ent_before(kb, pb, ka, pa) : ent_before(ka, pa, kb, pb);
                if (swap) { keys[lo] = kb; keys[hi] = ka; pos[lo] = pb; pos[hi] = pa; }
            }
        }
    }
    __syncthreads();
}

// The candidate buffer of one row: entries [0, have) of keys / pos, and once the row's list is full the k-th best
// (thr_key, thr_pos), which every further candidate must beat.
struct ListBuf {
    uint64_t keys[TOPK_CAP];
    uint32_t pos[TOPK_CAP];
    uint64_t thr_key;
    uint32_t thr_pos;
    int have;
};

__device__ __forceinline__ void list_put(ListBuf &b, int slot, int32_t id, double s) {
    b.keys[slot] = rs_sim_key(s);
    b.pos[slot] = (uint32_t)id | neg0_bit(s);
}

// Pad entries [have, n_pad) with the worst record and sort the first n_pad (a power of two) best first.
__device__ __forceinline__ void list_sort(ListBuf &b, int have, int n_pad) {
    for (int t = have + threadIdx.x; t < n_pad; t += blockDim.x) { b.keys[t] = 0; b.pos[t] = 0xffffffffu; }
    block_bitonic(b.keys, b.pos, n_pad);
}

// Seed: list `row` of idx / sim (k entries, best first, id -1 = empty: its entries are a prefix) becomes entries
// [0, have).  A FULL list gives the threshold right away (its last entry): almost every new candidate of a later
// slab is then rejected by one compare.  Returns have.
__device__ __forceinline__ int list_seed(ListBuf &b, int32_t k, int64_t row, const int32_t *idx, const double *sim) {
    int have = 0;
    for (int t0 = 0; t0 < k; t0 += blockDim.x) {
        const int t = t0 + threadIdx.x;
        const int32_t id = t < k ? idx[row * k + t] : -1;
        if (id >= 0) list_put(b, t, id, sim[row * k + t]);
        have += __syncthreads_count(id >= 0);
    }
    if (threadIdx.x == 0) {
        b.have = have;
        if (have == k) { b.thr_key = b.keys[k - 1]; b.thr_pos = b.pos[k - 1]; }
    }
    __syncthreads();
    return have;
}

// Scan: columns [lo, hi) of `row`, column j reported as id j + id_off, appended to the buffer (b.have set by the
// caller); have_thr = the list is full, so a candidate must beat the threshold.  When the buffer is within
// TOPK_THREADS of full it is sorted and cut to k, which raises the threshold.  Returns the entries held.
__device__ __forceinline__ int list_scan(ListBuf &b, const double *__restrict__ row, int32_t lo, int32_t hi,
                                         uint32_t id_off, int32_t k, bool have_thr) {
    for (int32_t base = lo; base < hi; base += TOPK_THREADS) {
        const int32_t j = base + threadIdx.x;
        bool take = false;
        uint64_t key = 0;
        uint32_t neg0 = 0;
        if (j < hi) {
            const double s = row[j];
            if (s == s) {
                key = rs_sim_key(s);
                take = !have_thr || ent_before(key, (uint32_t)j + id_off, b.thr_key, b.thr_pos);
                neg0 = neg0_bit(s);
            }
        }
        if (take) {
            int slot = atomicAdd(&b.have, 1);
            b.keys[slot] = key;
            b.pos[slot] = ((uint32_t)j + id_off) | neg0;
        }
        __syncthreads();
        // every thread must see the SAME count: read it, then a second barrier before anybody's next
        // atomicAdd can change it (otherwise a slow thread may take the branch below alone)
        const int have_now = b.have;
        __syncthreads();
        if (have_now > TOPK_CAP - TOPK_THREADS) {
            list_sort(b, have_now, TOPK_CAP);
            if (threadIdx.x == 0) {
                b.have = k;
                b.thr_key = b.keys[k - 1];
                b.thr_pos = b.pos[k - 1];
            }
            have_thr = true;
            __syncthreads();
        }
    }
    return b.have;
}

// Finish: sort the `have` entries and, with `write`, store the k best as list `row` of idx / sim (-1 / NaN past the
// end).
__device__ __forceinline__ void list_finish(ListBuf &b, int have, int32_t k, int64_t row, int32_t *__restrict__ idx,
                                            double *__restrict__ sim, bool write = true) {
    int n_pad = 32;
    while (n_pad < have) n_pad <<= 1;
    list_sort(b, have, n_pad);
    if (!write) return;
    for (int t = threadIdx.x; t < k; t += blockDim.x) {
        const int64_t o = row * k + t;
        if (t < have) { idx[o] = (int32_t)(b.pos[t] & ~NEG0); sim[o] = ent_sim(b.keys[t], b.pos[t]); }
        else { idx[o] = -1; sim[o] = __longlong_as_double(0x7ff8000000000001ll); }
    }
}

// Top k of each row of a row-major matrix (ld = row pitch, columns [0, n)).
__global__ void __launch_bounds__(TOPK_THREADS) topk_rows_kernel(const double *__restrict__ sims, int64_t ld_s,
                                                                 int32_t n, int32_t k, int32_t *__restrict__ idx,
                                                                 double *__restrict__ sim) {
    __shared__ ListBuf b;
    const int64_t r = blockIdx.x;
    if (threadIdx.x == 0) b.have = 0;
    __syncthreads();
    const int have = list_scan(b, sims + r * ld_s, 0, n, 0, k, false);
    list_finish(b, have, k, r, idx, sim);
}

// ---------------------------------------------------------------------------------------------
// Symmetric top-k slabs (RS_STORE_TOPK with shard_count >= 1).  A slab holds the rows
// [g0, g0+m) of the similarity matrix, of which only the entries right of the diagonal are used;
// each unordered pair {i, j} therefore feeds TWO neighbour lists: row i (through the slab) and row j
// (through the slab's transpose), and no pair is computed twice.
//   mode 0: src = slab,      block r <-> global row g0 + r, columns (g, n_cols), id = column
//   mode 1: src = transpose, block r <-> global row g0 + r, columns [0, min(m, r)), id = g0 + column
// The running list of the row (k entries, -1 = empty) is merged in: it seeds the candidate buffer.
__global__ void __launch_bounds__(TOPK_THREADS) topk_merge_kernel(const double *__restrict__ src, int64_t ld,
                                                                  int64_t g0, int32_t n_cols, int32_t m, int mode,
                                                                  int32_t k, int32_t *__restrict__ idx,
                                                                  double *__restrict__ sim) {
    __shared__ ListBuf b;
    const int64_t r = blockIdx.x;
    const int64_t g = g0 + r;
    int32_t clo, chi;
    uint32_t id_off;
    if (mode == 0) { clo = (int32_t)g + 1; chi = n_cols; id_off = 0; }
    else { clo = 0; chi = r < m ? (int32_t)r : m; id_off = (uint32_t)g0; }
    if (chi <= clo) return;                                   // nothing new for this row: the list stays
    const int seeded = list_seed(b, k, g, idx, sim);
    const int have = list_scan(b, src + r * ld, clo, chi, id_off, k, seeded == k);
    list_finish(b, have, k, g, idx, sim);
}

// ---------------------------------------------------------------------------------------------
// Fused top-k (sim_tensor.cu appends the survivors of each band to per-row candidate buffers): merge a
// row's buffer into its running list — top k of (list U candidates) under (similarity desc, id asc) —,
// publish the new k-th best as the row's threshold and empty the buffer.  A buffer that overflowed
// (more than `cap` survivors since the last merge: impossible unless the similarities are ordered
// adversarially along the diagonal distance) is NOT merged: what it holds only raises the threshold —
// every entry is a real similarity of the row, so the k-th best of (list U buffer) is a valid lower
// bound of the final one —, the row is flagged, and the band is run again for the flagged rows.
__global__ void __launch_bounds__(TOPK_THREADS) topk_compact_kernel(
    const int32_t *__restrict__ cand_id, const double *__restrict__ cand_sim, int32_t *__restrict__ cand_cnt,
    int32_t cap, int32_t k, int32_t *__restrict__ idx, double *__restrict__ sim, unsigned long long *__restrict__ thr_key,
    int32_t *__restrict__ thr_id, int32_t *__restrict__ row_flag, int32_t *__restrict__ overflow, int rerun) {
    __shared__ ListBuf b;
    const int64_t g = blockIdx.x;
    if (rerun && !row_flag[g]) return;                         // second pass of a band: flagged rows only
    const int cnt_all = cand_cnt[g];
    const bool over = cnt_all > cap;
    const int cnt = over ? cap : cnt_all;
    if (cnt == 0 && !rerun) return;                            // nothing new: list and threshold stay
    const int have = list_seed(b, k, g, idx, sim);
    for (int t = threadIdx.x; t < cnt; t += blockDim.x) list_put(b, have + t, cand_id[g * cap + t], cand_sim[g * cap + t]);
    const int total = have + cnt;
    list_finish(b, total, k, g, idx, sim, !over);
    if (threadIdx.x == 0) {
        // merged: the k-th best is IN the list, only strictly better entries matter from here on.  Overflowed:
        // the buffer is discarded, so the k-th best of (list U buffer) itself — a real entry that may belong
        // to the final list — and everything above it must be admitted again: threshold = just below it
        // (same key, id + 1).
        if (total >= k) { thr_key[g] = b.keys[k - 1]; thr_id[g] = (int32_t)(b.pos[k - 1] & ~NEG0) + (over ? 1 : 0); }
        else { thr_key[g] = 0ull; thr_id[g] = -1; }            // list not full: accept every valid similarity
        cand_cnt[g] = 0;
        row_flag[g] = over ? 1 : 0;
        if (over) atomicAdd(overflow, 1);
    }
}

// Second pass of a band: rows that did NOT overflow already hold the band's entries — their threshold is
// raised to "accept nothing" for the pass (restore = 0) and recomputed from their list afterwards (restore = 1).
__global__ void topk_mask_kernel(const int32_t *__restrict__ row_flag, const int32_t *__restrict__ idx,
                                 const double *__restrict__ sim, int32_t k, int64_t n, int restore,
                                 unsigned long long *__restrict__ thr_key, int32_t *__restrict__ thr_id) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n || row_flag[g]) return;
    if (!restore) { thr_key[g] = ~0ull; thr_id[g] = 0; return; }
    const int32_t id = idx[g * k + (k - 1)];
    if (id >= 0) { thr_key[g] = rs_sim_key(sim[g * k + (k - 1)]); thr_id[g] = id; }
    else { thr_key[g] = 0ull; thr_id[g] = -1; }
}

// T[(c - c0)][r] = S[r][c] for r in [0, m), c in [c0, n): 32 x 32 tiles through shared memory
__global__ void transpose_slab_kernel(const double *__restrict__ s, int64_t ld_s, int32_t m, int64_t c0, int32_t n,
                                      double *__restrict__ t, int64_t ld_t) {
    __shared__ double tile[32][33];
    const int64_t r0 = (int64_t)blockIdx.y * 32, c_base = c0 + (int64_t)blockIdx.x * 32;
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int64_t r = r0 + y, c = c_base + threadIdx.x;
        tile[y][threadIdx.x] = (r < m && c < n) ? s[r * ld_s + c] : 0.0;
    }
    __syncthreads();
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int64_t c = c_base + y, r = r0 + threadIdx.x;
        if (c < n && r < m) t[(c - c0) * ld_t + r] = tile[threadIdx.x][y];
    }
}

// Final neighbour lists from the partial lists of several ranks: out[row] = top k of the union of
// lists[l][row][*] (every (row, neighbour) pair occurs in exactly one partial list).
__global__ void __launch_bounds__(TOPK_THREADS) topk_union_kernel(const int32_t *__restrict__ idx_all,
                                                                  const double *__restrict__ sim_all, int32_t n_lists,
                                                                  int64_t n_rows, int32_t k, int32_t *__restrict__ idx,
                                                                  double *__restrict__ sim) {
    __shared__ ListBuf b;
    const int64_t g = blockIdx.x;
    if (threadIdx.x == 0) b.have = 0;
    __syncthreads();
    for (int t = threadIdx.x; t < n_lists * k; t += blockDim.x) {
        const int64_t o = ((int64_t)(t / k) * n_rows + g) * k + (t % k);
        const int32_t id = idx_all[o];
        if (id >= 0) list_put(b, atomicAdd(&b.have, 1), id, sim_all[o]);
    }
    __syncthreads();
    list_finish(b, b.have, k, g, idx, sim);
}


// ---------------------------------------------------------------------------------------------
// The three list schedules of an RS_STORE_TOPK Fit (rs_fit_lists chooses one, checks its k and allocates the lists).

// Rows of a slab: `m`, or RS_KNN_SLAB_ROWS (tests: many slabs on a small matrix), rounded down to a multiple of
// `unit` and at least `unit`.
int64_t slab_rows(int64_t m, int64_t unit) {
    if (const char *e = getenv("RS_KNN_SLAB_ROWS")) m = atoll(e);
    if (m < unit) m = unit;
    return m / unit * unit;
}

// FUSED (tensor path): the tensor kernel's epilogue tests every similarity against the current k-th best of its two
// rows and appends the survivors to per-row candidate buffers; the buffers are merged into the running lists between
// the waves of the tile schedule (sim_tensor.cu).  No similarity row, slab or transpose is ever written: the only
// N-proportional buffers are the lists (N x k) and the candidate buffers (N x cap).  Every pair is computed once; a
// multi-GPU Fit deals the tiles of each wave to the shards, every shard ends with PARTIAL lists for all rows (united
// after an all-gather).
int32_t lists_fused(rs_knn *h, int32_t k) {
    const int64_t n = h->n_left;
    RS_TRY(rs_alloc(h, &h->thr_key, (size_t)n));
    RS_TRY(rs_alloc(h, &h->thr_id, (size_t)n));
    RS_TRY(rs_alloc(h, &h->cand_cnt, (size_t)n));
    RS_TRY(rs_alloc(h, &h->row_flag, (size_t)n));
    RS_TRY(rs_alloc(h, &h->cand_id, (size_t)n * h->cand_cap));
    RS_TRY(rs_alloc(h, &h->cand_sim, (size_t)n * h->cand_cap));
    RS_CUDA(cudaMemsetAsync(h->thr_key, 0, (size_t)n * 8, h->stream));           // accept every valid similarity
    RS_CUDA(cudaMemsetAsync(h->thr_id, 0xFF, (size_t)n * 4, h->stream));
    RS_CUDA(cudaMemsetAsync(h->cand_cnt, 0, (size_t)n * 4, h->stream));
    RS_CUDA(cudaMemsetAsync(h->row_flag, 0, (size_t)n * 4, h->stream));
    int32_t *d_over = h->d_flags + 14;
    const auto mask = [&](int restore) -> int32_t {
        topk_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->row_flag, h->topk_idx, h->topk_sim, k,
                                                                              n, restore, h->thr_key, h->thr_id);
        h->prof.total_launches++;
        RS_CUDA(cudaGetLastError());
        return RS_OK;
    };
    RS_CUDA(cudaEventRecord(h->ev_b, h->stream));
    const int n_waves = rs_tensor_band_count(h);
    for (int w = 0; w < n_waves; w++) {
        for (int rerun = 0;; rerun = 1) {
            RS_CUDA(cudaMemsetAsync(d_over, 0, 4, h->stream));
            RS_TRY(rs_sim_tensor_band_launch(h, w));
            topk_compact_kernel<<<(unsigned)n, TOPK_THREADS, 0, h->stream>>>(
                h->cand_id, h->cand_sim, h->cand_cnt, h->cand_cap, k, h->topk_idx, h->topk_sim, h->thr_key, h->thr_id,
                h->row_flag, d_over, rerun);
            h->prof.total_launches++;
            RS_CUDA(cudaGetLastError());
            int32_t over = 0;
            RS_CUDA(cudaMemcpyAsync(&over, d_over, 4, cudaMemcpyDeviceToHost, h->stream));
            RS_CUDA(cudaStreamSynchronize(h->stream));
            if (rerun) RS_TRY(mask(1));                    // thresholds of the rows that sat the pass out
            if (over == 0) break;
            RS_TRY(mask(0));                               // run the band again for the flagged rows only
        }
    }
    return RS_OK;
}

// SYMMETRIC SLABS (see rs_knn_params::shard_count): slab s = rows [s*m, s*m+m); of each slab only the part right of
// the diagonal is computed, the slab feeds the lists of its own rows, its transpose the lists of the rows below it
// (topk_merge_kernel).  Half the similarity work of full rows, and the slabs of a multi-GPU job are dealt in snake
// order so every rank gets the same share of the triangle.
int32_t lists_symmetric_slabs(rs_knn *h, int path, int32_t k) {
    const int64_t n = h->n_left;
    int64_t m = (int64_t)(6ll << 30) / (h->ld_s * 8);        // ~6 GiB slab + the same for its transpose
    if (h->p.shard_count > 1) {
        // enough slabs for an even deal: at least 4 per shard (down to 1024 rows each)
        int64_t want = (n + 4ll * h->p.shard_count - 1) / (4ll * h->p.shard_count);
        want = (want + 255) / 256 * 256;
        if (want < 1024) want = 1024;
        if (want < m) m = want;
    }
    m = slab_rows(m, 256);
    if (m > n) m = (n + 15) / 16 * 16;
    const int64_t ld_t = m;
    double *tbuf = nullptr;
    RS_TRY(rs_alloc(h, &h->sims, (size_t)m * (size_t)h->ld_s));
    RS_TRY(rs_alloc(h, &tbuf, (size_t)n * (size_t)ld_t));
    RS_CUDA(cudaEventRecord(h->ev_b, h->stream));
    const int64_t n_slabs = (n + m - 1) / m;
    h->force_sym = true;
    for (int64_t sl = 0; sl < n_slabs; sl++) {
        // snake deal: slab sl costs ~ (n_slabs - sl); rounds alternate direction so that every
        // shard gets the same share of the triangle (8 GPUs, 25 slabs dealt plainly: max/mean 1.28)
        const int64_t round = sl / h->p.shard_count, posn = sl % h->p.shard_count;
        const int64_t owner = (round & 1) ? h->p.shard_count - 1 - posn : posn;
        if (owner != h->p.shard_index) continue;
        const int64_t r0 = sl * m, r1 = r0 + m < n ? r0 + m : n;
        h->row_begin = r0;
        h->row_end = r1;
        h->col_begin = r0;
        if (path == RS_PATH_STREAM) {
            // the stream kernel skips whole column chunks left of the diagonal: unset = NaN
            RS_CUDA(cudaMemsetAsync(h->sims, 0xFF, (size_t)(r1 - r0) * (size_t)h->ld_s * 8, h->stream));
            RS_TRY(rs_sim_stream_launch(h));
        } else {
            RS_TRY(rs_sim_tensor_launch(h, nullptr, 0, 0));
        }
        // the slab rows' own lists, then the rows r0 .. n-1 from the transpose
        const int32_t rows = (int32_t)(r1 - r0);
        topk_merge_kernel<<<(unsigned)rows, TOPK_THREADS, 0, h->stream>>>(h->sims, h->ld_s, r0, (int32_t)n, rows, 0, k,
                                                                           h->topk_idx, h->topk_sim);
        h->prof.total_launches++;
        const int64_t rest = n - r0;
        if (rest > 1) {
            dim3 grid((unsigned)((rest + 31) / 32), (unsigned)((rows + 31) / 32)), block(32, 8);
            transpose_slab_kernel<<<grid, block, 0, h->stream>>>(h->sims, h->ld_s, rows, r0, (int32_t)n, tbuf, ld_t);
            topk_merge_kernel<<<(unsigned)rest, TOPK_THREADS, 0, h->stream>>>(tbuf, ld_t, r0, (int32_t)n, rows, 1, k,
                                                                               h->topk_idx, h->topk_sim);
            h->prof.total_launches += 2;
        }
        RS_CUDA(cudaGetLastError());
    }
    return RS_OK;
}

// FULL-ROW SLABS: the similarity rows of the handle are produced slab by slab and reduced to neighbour lists; the
// N x N matrix never exists in HBM.
int32_t lists_row_slabs(rs_knn *h, int path, int32_t k) {
    const int64_t rb = h->row_begin, re = h->row_end;
    int64_t slab = slab_rows((int64_t)(2ull << 30) / ((int64_t)h->ld_s * 8), 128);   // ~2 GiB of rows at a time
    if (slab > re - rb) slab = re - rb;
    RS_TRY(rs_alloc(h, &h->sims, (size_t)slab * (size_t)h->ld_s));
    RS_CUDA(cudaEventRecord(h->ev_b, h->stream));
    for (int64_t r0 = rb; r0 < re; r0 += slab) {
        h->row_begin = r0;
        h->row_end = r0 + slab < re ? r0 + slab : re;
        RS_TRY(path == RS_PATH_TENSOR ? rs_sim_tensor_launch(h, nullptr, 0, 0) : rs_sim_stream_launch(h));
        if (path == RS_PATH_STREAM) RS_TRY(rs_symmetrize_launch(h));
        RS_TRY(rs_topk_rows_launch(h, h->sims, h->ld_s, h->n_left, h->row_end - r0, k, h->topk_idx + (r0 - rb) * k,
                                   h->topk_sim + (r0 - rb) * k));
    }
    return RS_OK;
}

}  // namespace

// The k the block top-k supports: TOPK_CAP - TOPK_THREADS candidates are kept between sorts, and k of them survive.
int32_t rs_topk_check_k(int32_t k) {
    if (k < 1 || k > TOPK_CAP / 4) {
        rs_set_error("top-k supports 1 <= k <= %d (got %d)", TOPK_CAP / 4, k);
        return RS_ERR_UNSUPPORTED;
    }
    return RS_OK;
}

// Top-k of `rows` rows of any row-major matrix of similarities or scores (ld = row pitch, n columns).
int32_t rs_topk_rows_launch(rs_knn *h, const double *src, int64_t ld, int32_t n, int64_t rows, int32_t k, int32_t *d_idx,
                            double *d_sim) {
    if (rows <= 0) return RS_OK;
    topk_rows_kernel<<<(unsigned)rows, TOPK_THREADS, 0, h->stream>>>(src, ld, n, k, d_idx, d_sim);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

// The neighbour lists of an RS_STORE_TOPK Fit, by the schedule the handle's sharding and path call for: FUSED into
// the tensor kernel, SYMMETRIC SLABS (shard_count >= 1), or FULL-ROW SLABS of the handle's rows.
int32_t rs_fit_lists(rs_knn *h, int path) {
    const int32_t k = rs_list_k(h);
    const bool sym = h->p.shard_count >= 1;
    const bool fused = sym && path == RS_PATH_TENSOR && rs_tensor_topk_fused(h);
    if (fused) {
        h->cand_cap = 1792;                          // band 0 brings at most 2 * (512 + 256) entries per row
        if (const char *e = getenv("RS_KNN_TOPK_CAP")) h->cand_cap = atoi(e);   // tests: force the overflow path
        if (k < 1 || k > 256 || h->cand_cap + k > TOPK_CAP || h->cand_cap < 1) {
            rs_set_error("fused top-k: k <= 256 and candidate capacity + k <= %d (k=%d cap=%d)", TOPK_CAP, k,
                         h->cand_cap);
            return RS_ERR_UNSUPPORTED;
        }
    } else {
        RS_TRY(rs_topk_check_k(k));
    }
    const int64_t rows = sym ? h->n_left : h->row_end - h->row_begin;
    RS_TRY(rs_alloc(h, &h->topk_idx, (size_t)rows * k));
    RS_TRY(rs_alloc(h, &h->topk_sim, (size_t)rows * k));
    h->topk_rows = rows;
    RS_CUDA(cudaMemsetAsync(h->topk_idx, 0xFF, (size_t)rows * k * 4, h->stream));   // -1 = empty
    RS_CUDA(cudaMemsetAsync(h->topk_sim, 0xFF, (size_t)rows * k * 8, h->stream));   // NaN
    // the slab schedules point the handle at one slab at a time
    const int64_t row_begin = h->row_begin, row_end = h->row_end, col_begin = h->col_begin;
    const int32_t rc = fused ? lists_fused(h, k) : sym ? lists_symmetric_slabs(h, path, k) : lists_row_slabs(h, path, k);
    h->row_begin = row_begin;
    h->row_end = row_end;
    h->col_begin = col_begin;
    h->force_sym = false;
    return rc;
}

extern "C" int32_t rs_knn_topk_union_device(int32_t n_lists, int64_t n_rows, int32_t k, const int32_t *d_idx_all,
                                            const double *d_sim_all, int32_t *d_idx, double *d_sim,
                                            void *cuda_stream) {
    if (n_lists < 1 || n_rows < 1 || k < 1 || !d_idx_all || !d_sim_all || !d_idx || !d_sim) {
        rs_set_error("rs_knn_topk_union: bad argument");
        return RS_ERR_INVALID;
    }
    if ((int64_t)n_lists * k > TOPK_CAP) {
        rs_set_error("rs_knn_topk_union: n_lists * k = %lld exceeds %d", (long long)n_lists * k, TOPK_CAP);
        return RS_ERR_UNSUPPORTED;
    }
    topk_union_kernel<<<(unsigned)n_rows, TOPK_THREADS, 0, reinterpret_cast<cudaStream_t>(cuda_stream)>>>(
        d_idx_all, d_sim_all, n_lists, n_rows, k, d_idx, d_sim);
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}
