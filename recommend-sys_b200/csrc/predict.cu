// predict.cu — batched KNN.Predict (core/knn.go:75-141) and per-row top-k.
//
// Predict: one warp per (left,right) test pair.
//   1. candidates = entries of the right row (core/knn.go:95-99), similarity gathered from
//      the left row of the HBM-resident matrix; NaN filtered; count <= mink -> GlobalMean.
//   2. the candidates are ordered by (similarity desc, inner id asc) — the canonical tie
//      policy — with a warp-level bitonic sort over (key,pos) records in shared memory
//      (right rows are id-sorted, so position order == id order);
//   3. the first min(k,count) are accumulated SEQUENTIALLY in that order exactly as
//      core/knn.go:116-130 does, so the prediction is bit-identical to the restated
//      reference under the canonical policy.
// HBM-bound by design: per prediction C*(4 B id + 8 B rating + 8 B similarity [+ 8 B mean/bias]).
#include <cub/cub.cuh>

#include <cstdlib>

#include "common.cuh"
#include "select.cuh"

namespace {

// Main predict kernel: one warp per test pair, the selection and weighted sum of select.cuh (select_loop).
template <int R>
__global__ void __launch_bounds__(SEL_WARPS * 32) predict_select_kernel(PredArgs a, int scap) {
    constexpr int CAP = 32 * R;
    // per-warp staging of the gathered similarities: pass A gathers each candidate's similarity
    // from HBM/L2 once (4 independent gathers per lane in flight) and parks the first `scap` of
    // them here; the selection passes read them back instead of gathering again
    extern __shared__ unsigned long long s_stage[];
    __shared__ uint32_t s_hist[SEL_WARPS][256];
    __shared__ uint64_t s_key[SEL_WARPS][CAP];
    __shared__ uint32_t s_pos[SEL_WARPS][CAP];
    __shared__ double s_av[SEL_WARPS][CAP];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t *hist = s_hist[warp];
    uint64_t *ckey = s_key[warp];
    uint32_t *cpos = s_pos[warp];
    uint64_t *sbuf = reinterpret_cast<uint64_t *>(s_stage) + (size_t)warp * scap;
    // keys that do not fit the shared-memory stage are parked in a per-warp slice of global memory
    // (written once, re-read coalesced by the selection passes — it stays in L2), NOT gathered again:
    // a second dependent gather per pass was 39 % of this kernel's stall samples (profiles/r02_predict_notes.md)
    uint64_t *gbuf = a.gstage + ((size_t)blockIdx.x * SEL_WARPS + warp) * (size_t)a.gcap - scap;
    const double nan_v = __longlong_as_double(0x7ff8000000000001ll);
    const int64_t n_eff = a.n_dev ? (int64_t)*a.n_dev : a.n;

    // Positions are handed out in order from one counter, so the predictions in flight are always
    // a contiguous window of the (row-grouped) order however unevenly long they take — with a
    // static stride the warps drift apart and the window grows past L2 (137 GB of DRAM reads per
    // 4 M predictions on the MovieLens-20M shape, profiles/r01_predict_ml20m_summary.txt).
    const auto item = [&](int64_t w, PredItem &c) -> bool {
        const int64_t p = a.perm ? (int64_t)a.perm[w] : w;
        const int32_t l = a.left[p], r = a.right[p];
        if (a.nb_count && lane == 0) *a.nb_count = 0;
        if (l < a.row_begin || l >= a.row_end || (a.cyc_R > 1 && l >= 0 && !rs_cyc_owns(l, a.cyc_R, a.cyc_r))) {
            if (l >= 0) {                                   // a known row of another shard
                if (lane == 0) a.out[p] = a.foreign_zero ? 0.0 : nan_v;
                return false;
            }
        }
        if (l < 0 || r < 0 || r >= a.n_right) {            // core/knn.go:89-91 (newID)
            const bool mine = !(a.foreign_zero && a.cyc_R > 1 && l < 0) || (int)(p % a.cyc_R) == a.cyc_r;
            if (lane == 0) a.out[p] = mine ? a.global_mean : 0.0;
            return false;
        }
        c.l = l;
        c.cb = a.r_ptr[r];
        c.cnt = (int)(a.r_ptr[r + 1] - c.cb);              // a right row has at most n_left entries
        c.row = a.sims + (a.cyc_R > 1 ? rs_cyc_local(l, a.cyc_R) : l - a.row_begin) * a.ld_s;
        c.dst = a.out + p;
        return true;
    };
    select_loop<R>(a, a.work, n_eff, item, lane, hist, ckey, cpos, s_av[warp], sbuf, gbuf, scap);
}


// ---------------- per-row top-k from the resident matrix ----------------
// +-0 share one key: they tie and are ordered by id, as the reference's float comparison does.  The block
// top-k kernels carry the sign of a zero in bit 31 of the id word, so that a list reports the exact
// similarity (-0.0 included) while the order stays that of (key, id).
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

__global__ void __launch_bounds__(TOPK_THREADS) topk_rows_kernel(const double *__restrict__ sims, int64_t ld_s,
                                                                 int32_t n, int32_t k, int32_t *__restrict__ idx,
                                                                 double *__restrict__ sim) {
    __shared__ uint64_t keys[TOPK_CAP];
    __shared__ uint32_t pos[TOPK_CAP];
    __shared__ int s_have;
    __shared__ uint64_t s_thr_key;
    __shared__ uint32_t s_thr_pos;
    const int64_t r = blockIdx.x;
    const double *row = sims + r * ld_s;
    if (threadIdx.x == 0) { s_have = 0; s_thr_key = 0; s_thr_pos = 0xffffffffu; }
    __syncthreads();
    bool have_thr = false;
    for (int32_t base = 0; base < n; base += TOPK_THREADS) {
        const int32_t j = base + threadIdx.x;
        bool take = false;
        uint64_t key = 0;
        uint32_t neg0 = 0;
        if (j < n) {
            const double s = row[j];
            if (s == s) {
                key = rs_sim_key(s);
                take = !have_thr || ent_before(key, (uint32_t)j, s_thr_key, s_thr_pos);
                neg0 = neg0_bit(s);
            }
        }
        if (take) {
            int slot = atomicAdd(&s_have, 1);
            keys[slot] = key;
            pos[slot] = (uint32_t)j | neg0;
        }
        __syncthreads();
        // every thread must see the SAME count: read it, then a second barrier before anybody's next
        // atomicAdd can change it (otherwise a slow thread may take the branch below alone)
        const int have_now = s_have;
        __syncthreads();
        if (have_now > TOPK_CAP - TOPK_THREADS) {
            const int have = have_now;
            for (int t = have + threadIdx.x; t < TOPK_CAP; t += blockDim.x) { keys[t] = 0; pos[t] = 0xffffffffu; }
            block_bitonic(keys, pos, TOPK_CAP);
            if (threadIdx.x == 0) {
                s_have = k;
                s_thr_key = keys[k - 1];
                s_thr_pos = pos[k - 1];
            }
            have_thr = true;
            __syncthreads();
        }
    }
    const int have = s_have;
    int n_pad = 32;
    while (n_pad < have) n_pad <<= 1;
    for (int t = have + threadIdx.x; t < n_pad; t += blockDim.x) { keys[t] = 0; pos[t] = 0xffffffffu; }
    block_bitonic(keys, pos, n_pad);
    for (int t = threadIdx.x; t < k; t += blockDim.x) {
        const int64_t o = r * k + t;
        if (t < have) { idx[o] = (int32_t)(pos[t] & ~NEG0); sim[o] = ent_sim(keys[t], pos[t]); }
        else { idx[o] = -1; sim[o] = __longlong_as_double(0x7ff8000000000001ll); }
    }
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
    __shared__ uint64_t keys[TOPK_CAP];
    __shared__ uint32_t pos[TOPK_CAP];
    __shared__ int s_have;
    __shared__ uint64_t s_thr_key;
    __shared__ uint32_t s_thr_pos;
    const int64_t r = blockIdx.x;
    const int64_t g = g0 + r;
    const double *row = src + r * ld;
    int32_t clo, chi;
    uint32_t id_off;
    if (mode == 0) { clo = (int32_t)g + 1; chi = n_cols; id_off = 0; }
    else { clo = 0; chi = r < m ? (int32_t)r : m; id_off = (uint32_t)g0; }
    if (chi <= clo) return;                                   // nothing new for this row: the list stays
    if (threadIdx.x == 0) { s_have = 0; s_thr_key = 0; s_thr_pos = 0xffffffffu; }
    __syncthreads();
    // seed with the running list; it is stored best first, so a FULL list gives the threshold right
    // away (its last entry): almost every new candidate of a later slab is rejected by one compare
    for (int t = threadIdx.x; t < k; t += blockDim.x) {
        const int32_t id = idx[g * k + t];
        if (id >= 0) {
            const int slot = atomicAdd(&s_have, 1);
            keys[slot] = rs_sim_key(sim[g * k + t]);
            pos[slot] = (uint32_t)id | neg0_bit(sim[g * k + t]);
        }
    }
    bool have_thr = idx[g * k + (k - 1)] >= 0;
    if (have_thr && threadIdx.x == 0) {
        s_thr_key = rs_sim_key(sim[g * k + (k - 1)]);
        s_thr_pos = (uint32_t)idx[g * k + (k - 1)];
    }
    __syncthreads();
    for (int32_t base = clo; base < chi; base += TOPK_THREADS) {
        const int32_t j = base + threadIdx.x;
        bool take = false;
        uint64_t key = 0;
        uint32_t neg0 = 0;
        if (j < chi) {
            const double s = row[j];
            if (s == s) {
                key = rs_sim_key(s);
                take = !have_thr || ent_before(key, (uint32_t)j + id_off, s_thr_key, s_thr_pos);
                neg0 = neg0_bit(s);
            }
        }
        if (take) {
            int slot = atomicAdd(&s_have, 1);
            keys[slot] = key;
            pos[slot] = ((uint32_t)j + id_off) | neg0;
        }
        __syncthreads();
        // every thread must see the SAME count: read it, then a second barrier before anybody's next
        // atomicAdd can change it (otherwise a slow thread may take the branch below alone)
        const int have_now = s_have;
        __syncthreads();
        if (have_now > TOPK_CAP - TOPK_THREADS) {
            const int have = have_now;
            for (int t = have + threadIdx.x; t < TOPK_CAP; t += blockDim.x) { keys[t] = 0; pos[t] = 0xffffffffu; }
            block_bitonic(keys, pos, TOPK_CAP);
            if (threadIdx.x == 0) {
                s_have = k;
                s_thr_key = keys[k - 1];
                s_thr_pos = pos[k - 1];
            }
            have_thr = true;
            __syncthreads();
        }
    }
    const int have = s_have;
    int n_pad = 32;
    while (n_pad < have) n_pad <<= 1;
    for (int t = have + threadIdx.x; t < n_pad; t += blockDim.x) { keys[t] = 0; pos[t] = 0xffffffffu; }
    block_bitonic(keys, pos, n_pad);
    for (int t = threadIdx.x; t < k; t += blockDim.x) {
        const int64_t o = g * k + t;
        if (t < have) { idx[o] = (int32_t)(pos[t] & ~NEG0); sim[o] = ent_sim(keys[t], pos[t]); }
        else { idx[o] = -1; sim[o] = __longlong_as_double(0x7ff8000000000001ll); }
    }
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
    __shared__ uint64_t keys[TOPK_CAP];
    __shared__ uint32_t pos[TOPK_CAP];
    const int64_t g = blockIdx.x;
    if (rerun && !row_flag[g]) return;                         // second pass of a band: flagged rows only
    const int cnt_all = cand_cnt[g];
    const bool over = cnt_all > cap;
    const int cnt = over ? cap : cnt_all;
    if (cnt == 0 && !rerun) return;                            // nothing new: list and threshold stay
    int have = 0;                                              // the list is stored best first: its entries are a prefix
    for (int t = threadIdx.x; t < k; t += blockDim.x) {
        const int32_t id = idx[g * k + t];
        keys[t] = id >= 0 ? rs_sim_key(sim[g * k + t]) : 0ull;
        pos[t] = id >= 0 ? (uint32_t)id | neg0_bit(sim[g * k + t]) : 0xffffffffu;
    }
    __syncthreads();
    // number of list entries (prefix length)
    __shared__ int s_have;
    if (threadIdx.x == 0) s_have = 0;
    __syncthreads();
    for (int t = threadIdx.x; t < k; t += blockDim.x)
        if (pos[t] != 0xffffffffu) atomicAdd(&s_have, 1);
    __syncthreads();
    have = s_have;
    for (int t = threadIdx.x; t < cnt; t += blockDim.x) {
        keys[have + t] = rs_sim_key(cand_sim[g * cap + t]);
        pos[have + t] = (uint32_t)cand_id[g * cap + t] | neg0_bit(cand_sim[g * cap + t]);
    }
    const int total = have + cnt;
    int n_pad = 32;
    while (n_pad < total) n_pad <<= 1;
    __syncthreads();
    for (int t = total + threadIdx.x; t < n_pad; t += blockDim.x) { keys[t] = 0; pos[t] = 0xffffffffu; }
    block_bitonic(keys, pos, n_pad);
    if (!over) {
        for (int t = threadIdx.x; t < k; t += blockDim.x) {
            const int64_t o = g * k + t;
            if (t < total) { idx[o] = (int32_t)(pos[t] & ~NEG0); sim[o] = ent_sim(keys[t], pos[t]); }
            else { idx[o] = -1; sim[o] = __longlong_as_double(0x7ff8000000000001ll); }
        }
    }
    if (threadIdx.x == 0) {
        // merged: the k-th best is IN the list, only strictly better entries matter from here on.  Overflowed:
        // the buffer is discarded, so the k-th best of (list U buffer) itself — a real entry that may belong
        // to the final list — and everything above it must be admitted again: threshold = just below it
        // (same key, id + 1).
        if (total >= k) { thr_key[g] = keys[k - 1]; thr_id[g] = (int32_t)(pos[k - 1] & ~NEG0) + (over ? 1 : 0); }
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
    __shared__ uint64_t keys[TOPK_CAP];
    __shared__ uint32_t pos[TOPK_CAP];
    __shared__ int s_have;
    const int64_t g = blockIdx.x;
    if (threadIdx.x == 0) s_have = 0;
    __syncthreads();
    for (int t = threadIdx.x; t < n_lists * k; t += blockDim.x) {
        const int64_t o = ((int64_t)(t / k) * n_rows + g) * k + (t % k);
        const int32_t id = idx_all[o];
        if (id >= 0) {
            const int slot = atomicAdd(&s_have, 1);
            keys[slot] = rs_sim_key(sim_all[o]);
            pos[slot] = (uint32_t)id | neg0_bit(sim_all[o]);
        }
    }
    __syncthreads();
    const int have = s_have;
    int n_pad = 32;
    while (n_pad < have) n_pad <<= 1;
    for (int t = have + threadIdx.x; t < n_pad; t += blockDim.x) { keys[t] = 0; pos[t] = 0xffffffffu; }
    block_bitonic(keys, pos, n_pad);
    for (int t = threadIdx.x; t < k; t += blockDim.x) {
        const int64_t o = g * k + t;
        if (t < have) { idx[o] = (int32_t)(pos[t] & ~NEG0); sim[o] = ent_sim(keys[t], pos[t]); }
        else { idx[o] = -1; sim[o] = __longlong_as_double(0x7ff8000000000001ll); }
    }
}


// ---------------------------------------------------------------------------------------------
// SlopeOne.Predict (core/slope_one.go:22-45).  One warp per (item, user) pair:
//   prediction = userMeans[u] (GlobalMean for an unknown user); for a known item,
//   += ( sum over the user's ratings, in DATASET order, of dev[item][rated item] ) / (number of ratings).
// The lanes gather 32 deviations at a time into shared memory and every lane then adds them in
// order (the reference's sequential float64 sum), so the result is bit-identical.
constexpr int SLOPE_WARPS = 8;
__global__ void __launch_bounds__(SLOPE_WARPS * 32) slope_predict_kernel(
    const int32_t *__restrict__ left, const int32_t *__restrict__ right, int64_t n, double *__restrict__ out,
    const int64_t *__restrict__ r_ptr, const int32_t *__restrict__ rd_col, const double *__restrict__ right_means,
    const double *__restrict__ dev, int64_t ld, int64_t row_begin, int64_t row_end, int32_t n_left, int32_t n_right,
    double global_mean, unsigned long long *work) {
    __shared__ double s_d[SLOPE_WARPS][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const double nan_v = __longlong_as_double(0x7ff8000000000001ll);
    for (;;) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(work, (unsigned long long)PRED_GRAB);
        base = __shfl_sync(0xffffffffu, base, 0);
        if ((int64_t)base >= n) break;
        const int64_t w_end = (int64_t)base + PRED_GRAB < n ? (int64_t)base + PRED_GRAB : n;
        for (int64_t p = (int64_t)base; p < w_end; p++) {
            const int32_t item = left[p], user = right[p];
            if (user < 0 || user >= n_right) {                       // unknown user: core/slope_one.go:30-32
                if (lane == 0) out[p] = global_mean;
                continue;
            }
            double prediction = right_means[user];
            if (item < 0 || item >= n_left) {                        // unknown item: the user's mean
                if (lane == 0) out[p] = prediction;
                continue;
            }
            if (item < row_begin || item >= row_end) {               // not in this shard
                if (lane == 0) out[p] = nan_v;
                continue;
            }
            const double *row = dev + (item - row_begin) * ld;
            const int64_t b = r_ptr[user], e = r_ptr[user + 1];
            double sum = 0.0;
            for (int64_t x0 = b; x0 < e; x0 += 32) {
                const int64_t x = x0 + lane;
                s_d[warp][lane] = x < e ? row[rd_col[x]] : 0.0;
                __syncwarp();
                const int lim = (e - x0) < 32 ? (int)(e - x0) : 32;
                for (int t = 0; t < lim; t++) sum += s_d[warp][t];   // core/slope_one.go:36, in order
                __syncwarp();
            }
            const double count = (double)(e - b);
            if (count > 0) prediction += sum / count;                // core/slope_one.go:39-41
            if (lane == 0) out[p] = prediction;
        }
    }
}

}  // namespace

// Sharded Predict: sort key that puts the shard's OWN pairs first, grouped by left row; foreign pairs (answered with
// +0.0 by a memset) get the largest key and are never visited.  own = the left row belongs to the shard, or the pair is
// a cold start (left = -1: GlobalMean) dealt to this shard by position.
__global__ void own_key_kernel(const int32_t *__restrict__ left, int64_t n, int32_t count, int32_t index,
                               int32_t *__restrict__ key, int32_t *__restrict__ iota, long long *__restrict__ n_own) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool own = false;
    if (i < n) {
        const int32_t l = left[i];
        own = l < 0 ? (int)(i % count) == index : rs_cyc_owns(l, count, index);
        key[i] = own ? l + 1 : 0x7fffffff;
        iota[i] = (int32_t)i;
    }
    const uint32_t m = __ballot_sync(0xffffffffu, own);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(reinterpret_cast<unsigned long long *>(n_own), (unsigned long long)__popc(m));
}

__global__ void iota_kernel(int32_t *out, int32_t n) {
    const int32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x < n) out[x] = x;
}

template <int R>
static int32_t launch_select(const PredArgs &a, unsigned blocks, size_t smem, int scap, cudaStream_t st) {
    auto kern = predict_select_kernel<R>;
    RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<blocks, SEL_WARPS * 32, smem, st>>>(a, scap);
    return RS_OK;
}

int32_t rs_predict_launch(rs_knn *h, const int32_t *d_left, const int32_t *d_right, int64_t n, double *d_out,
                          int32_t *d_nb_ids, double *d_nb_sims, int32_t *d_nb_count, int32_t nb_cap, int32_t foreign_zero) {
    if (n <= 0) return RS_OK;
    if (h->p.k > PRED_CAP / 2) {
        rs_set_error("k=%d exceeds the %d neighbours the predict kernel supports", h->p.k, PRED_CAP / 2);
        return RS_ERR_UNSUPPORTED;
    }
    if (n >= (1ll << 31)) {
        rs_set_error("at most 2^31-1 predictions per call");
        return RS_ERR_UNSUPPORTED;
    }
    PredArgs a{};
    a.left = d_left; a.right = d_right; a.n = n; a.out = d_out;
    a.r_ptr = h->r_ptr; a.r_col = h->r_col; a.r_val = h->r_val;
    a.sims = h->sims; a.ld_s = h->ld_s; a.row_begin = h->row_begin; a.row_end = h->row_end;
    a.cyc_R = h->cyc_R; a.cyc_r = h->cyc_r;
    a.foreign_zero = foreign_zero;
    a.means = h->means; a.stddevs = h->stddevs; a.bias = h->left_bias;
    a.global_mean = h->global_mean; a.n_right = h->n_right;
    a.k = h->p.k; a.min_k = h->p.min_k; a.knn_type = h->p.knn_type;
    a.nb_ids = d_nb_ids; a.nb_sims = d_nb_sims; a.nb_count = d_nb_count; a.nb_cap = nb_cap;
    // Large batches are processed grouped by left row: the gathers of one prediction all fall in
    // ONE row of the similarity matrix (N x 8 B), so test pairs of the same row, run by neighbouring
    // warps at the same time, find that row in L2 instead of fetching it from HBM once per pair
    // (MovieLens-20M item shape: 150 test pairs per row, 5.7 GB matrix).  Stable radix sort of
    // (left id, index) — CUB, plumbing — and the kernel walks the permutation.
    a.perm = nullptr;
    a.n_dev = nullptr;
    if (foreign_zero && h->cyc_R > 1 && n >= 4096) {
        // sharded Predict over the FULL test set: the foreign pairs are answered by a memset (+0.0) and the kernel
        // only visits the shard's own pairs, found — and grouped by left row — by ONE radix sort whose key puts
        // foreign pairs last (walking all positions to skip 7 of 8 cost 2.7 ms of a 4.8 ms launch at 8 shards)
        void *keys_in, *keys_out, *iota, *perm, *tmp, *cnt;
        RS_TRY(rs_scratch_get(h, RS_SCR_PRED_KEYS_IN, (size_t)n * 4, &keys_in));
        RS_TRY(rs_scratch_get(h, RS_SCR_PRED_KEYS, (size_t)n * 4, &keys_out));
        RS_TRY(rs_scratch_get(h, RS_SCR_PRED_IOTA, (size_t)n * 4, &iota));
        RS_TRY(rs_scratch_get(h, RS_SCR_PRED_PERM, (size_t)n * 4, &perm));
        RS_TRY(rs_scratch_get(h, RS_SCR_PRED_OWN_COUNT, 8, &cnt));
        size_t need = 0;
        RS_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, need, (int32_t *)keys_in, (int32_t *)keys_out, (int32_t *)iota,
                                                (int32_t *)perm, (int)n, 0, 31, h->stream));
        RS_TRY(rs_scratch_get(h, RS_SCR_PRED_SORT_TMP, need + 256, &tmp));
        RS_CUDA(cudaMemsetAsync(cnt, 0, 8, h->stream));
        RS_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n * 8, h->stream));
        own_key_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(d_left, n, h->cyc_R, h->cyc_r, (int32_t *)keys_in,
                                                                            (int32_t *)iota, (long long *)cnt);
        RS_CUDA(cub::DeviceRadixSort::SortPairs(tmp, need, (int32_t *)keys_in, (int32_t *)keys_out, (int32_t *)iota,
                                                (int32_t *)perm, (int)n, 0, 31, h->stream));
        a.perm = (const int32_t *)perm;
        a.n_dev = (const long long *)cnt;
        h->prof.total_launches += 1;
    } else if (n >= 65536 && (size_t)h->rows_local * (size_t)h->ld_s * 8 > ((size_t)64 << 20) &&
        !getenv("RS_KNN_PRED_NOSORT")) {
        void *keys_out, *iota, *perm, *tmp;
        RS_TRY(rs_scratch_get(h, RS_SCR_PRED_KEYS, (size_t)n * 4, &keys_out));
        RS_TRY(rs_scratch_get(h, RS_SCR_PRED_IOTA, (size_t)n * 4, &iota));
        RS_TRY(rs_scratch_get(h, RS_SCR_PRED_PERM, (size_t)n * 4, &perm));
        size_t need = 0;
        int bits = 1;
        while ((1ll << bits) < (long long)h->n_left && bits < 31) bits++;
        RS_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, need, d_left, (int32_t *)keys_out, (int32_t *)iota,
                                                (int32_t *)perm, (int)n, 0, bits, h->stream));
        RS_TRY(rs_scratch_get(h, RS_SCR_PRED_SORT_TMP, need + 256, &tmp));
        iota_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((int32_t *)iota, (int32_t)n);
        RS_CUDA(cub::DeviceRadixSort::SortPairs(tmp, need, d_left, (int32_t *)keys_out, (int32_t *)iota,
                                                (int32_t *)perm, (int)n, 0, bits, h->stream));
        a.perm = (const int32_t *)perm;
        h->prof.total_launches += 1;   // own kernels only
    }
    {
        void *work;
        RS_TRY(rs_scratch_get(h, RS_SCR_WORK, 8, &work));
        RS_CUDA(cudaMemsetAsync(work, 0, 8, h->stream));
        a.work = reinterpret_cast<unsigned long long *>(work);
    }
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    int64_t blocks = (n + SEL_WARPS * PRED_GRAB - 1) / (SEL_WARPS * PRED_GRAB);
    const int64_t cap = (int64_t)sms * 8;   // resident CTAs; warps stride over the predictions
    if (blocks > cap) blocks = cap;
    // staging capacity per warp (similarities parked in shared memory between the passes)
    // with the global spill behind it a small stage wins (more resident warps): ML-20M shape, 4 M predictions:
    // 128: 17.5 ms, 256: 16.8, 512: 20.6, 1024: 24.5
    int scap = 256;
    if (const char *e = getenv("RS_KNN_PRED_SCAP")) scap = atoi(e);
    if (scap < 0) scap = 0;
    if (scap > 2048) scap = 2048;
    scap = scap / 32 * 32;
    const size_t smem = (size_t)SEL_WARPS * scap * sizeof(double);
    const int64_t per_sm = smem ? (int64_t)(200 * 1024) / (int64_t)(smem + 16 * 1024) : 8;
    if (blocks > (int64_t)sms * (per_sm > 0 ? per_sm : 1)) blocks = (int64_t)sms * (per_sm > 0 ? per_sm : 1);
    {
        // global spill of the staged keys: one slice per resident warp, sized by the longest right row
        const int64_t gcap = h->max_right_len > scap ? (((int64_t)h->max_right_len - scap + 31) / 32 * 32) : 32;
        void *g;
        RS_TRY(rs_scratch_get(h, RS_SCR_KEY_SPILL, (size_t)blocks * SEL_WARPS * (size_t)gcap * 8, &g));
        a.gstage = reinterpret_cast<uint64_t *>(g);
        a.gcap = gcap;
    }
    // register capacity of the selection kernel: room for k plus a boundary bucket
    if (h->p.k <= 44) RS_TRY(launch_select<2>(a, (unsigned)blocks, smem, scap, h->stream));
    else if (h->p.k <= 104) RS_TRY(launch_select<4>(a, (unsigned)blocks, smem, scap, h->stream));
    else RS_TRY(launch_select<8>(a, (unsigned)blocks, smem, scap, h->stream));
    h->prof.predict_launches++;
    h->prof.total_launches += 1;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

// The neighbour report of a single prediction (rs_knn_predict_neighbors): the selection kernel writes the
// similarity its record was sorted by, where -0.0 has become +0.0; the list reports the matrix cells themselves.
__global__ void nb_cells_kernel(const double *__restrict__ sims, int64_t ld_s, int64_t row_begin, int32_t cyc_R,
                                const int32_t *__restrict__ left, const int32_t *__restrict__ nb_ids,
                                const int32_t *__restrict__ nb_count, double *__restrict__ nb_sims) {
    const int32_t l = *left, cnt = *nb_count;
    if (cnt <= 0) return;                                     // cold start / mink: nothing was reported
    const double *row = sims + (cyc_R > 1 ? rs_cyc_local(l, cyc_R) : l - row_begin) * ld_s;
    for (int e = threadIdx.x; e < cnt; e += blockDim.x) nb_sims[e] = row[nb_ids[e]];
}

int32_t rs_nb_cells_launch(rs_knn *h, const int32_t *d_left, const int32_t *d_nb_ids, const int32_t *d_nb_count,
                           double *d_nb_sims) {
    nb_cells_kernel<<<1, 256, 0, h->stream>>>(h->sims, h->ld_s, h->row_begin, h->cyc_R, d_left, d_nb_ids, d_nb_count,
                                              d_nb_sims);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

int32_t rs_topk_launch(rs_knn *h, int32_t k, int32_t *d_idx, double *d_sim) {
    const int64_t rows = h->cyc_R > 1 ? h->rows_local : h->row_end - h->row_begin;
    if (rows <= 0) return RS_OK;
    if (k < 1 || k > TOPK_CAP / 4) {
        rs_set_error("top-k supports 1 <= k <= %d (got %d)", TOPK_CAP / 4, k);
        return RS_ERR_UNSUPPORTED;
    }
    topk_rows_kernel<<<(unsigned)rows, TOPK_THREADS, 0, h->stream>>>(h->sims, h->ld_s, h->n_left, k, d_idx, d_sim);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
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

// Symmetric slab: merge the slab rows [g0, g0+m) (entries right of the diagonal) and their transpose
// into the running neighbour lists of all rows >= g0 (see topk_merge_kernel).
int32_t rs_topk_slab_launch(rs_knn *h, int64_t g0, int32_t m, double *tbuf, int64_t ld_t, int32_t k) {
    if (k < 1 || k > TOPK_CAP / 4) {
        rs_set_error("top-k supports 1 <= k <= %d (got %d)", TOPK_CAP / 4, k);
        return RS_ERR_UNSUPPORTED;
    }
    const int32_t n = h->n_left;
    topk_merge_kernel<<<(unsigned)m, TOPK_THREADS, 0, h->stream>>>(h->sims, h->ld_s, g0, n, m, 0, k, h->topk_idx,
                                                                 h->topk_sim);
    const int64_t rest = (int64_t)n - g0;                     // rows g0 .. n-1 receive transposed contributions
    if (rest > 1) {
        dim3 grid((unsigned)((rest + 31) / 32), (unsigned)((m + 31) / 32)), block(32, 8);
        transpose_slab_kernel<<<grid, block, 0, h->stream>>>(h->sims, h->ld_s, m, g0, n, tbuf, ld_t);
        topk_merge_kernel<<<(unsigned)rest, TOPK_THREADS, 0, h->stream>>>(tbuf, ld_t, g0, n, m, 1, k, h->topk_idx,
                                                                        h->topk_sim);
        h->prof.total_launches += 2;
    }
    h->prof.total_launches += 1;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

int32_t rs_topk_compact_launch(rs_knn *h, int32_t k, int32_t *d_overflow, int rerun) {
    if (k < 1 || k > TOPK_CAP / 4 || h->cand_cap + k > TOPK_CAP) {
        rs_set_error("fused top-k supports k <= %d and cap + k <= %d (got k=%d cap=%d)", TOPK_CAP / 4, TOPK_CAP, k, h->cand_cap);
        return RS_ERR_UNSUPPORTED;
    }
    topk_compact_kernel<<<(unsigned)h->n_left, TOPK_THREADS, 0, h->stream>>>(
        h->cand_id, h->cand_sim, h->cand_cnt, h->cand_cap, k, h->topk_idx, h->topk_sim, h->thr_key, h->thr_id,
        h->row_flag, d_overflow, rerun);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

int32_t rs_topk_mask_launch(rs_knn *h, int32_t k, int restore) {
    topk_mask_kernel<<<(unsigned)((h->n_left + 255) / 256), 256, 0, h->stream>>>(h->row_flag, h->topk_idx, h->topk_sim, k,
                                                                                h->n_left, restore, h->thr_key, h->thr_id);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
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

int32_t rs_slope_predict_launch(rs_knn *h, const int32_t *d_left, const int32_t *d_right, int64_t n, double *d_out) {
    if (n <= 0) return RS_OK;
    if (!h->rd_col || !h->right_means) {
        rs_set_error("rs_knn_predict_batch: the handle was not fitted with RS_SIM_SLOPE_ONE");
        return RS_ERR_INVALID;
    }
    void *work;
    RS_TRY(rs_scratch_get(h, RS_SCR_WORK, 8, &work));
    RS_CUDA(cudaMemsetAsync(work, 0, 8, h->stream));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    int64_t blocks = (n + SLOPE_WARPS * PRED_GRAB - 1) / (SLOPE_WARPS * PRED_GRAB);
    if (blocks > (int64_t)sms * 8) blocks = (int64_t)sms * 8;
    slope_predict_kernel<<<(unsigned)blocks, SLOPE_WARPS * 32, 0, h->stream>>>(
        d_left, d_right, n, d_out, h->r_ptr, h->rd_col, h->right_means, h->sims, h->ld_s, h->row_begin, h->row_end,
        h->n_left, h->n_right, h->global_mean, reinterpret_cast<unsigned long long *>(work));
    h->prof.predict_launches++;
    h->prof.total_launches += 1;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

