// predict.cu — batched KNN.Predict (core/knn.go:75-141) and SlopeOne.Predict.
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

