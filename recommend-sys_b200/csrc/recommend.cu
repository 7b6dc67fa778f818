// recommend.cu — top-N recommendation: the score of EVERY target of a query (Predict at catalogue scale), rated
// targets excluded, and the N best under (score desc, target id asc).
//
// A score is the prediction rs_knn_predict_batch makes for the same pair, bit for bit: both run the selection and
// weighted sum of select.cuh on the same candidates, in the same order, with the same similarities.
//   right query q (item-based: q is a user, the targets are the items t, score(t) = Predict(left = t, right = q)):
//     every target has the same candidates, the left ids R(q) of right row q, gathered from row S[t].  The scores
//     are handed out target-major, so the warps in flight gather from the same row S[t] for different queries and
//     find it in L2: the grouping by left row that Predict gets from a radix sort of its pairs, without the pairs.
//     (Reading the transposed rows S[j][t0 .. t0 + 32) of the symmetric matrix coalesced and parking them per target
//     was measured slower: DESIGN.md §5.3b.)
//   left query q (user-based: q is a user, the targets are the items t, score(t) = Predict(left = q, right = t)):
//     all gathers of the query come from ONE matrix row, S[q][.]; the scores are handed out query-major, so the
//     warps in flight share that row in L2.
// Rated targets are then overwritten with NaN and topk_rows_kernel (predict.cu) picks the N best of each row.
#include <cstdlib>

#include "common.cuh"
#include "select.cuh"

namespace {

struct RecArgs {
    const int32_t *queries;
    int64_t nq;
    int32_t side;           // enum rs_side
    int32_t n_side;         // ids of the query side: a query outside [0, n_side) is treated as -1 (cold start)
    int32_t n_targets;
    double *out;            // [nq][ld_out]
    int64_t ld_out;
    unsigned long long *work;
};

// One warp per (query, target) score, handed out in order from one counter.  Left queries are walked query-major
// (the warps in flight gather from the same row S[q]), right queries target-major (the warps in flight gather from
// the same row S[t], for the candidates R(q) of different queries), so the row of the moment stays in L2.
template <int R>
__global__ void __launch_bounds__(SEL_WARPS * 32) recommend_kernel(PredArgs a, RecArgs ra, int scap) {
    constexpr int CAP = 32 * R;
    extern __shared__ unsigned long long s_stage[];
    __shared__ uint32_t s_hist[SEL_WARPS][256];
    __shared__ uint64_t s_key[SEL_WARPS][CAP];
    __shared__ uint32_t s_pos[SEL_WARPS][CAP];
    __shared__ double s_av[SEL_WARPS][CAP];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint64_t *sbuf = reinterpret_cast<uint64_t *>(s_stage) + (size_t)warp * scap;
    uint64_t *gbuf = a.gstage + ((size_t)blockIdx.x * SEL_WARPS + warp) * (size_t)a.gcap - scap;
    const auto score = [&](int64_t w, PredItem &c) -> bool {
        const bool left = ra.side == RS_SIDE_LEFT;
        const int64_t b = left ? w / ra.n_targets : w % ra.nq;
        const int32_t t = (int32_t)(left ? w % ra.n_targets : w / ra.nq);
        const int32_t q = ra.queries[b];
        double *dst = ra.out + b * ra.ld_out + t;
        if (q < 0 || q >= ra.n_side) {                      // newID: GlobalMean (core/knn.go:89-91)
            if (lane == 0) *dst = a.global_mean;
            return false;
        }
        const int32_t l = left ? q : t, r = left ? t : q;  // the pair Predict(left = l, right = r)
        c.l = l;
        c.cb = a.r_ptr[r];
        c.cnt = (int)(a.r_ptr[r + 1] - c.cb);
        c.row = a.sims + (int64_t)l * a.ld_s;
        c.dst = dst;
        return true;
    };
    select_loop<R>(a, ra.work, ra.nq * ra.n_targets, score, lane, s_hist[warp], s_key[warp], s_pos[warp],
                              s_av[warp], sbuf, gbuf, scap);
}

// Rated targets: the query's row of the right CSR (right queries) or of the left CSR (left queries) -> NaN.
__global__ void recommend_exclude_kernel(const int32_t *__restrict__ queries, int32_t n_side,
                                         const int64_t *__restrict__ ptr, const int32_t *__restrict__ col,
                                         double *__restrict__ out, int64_t ld_out) {
    const int64_t b = blockIdx.x;
    const int32_t q = queries[b];
    if (q < 0 || q >= n_side) return;
    const double nan_v = __longlong_as_double(0x7ff8000000000001ll);
    for (int64_t e = ptr[q] + threadIdx.x; e < ptr[q + 1]; e += blockDim.x) out[b * ld_out + col[e]] = nan_v;
}

template <int R>
int32_t launch_scores(const PredArgs &a, const RecArgs &ra, unsigned blocks, size_t smem, int scap, cudaStream_t st) {
    auto kern = recommend_kernel<R>;
    RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<blocks, SEL_WARPS * 32, smem, st>>>(a, ra, scap);
    return RS_OK;
}

// Scores of the queries d_q[0 .. nq) into out[nq][ld_out], rated targets NaN.
int32_t score_rows(rs_knn *h, int32_t side, const int32_t *d_q, int64_t nq, double *out, int64_t ld_out) {
    PredArgs a{};
    a.r_ptr = h->r_ptr; a.r_col = h->r_col; a.r_val = h->r_val;
    a.sims = h->sims; a.ld_s = h->ld_s;
    a.means = h->means; a.stddevs = h->stddevs; a.bias = h->left_bias;
    a.global_mean = h->global_mean; a.n_right = h->n_right;
    a.k = h->p.k; a.min_k = h->p.min_k; a.knn_type = h->p.knn_type;
    RecArgs ra{};
    ra.queries = d_q; ra.nq = nq; ra.side = side;
    ra.n_side = side == RS_SIDE_RIGHT ? h->n_right : h->n_left;
    ra.n_targets = side == RS_SIDE_RIGHT ? h->n_left : h->n_right;
    ra.out = out; ra.ld_out = ld_out;
    void *work;
    RS_TRY(rs_scratch_get(h, 16, 8, &work));
    RS_CUDA(cudaMemsetAsync(work, 0, 8, h->stream));
    ra.work = reinterpret_cast<unsigned long long *>(work);
    a.work = ra.work;

    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    // the same per-warp stage as Predict (select.cuh): 256 keys in shared memory, the rest in a global slice
    const int scap = 256;
    const size_t smem = (size_t)SEL_WARPS * scap * sizeof(double);
    const int64_t warps = nq * ra.n_targets;
    int64_t blocks = (int64_t)sms * ((200 * 1024) / (int64_t)(smem + 16 * 1024));   // resident CTAs, as Predict sizes them
    if (blocks > (warps + SEL_WARPS - 1) / SEL_WARPS) blocks = (warps + SEL_WARPS - 1) / SEL_WARPS;
    const int64_t gcap = h->max_right_len > scap ? (((int64_t)h->max_right_len - scap + 31) / 32 * 32) : 32;
    void *g;
    RS_TRY(rs_scratch_get(h, 17, (size_t)blocks * SEL_WARPS * (size_t)gcap * 8, &g));
    a.gstage = reinterpret_cast<uint64_t *>(g);
    a.gcap = gcap;
    if (h->p.k <= 44) RS_TRY(launch_scores<2>(a, ra, (unsigned)blocks, smem, scap, h->stream));
    else if (h->p.k <= 104) RS_TRY(launch_scores<4>(a, ra, (unsigned)blocks, smem, scap, h->stream));
    else RS_TRY(launch_scores<8>(a, ra, (unsigned)blocks, smem, scap, h->stream));
    recommend_exclude_kernel<<<(unsigned)nq, 128, 0, h->stream>>>(d_q, ra.n_side, side == RS_SIDE_RIGHT ? h->r_ptr : h->l_ptr,
                                                                  side == RS_SIDE_RIGHT ? h->r_col : h->l_col, out, ld_out);
    h->prof.total_launches += 2;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

}  // namespace

int32_t rs_score_all_launch(rs_knn *h, int32_t side, const int32_t *d_q, int64_t n, double *d_out) {
    if (n <= 0) return RS_OK;
    const int64_t n_targets = side == RS_SIDE_RIGHT ? h->n_left : h->n_right;
    return score_rows(h, side, d_q, n, d_out, n_targets);
}

int32_t rs_recommend_launch(rs_knn *h, int32_t side, const int32_t *d_q, int64_t n, int32_t n_top, int32_t *d_ids,
                            double *d_scores) {
    if (n <= 0) return RS_OK;
    const int64_t n_targets = side == RS_SIDE_RIGHT ? h->n_left : h->n_right;
    // queries are scored in batches into a bounded slab of full score rows, ~256 MiB
    int64_t batch = ((int64_t)256 << 20) / (n_targets * 8);
    if (const char *e = getenv("RS_KNN_REC_BATCH")) batch = atoll(e);   // tests: force several batches
    if (batch < 1) batch = 1;
    if (batch > n) batch = n;
    void *slab;
    RS_TRY(rs_scratch_get(h, 23, (size_t)batch * n_targets * 8, &slab));
    for (int64_t b0 = 0; b0 < n; b0 += batch) {
        const int64_t nb = n - b0 < batch ? n - b0 : batch;
        RS_TRY(score_rows(h, side, d_q + b0, nb, (double *)slab, n_targets));
        RS_TRY(rs_topk_rows_launch(h, (const double *)slab, n_targets, (int32_t)n_targets, nb, n_top,
                                   d_ids + b0 * n_top, d_scores + b0 * n_top));
    }
    return RS_OK;
}
