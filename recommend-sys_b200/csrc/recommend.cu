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
// Rated targets are then overwritten with NaN and topk_rows_kernel (topk.cu) picks the N best of each row.
//
// Row shards (rs_knn_*_sharded_device): a shard holds complete rows of the similarity matrix and both CSRs.
//   right queries: the targets are the left rows, so a shard scores the targets it owns (local row t, global id
//     map.global(t)) for every query; the global top N is contained in the union of the shards' top-N lists.
//   left queries: a query needs row S[q] only; the owner of q scores it completely (a -1 query: the owner of row 0).
//     The queries the shard answers are compacted first, scored query-major as above, and their lists scattered back.
//
// Queries given as rating lists (rs_knn_*_given, lists prepared by given.cu): query b is list b of the call.
//   right: the list, sorted by id, is the right row of the query: it replaces the handle's right CSR as the candidate
//     CSR (a.r_ptr / r_col / r_val, r = b), and it is the query's rated targets.
//   left: the gathered row is the query's row of S* (given_sims_kernel, in a slab beside the score slab), and the
//     query's own mean / stddev follow the fitted rows' in one statistics array: Predict's left row is n_left + b.
#include <cstdlib>

#include <cub/cub.cuh>

#include "common.cuh"
#include "select.cuh"

namespace {

// Which left rows the handle holds, and where.  A full handle (row_begin 0, row_end n_left, no cyclic shards) maps
// every row to itself.
struct RowMap {
    int64_t row_begin, row_end;
    int32_t cyc_R, cyc_r;
    __host__ __device__ bool owns(int64_t i) const {
        return i >= row_begin && i < row_end && (cyc_R < 2 || rs_cyc_owns(i, cyc_R, cyc_r));
    }
    __host__ __device__ int64_t local(int64_t i) const { return cyc_R > 1 ? rs_cyc_local(i, cyc_R) : i - row_begin; }
    // Strictly increasing in `loc` under both schemes (cyclic: blocks of 32 dealt in order, rows in order inside a
    // block; contiguous: an offset).  So an order on local ids (the tie break "id asc" of topk_rows_kernel on a slab of
    // local columns) is the same order on global ids, and a shard's top-N list of its own targets is exactly the
    // prefix of the full ranking restricted to those targets: the union of the shards' lists is the full list.
    __host__ __device__ int64_t global(int64_t loc) const {
        return cyc_R > 1 ? rs_cyc_global(loc, cyc_R, cyc_r) : row_begin + loc;
    }
};

RowMap row_map(const rs_knn *h) { return RowMap{h->row_begin, h->row_end, h->cyc_R, h->cyc_r}; }

struct RecArgs {
    const int32_t *queries;
    const int32_t *rows;    // optional: the output row of query b (else b)
    int64_t nq;
    int32_t side;           // enum rs_side
    int32_t n_side;         // ids of the query side: a query outside [0, n_side) is treated as -1 (cold start)
    int32_t n_targets;      // targets scored per query: every id of the other side, or, for right queries on a row
                            // shard, the shard's own rows by local index
    int32_t out_global;     // right queries on a row shard: local target t goes to column map.global(t) (else t)
    int32_t given;          // queries given as rating lists: query b is list b (queries unused)
    int32_t qstat;          // left given: the statistics of query b are entry qstat + b of a.means / a.stddevs
    const double *gsims;    // left given: the similarity rows S*[b] of the batch
    int64_t ld_g;
    RowMap map;
    double *out;            // [rows][ld_out]
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
        const int32_t q = ra.given ? (int32_t)b : ra.queries[b];
        const int32_t tg = left ? t : (int32_t)ra.map.global(t);     // right queries: t is a local row
        double *dst = ra.out + (ra.rows ? (int64_t)ra.rows[b] : b) * ra.ld_out + (ra.out_global ? tg : t);
        if (!ra.given && (q < 0 || q >= ra.n_side)) {       // newID: GlobalMean (core/knn.go:89-91)
            if (lane == 0) *dst = a.global_mean;
            return false;
        }
        const int32_t l = left ? q : tg, r = left ? t : q;  // the pair Predict(left = l, right = r)
        c.l = left && ra.given ? ra.qstat + q : l;
        c.cb = a.r_ptr[r];
        c.cnt = (int)(a.r_ptr[r + 1] - c.cb);
        if (left && ra.given) c.row = ra.gsims + b * ra.ld_g;
        else c.row = a.sims + (left ? ra.map.local(q) : (int64_t)t) * a.ld_s;   // a left query is one the shard owns
        c.dst = dst;
        return true;
    };
    select_loop<R>(a, ra.work, ra.nq * ra.n_targets, score, lane, s_hist[warp], s_key[warp], s_pos[warp],
                              s_av[warp], sbuf, gbuf, scap);
}

// Rated targets: the query's row of the right CSR (right queries) or of the left CSR (left queries) -> NaN.  Right
// queries on a row shard: only the rated targets the shard owns, at their local or global column.  Given lists: list
// b of the given CSR.
__global__ void recommend_exclude_kernel(const RecArgs ra, const int64_t *__restrict__ ptr,
                                         const int32_t *__restrict__ col) {
    const int64_t b = blockIdx.x;
    const int32_t q = ra.given ? (int32_t)b : ra.queries[b];
    if (!ra.given && (q < 0 || q >= ra.n_side)) return;
    const bool right = ra.side == RS_SIDE_RIGHT;
    double *row = ra.out + (ra.rows ? (int64_t)ra.rows[b] : b) * ra.ld_out;
    const double nan_v = __longlong_as_double(0x7ff8000000000001ll);
    for (int64_t e = ptr[q] + threadIdx.x; e < ptr[q + 1]; e += blockDim.x) {
        int64_t t = col[e];
        if (right) {
            if (!ra.map.owns(t)) continue;
            if (!ra.out_global) t = ra.map.local(t);
        }
        row[t] = nan_v;
    }
}

// Left queries on a row shard: the queries this shard answers.  Its own rows, and -1 (or an id out of range) on the
// shard that owns row 0 only, so that a cold-start list is not produced twice.
__global__ void own_query_kernel(const int32_t *__restrict__ q, int64_t n, int32_t n_side, RowMap map,
                                 uint8_t *__restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t v = q[i];
    flag[i] = map.owns(v >= 0 && v < n_side ? v : 0) ? 1 : 0;
}

// Empty lists: id -1, score NaN.
__global__ void empty_lists_kernel(int32_t *__restrict__ ids, double *__restrict__ scores, int64_t cnt) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cnt) return;
    ids[i] = -1;
    scores[i] = __longlong_as_double(0x7ff8000000000001ll);
}

// Sharded lists: list b of the staging buffer goes to row rows[b] (else row0 + b) of the output; slab columns are
// local rows for right queries and become global ids here (the map keeps their order).
__global__ void place_lists_kernel(const int32_t *__restrict__ src_ids, const double *__restrict__ src_scores,
                                   int32_t n_top, const int32_t *__restrict__ rows, int64_t row0, int32_t map_ids,
                                   RowMap map, int32_t *__restrict__ ids, double *__restrict__ scores) {
    const int64_t b = blockIdx.x;
    const int64_t o = (rows ? (int64_t)rows[b] : row0 + b) * n_top;
    for (int t = threadIdx.x; t < n_top; t += blockDim.x) {
        int32_t id = src_ids[b * n_top + t];
        if (map_ids && id >= 0) id = (int32_t)map.global(id);
        ids[o + t] = id;
        scores[o + t] = src_scores[b * n_top + t];
    }
}

template <int R>
int32_t launch_scores(const PredArgs &a, const RecArgs &ra, unsigned blocks, size_t smem, int scap, cudaStream_t st) {
    auto kern = recommend_kernel<R>;
    RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<blocks, SEL_WARPS * 32, smem, st>>>(a, ra, scap);
    return RS_OK;
}

// Given lists of one batch: the lists (right queries: the candidate CSR), and for left queries the S* rows and the
// statistics arrays that hold the queries' own after the fitted rows'.
struct GivenBatch {
    const int64_t *ptr;
    const int32_t *ids;
    const double *vals;
    int64_t max_len;
    const double *means, *stddevs;
};

// Runs the scores of `ra`, then sets the rated targets to NaN.  g: the batch's given lists (ra.given).
int32_t score_rows(rs_knn *h, RecArgs ra, const GivenBatch *g = nullptr) {
    if (ra.nq <= 0 || ra.n_targets <= 0) return RS_OK;    // a shard without rows scores nothing
    const bool right = ra.side == RS_SIDE_RIGHT;
    PredArgs a{};
    a.r_ptr = h->r_ptr; a.r_col = h->r_col; a.r_val = h->r_val;
    a.sims = h->sims; a.ld_s = h->ld_s;
    a.means = h->means; a.stddevs = h->stddevs; a.bias = h->left_bias;
    int64_t max_cand = h->max_right_len;
    if (g && right) {                                     // the lists are the candidates
        a.r_ptr = g->ptr; a.r_col = g->ids; a.r_val = g->vals;
        max_cand = g->max_len;
    } else if (g) {
        a.means = g->means; a.stddevs = g->stddevs;
    }
    a.global_mean = h->global_mean; a.n_right = h->n_right;
    a.k = h->p.k; a.min_k = h->p.min_k; a.knn_type = h->p.knn_type;
    void *work;
    RS_TRY(rs_scratch_get(h, RS_SCR_WORK, 8, &work));
    RS_CUDA(cudaMemsetAsync(work, 0, 8, h->stream));
    ra.work = reinterpret_cast<unsigned long long *>(work);
    a.work = ra.work;

    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    // the same per-warp stage as Predict (select.cuh): 256 keys in shared memory, the rest in a global slice
    const int scap = 256;
    const size_t smem = (size_t)SEL_WARPS * scap * sizeof(double);
    const int64_t warps = ra.nq * ra.n_targets;
    int64_t blocks = (int64_t)sms * ((200 * 1024) / (int64_t)(smem + 16 * 1024));   // resident CTAs, as Predict sizes them
    if (blocks > (warps + SEL_WARPS - 1) / SEL_WARPS) blocks = (warps + SEL_WARPS - 1) / SEL_WARPS;
    const int64_t gcap = max_cand > scap ? ((max_cand - scap + 31) / 32 * 32) : 32;
    void *gst;
    RS_TRY(rs_scratch_get(h, RS_SCR_KEY_SPILL, (size_t)blocks * SEL_WARPS * (size_t)gcap * 8, &gst));
    a.gstage = reinterpret_cast<uint64_t *>(gst);
    a.gcap = gcap;
    if (h->p.k <= 44) RS_TRY(launch_scores<2>(a, ra, (unsigned)blocks, smem, scap, h->stream));
    else if (h->p.k <= 104) RS_TRY(launch_scores<4>(a, ra, (unsigned)blocks, smem, scap, h->stream));
    else RS_TRY(launch_scores<8>(a, ra, (unsigned)blocks, smem, scap, h->stream));
    if (g) recommend_exclude_kernel<<<(unsigned)ra.nq, 128, 0, h->stream>>>(ra, g->ptr, g->ids);
    else recommend_exclude_kernel<<<(unsigned)ra.nq, 128, 0, h->stream>>>(ra, right ? h->r_ptr : h->l_ptr,
                                                                          right ? h->r_col : h->l_col);
    h->prof.total_launches += 2;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

}  // namespace

// Rows per batch of a slab of `width` doubles per row: ~256 MiB.
int64_t slab_batch(int64_t width, int64_t n) {
    int64_t batch = ((int64_t)256 << 20) / (width * 8);
    if (const char *e = getenv("RS_KNN_REC_BATCH")) batch = atoll(e);   // tests: force several batches
    if (batch < 1) batch = 1;
    if (batch > n) batch = n;
    return batch;
}

namespace {

// Left queries on a row shard: the queries this shard answers (values and positions), compacted; their count is read
// back to size the batches.
int32_t own_queries(rs_knn *h, const int32_t *d_q, int64_t n, const int32_t **q_own, const int32_t **pos,
                    int64_t *n_own) {
    void *flag, *qo, *po, *cnt, *tmp;
    RS_TRY(rs_scratch_get(h, RS_SCR_OWN_FLAG, (size_t)n, &flag));
    RS_TRY(rs_scratch_get(h, RS_SCR_OWN_QUERIES, (size_t)n * 4, &qo));
    RS_TRY(rs_scratch_get(h, RS_SCR_OWN_POS, (size_t)n * 4, &po));
    RS_TRY(rs_scratch_get(h, RS_SCR_OWN_COUNT, 8, &cnt));
    const cub::CountingInputIterator<int32_t> iota(0);
    size_t need_q = 0, need_p = 0;
    RS_CUDA(cub::DeviceSelect::Flagged(nullptr, need_q, d_q, (const uint8_t *)flag, (int32_t *)qo, (int32_t *)cnt,
                                       (int)n, h->stream));
    RS_CUDA(cub::DeviceSelect::Flagged(nullptr, need_p, iota, (const uint8_t *)flag, (int32_t *)po, (int32_t *)cnt,
                                       (int)n, h->stream));
    const size_t need = need_q > need_p ? need_q : need_p;
    RS_TRY(rs_scratch_get(h, RS_SCR_OWN_TMP, need + 256, &tmp));
    own_query_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(d_q, n, h->n_left, row_map(h),
                                                                          (uint8_t *)flag);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    size_t t_bytes = need;
    RS_CUDA(cub::DeviceSelect::Flagged(tmp, t_bytes, d_q, (const uint8_t *)flag, (int32_t *)qo, (int32_t *)cnt, (int)n,
                                       h->stream));
    t_bytes = need;
    RS_CUDA(cub::DeviceSelect::Flagged(tmp, t_bytes, iota, (const uint8_t *)flag, (int32_t *)po, (int32_t *)cnt, (int)n,
                                       h->stream));
    int32_t c = 0;
    RS_CUDA(cudaMemcpyAsync(&c, cnt, 4, cudaMemcpyDeviceToHost, h->stream));
    RS_CUDA(cudaStreamSynchronize(h->stream));
    *q_own = (const int32_t *)qo;
    *pos = (const int32_t *)po;
    *n_own = c;
    return RS_OK;
}

int32_t empty_lists(rs_knn *h, int32_t *d_ids, double *d_scores, int64_t cnt) {
    empty_lists_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, h->stream>>>(d_ids, d_scores, cnt);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

}  // namespace

// Every recommendation entry point (api.cu, after its checks): resolve the queries, choose one batch size, then per
// batch the S* rows of left lists, the scores, and for list outputs topk_rows_kernel, written directly or, on a row
// shard, staged and placed.
int32_t rs_recommend_run(rs_knn *h, const rs_rec_call &c) {
    if (c.n <= 0) return RS_OK;
    const bool left = c.side == RS_SIDE_LEFT;
    const int64_t n_targets = rs_n_targets(h, c.side);
    // 1. the queries: q[0 .. n) (a shard's left queries: the ones it answers, their rows pos[b]) or the lists gl, and
    //    `width`, the targets scored per query
    const int32_t *q = c.queries, *pos = nullptr;
    int64_t n = c.n, width = n_targets;
    if (c.sharded) {
        // every cell this shard does not answer is +0.0 (all bits zero), for an integer SUM all-reduce; every list it
        // does not produce is empty
        if (!c.lists) RS_CUDA(cudaMemsetAsync(c.rows, 0, (size_t)n * n_targets * 8, h->stream));
        if (left) {
            RS_TRY(own_queries(h, c.queries, c.n, &q, &pos, &n));
            if (c.lists) RS_TRY(empty_lists(h, c.top_ids, c.top_scores, c.n * c.n_top));
        } else {
            width = h->rows_local;
            if (width == 0) return c.lists ? empty_lists(h, c.top_ids, c.top_scores, c.n * c.n_top) : RS_OK;
        }
        if (n == 0) return RS_OK;
    }
    rs_given_lists gl{};
    GivenBatch g{};
    const double *qpmeans = nullptr;
    if (c.given) {
        RS_TRY(rs_given_prepare(h, (int32_t)n_targets, c.ptr, c.ids, c.vals, n, &gl));
        g.ids = gl.ids; g.vals = gl.vals; g.max_len = gl.max_len;
        if (left) {   // the statistics arrays: the fitted rows' followed by the lists'
            void *m, *sd, *pm;
            const size_t rows = (size_t)h->n_left + (size_t)n;
            RS_TRY(rs_scratch_get(h, RS_SCR_GIVEN_MEANS, rows * 8, &m));
            RS_TRY(rs_scratch_get(h, RS_SCR_GIVEN_STDDEVS, rows * 8, &sd));
            RS_TRY(rs_scratch_get(h, RS_SCR_GIVEN_PMEANS, (size_t)n * 8, &pm));
            RS_CUDA(cudaMemcpyAsync(m, h->means, (size_t)h->n_left * 8, cudaMemcpyDeviceToDevice, h->stream));
            RS_CUDA(cudaMemcpyAsync(sd, h->stddevs, (size_t)h->n_left * 8, cudaMemcpyDeviceToDevice, h->stream));
            // core/knn.go:167-177 over the caller's order; Pearson's mean over ascending ids (core/sim.go:49-54)
            RS_TRY(rs_row_stats_launch(h, gl.ptr, gl.vals_in, gl.vals, n, h->p.knn_type == RS_KNN_ZSCORE,
                                       (double *)m + h->n_left, (double *)sd + h->n_left, (double *)pm));
            g.means = (const double *)m; g.stddevs = (const double *)sd;
            qpmeans = (const double *)pm;
        }
    }
    // 2. the batch: score rows by id go to the caller's rows in one pass; everything else is scored in batches, into
    //    a slab of `width` columns for lists and, for left lists, the S* slab beside it (~256 MiB together)
    const int64_t batch = !c.lists && !c.given ? n : slab_batch(width + (c.given && left ? h->n_left : 0), n);
    void *slab = nullptr, *st_ids = nullptr, *st_scores = nullptr, *sslab = nullptr;
    if (c.lists) RS_TRY(rs_scratch_get(h, RS_SCR_REC_SLAB, (size_t)batch * width * 8, &slab));
    if (c.lists && c.sharded) {
        RS_TRY(rs_scratch_get(h, RS_SCR_REC_STAGE_IDS, (size_t)batch * c.n_top * 4, &st_ids));
        RS_TRY(rs_scratch_get(h, RS_SCR_REC_STAGE_SCORES, (size_t)batch * c.n_top * 8, &st_scores));
    }
    if (c.given && left) RS_TRY(rs_scratch_get(h, RS_SCR_GIVEN_SIMS, (size_t)batch * h->n_left * 8, &sslab));
    // 3. one loop
    for (int64_t b0 = 0; b0 < n; b0 += batch) {
        const int64_t nb = n - b0 < batch ? n - b0 : batch;
        RecArgs ra{};
        ra.queries = q ? q + b0 : nullptr; ra.nq = nb; ra.side = c.side;
        ra.n_side = left ? h->n_left : h->n_right;
        ra.n_targets = (int32_t)width;
        ra.map = row_map(h);
        ra.out = c.lists ? (double *)slab : c.rows + b0 * n_targets;
        ra.ld_out = c.lists ? width : n_targets;
        if (!c.lists && c.sharded) {       // a shard's rows: left queries to their rows, right targets to global columns
            ra.rows = pos;
            ra.out_global = !left;
        }
        if (c.given) {
            ra.given = 1;
            g.ptr = gl.ptr + b0;
            if (left) {
                RS_TRY(rs_given_sims_launch(h, g.ptr, gl.ids, gl.vals, qpmeans + b0, nb, (double *)sslab, h->n_left));
                ra.gsims = (const double *)sslab;
                ra.ld_g = h->n_left;
                ra.qstat = (int32_t)(h->n_left + b0);
            }
        }
        RS_TRY(score_rows(h, ra, c.given ? &g : nullptr));
        if (!c.lists) continue;
        if (!c.sharded) {
            RS_TRY(rs_topk_rows_launch(h, (const double *)slab, width, (int32_t)width, nb, c.n_top,
                                       c.top_ids + b0 * c.n_top, c.top_scores + b0 * c.n_top));
            continue;
        }
        RS_TRY(rs_topk_rows_launch(h, (const double *)slab, width, (int32_t)width, nb, c.n_top, (int32_t *)st_ids,
                                   (double *)st_scores));
        place_lists_kernel<<<(unsigned)nb, 128, 0, h->stream>>>((const int32_t *)st_ids, (const double *)st_scores,
                                                                c.n_top, pos ? pos + b0 : nullptr, b0, !left,
                                                                row_map(h), c.top_ids, c.top_scores);
        h->prof.total_launches++;
        RS_CUDA(cudaGetLastError());
    }
    return RS_OK;
}
