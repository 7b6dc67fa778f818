// given.cu — queries given as rating lists (rs_knn_score_all_given / rs_knn_recommend_given): the preparation of the
// lists and, for user-based (left) queries, the similarity row of each list against every fitted left row.
//
// A list plays the role of a right row (item-based: its entries are the candidates of every target) or of a left row
// (user-based: it is one more row of the similarity matrix).  The scoring itself is recommend_kernel (recommend.cu)
// on those candidates / that row; nothing of the fitted model changes.
//
// given_sims_kernel: S*[b][v] = Sim(list b sorted by id, L(v)) for every fitted left row v, bit for bit what the
// reference's Sim (core/sim.go) returns for the pair: the terms of one pair arrive in ascending right id c, each with
// the IEEE operations of the exact sparse Fit (stream_update / sim_value, sim_terms.cuh).
//   work item: (list b, block of GS_JC consecutive left rows), one warp, the block's accumulators in shared memory.
//   The warp walks list b in ascending c; the raters of c inside the block are a contiguous slice of c's id-sorted
//   list in the right CSR, found by two binary searches (one lane per entry, 32 entries at a time), and the lanes
//   update the accumulators of those raters — every v at most once per c, c strictly in order.
//   It reads r_ptr / r_col / r_val and pmeans, which every RS_STORE_MATRIX handle holds (tensor-path Fits too).
// given_sims_kernel<SIM, true>: the same values for the rows a cyclic row shard owns only, S*[b][loc] = Sim(list b,
// L(v)) at v's local row loc (rs_knn_update_sharded_device: the columns a shard stores of rows it does not own).  A
// work item is a block of GS_JC consecutive local rows; its raters are found over the global id range the block
// spans, and the raters of other shards are skipped.  Every v still sees its entries c in ascending order.
#include <cub/cub.cuh>

#include "common.cuh"
#include "sim_terms.cuh"

namespace {

constexpr int GS_JC = 256;     // left rows per work item
constexpr int GS_WARPS = 8;

// ptr checks (one thread per list boundary): the lists rebased to entry 0, hdr = {ptr[0], ptr[n], bad, longest}
__global__ void given_ptr_kernel(const int64_t *__restrict__ ptr, int64_t n, int64_t *__restrict__ gp,
                                 unsigned long long *__restrict__ hdr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    const int64_t p0 = ptr[0];
    gp[i] = ptr[i] - p0;
    if (i == 0) {
        hdr[0] = (unsigned long long)p0;
        hdr[1] = (unsigned long long)ptr[n];
        if (p0 < 0) atomicOr(&hdr[2], 1ull);
    }
    if (i < n) {
        const int64_t len = ptr[i + 1] - ptr[i];
        if (len < 0) atomicOr(&hdr[2], 1ull);
        else atomicMax(&hdr[3], (unsigned long long)len);
    }
}

// entry checks on the sorted lists (one block per list): flags[0] an id outside [0, n_targets) or a NaN rating,
// flags[1] an id twice in one list
__global__ void given_check_kernel(const int64_t *__restrict__ gp, const int32_t *__restrict__ ids,
                                   const double *__restrict__ vals, int32_t n_targets, int32_t *__restrict__ flags) {
    const int64_t b = blockIdx.x;
    const int64_t eb = gp[b], ee = gp[b + 1];
    for (int64_t e = eb + threadIdx.x; e < ee; e += blockDim.x) {
        const int32_t id = ids[e];
        const double v = vals[e];
        if (id < 0 || id >= n_targets || v != v) flags[0] = 1;
        if (e > eb && ids[e - 1] == id) flags[1] = 1;
    }
}

struct GivenSimArgs {
    const int64_t *ptr;       // list b: entries ptr[b] .. ptr[b+1) of ids / vals, ascending right id
    const int32_t *ids;
    const double *vals;
    const double *qpmeans;    // Pearson: each list's own mean, summed in ascending id order (core/sim.go:49-54)
    const int32_t *rows;      // list b is list rows[b] of ptr / qpmeans (null: list b)
    int64_t nq;
    const int64_t *r_ptr;
    const int32_t *r_col;
    const double *r_val;
    const double *pmeans;     // Pearson: the fitted rows' own means
    int32_t n_left, n_blk;
    double *out;              // [nq][ld]
    int64_t ld;
    unsigned long long *counter;
    int32_t cyc_R, cyc_r;     // OWN: the shard; n_left / n_blk count its local rows
    uint32_t cyc_div;         // ceil(2^32 / cyc_R): __umulhi(blk, cyc_div) = blk / cyc_R for every block blk < 2^26
};

template <int SIM, bool OWN = false>
__global__ void __launch_bounds__(GS_WARPS * 32) given_sims_kernel(GivenSimArgs a) {
    extern __shared__ double s_gs[];                  // [GS_WARPS][3][GS_JC] accumulators, then [GS_WARPS][32] a-side terms
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *acc = s_gs + (size_t)warp * 3 * GS_JC;
    double *s_ra = s_gs + (size_t)GS_WARPS * 3 * GS_JC + warp * 32;
    const int64_t n_items = a.nq * a.n_blk;
    for (;;) {
        unsigned long long item = 0;
        if (lane == 0) item = atomicAdd(a.counter, 1ull);
        item = __shfl_sync(0xffffffffu, item, 0);
        if ((int64_t)item >= n_items) break;
        const int64_t b = (int64_t)item / a.n_blk;    // list-major: the warps in flight walk the same list
        // OWN: local rows [l0, l1) of the shard, the global ids v0 .. v1-1 they span; else v0 .. v1-1 themselves
        const int32_t l0 = (int32_t)((int64_t)item % a.n_blk) * GS_JC;
        const int32_t l1 = l0 + GS_JC < a.n_left ? l0 + GS_JC : a.n_left;
        const int32_t v0 = OWN ? (int32_t)rs_cyc_global(l0, a.cyc_R, a.cyc_r) : l0;
        const int32_t v1 = OWN ? (int32_t)rs_cyc_global(l1 - 1, a.cyc_R, a.cyc_r) + 1 : l1;
        __syncwarp();                                 // the previous item has finished with acc
        for (int x = lane; x < 3 * GS_JC; x += 32) acc[x] = 0.0;
        const int64_t lb = a.rows ? a.rows[b] : b;
        const double aq = SIM == RS_SIM_PEARSON ? a.qpmeans[lb] : 0.0;
        const int64_t eb = a.ptr[lb], ee = a.ptr[lb + 1];
        for (int64_t x0 = eb; x0 < ee; x0 += 32) {
            // each lane prepares one entry (c, x) of the list: its a-side term and the slice of c's raters in [v0, v1)
            const int64_t e = x0 + lane;
            double ra = 0.0;
            int64_t lo = 0;
            int n = 0;
            if (e < ee) {
                const int32_t c = a.ids[e];
                const double x = a.vals[e];
                ra = SIM == RS_SIM_PEARSON ? x - aq : x;                          // core/sim.go:73
                const int64_t cb = a.r_ptr[c], ce = a.r_ptr[c + 1];
                lo = lower_bound_id(a.r_col, cb, ce, v0);
                n = (int)(lower_bound_id(a.r_col, lo, ce, v1) - lo);
            }
            __syncwarp();
            s_ra[lane] = ra;
            __syncwarp();
            const int lim = (ee - x0) < 32 ? (int)(ee - x0) : 32;
            for (int u = 0; u < lim; u++) {
                const int nn = __shfl_sync(0xffffffffu, n, u);
                const int64_t lo_u = __shfl_sync(0xffffffffu, lo, u);
                if (nn == 0) continue;                                            // warp-uniform
                const double ra_u = s_ra[u];
                const double raa_u = ra_u * ra_u;                                 // core/sim.go:19 / :75
                for (int t = lane; t < nn; t += 32) {
                    const int32_t v = a.r_col[lo_u + t];
                    int32_t j = v - v0;
                    if (OWN) {                                                    // rs_cyc_owns / rs_cyc_local
                        const uint32_t blk = (uint32_t)v / RS_CYC_B, q = __umulhi(blk, a.cyc_div);
                        j = blk - q * a.cyc_R == (uint32_t)a.cyc_r ? (int32_t)(q * RS_CYC_B + (uint32_t)v % RS_CYC_B) - l0
                                                                   : -1;
                    }
                    if (!OWN || j >= 0) {
                        double rb = a.r_val[lo_u + t];
                        if (SIM == RS_SIM_PEARSON) rb = rb - a.pmeans[v];         // core/sim.go:74, as build_rdev_kernel
                        stream_update<SIM, false, GS_JC>(acc, j, ra_u, raa_u, rb);
                    }
                }
                __syncwarp();   // entry c is complete before entry c+1 touches the same v
            }
        }
        __syncwarp();
        double *out = a.out + b * a.ld;
        for (int j = lane; j < l1 - l0; j += 32)
            out[l0 + j] = sim_value<SIM, false>(acc + j, GS_JC, 0.0);
    }
}

template <int SIM>
int32_t launch_given_sims(rs_knn *h, const GivenSimArgs &a, bool own) {
    const size_t smem = (size_t)GS_WARPS * (3 * GS_JC + 32) * sizeof(double);
    auto kern = own ? given_sims_kernel<SIM, true> : given_sims_kernel<SIM>;
    RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    int per_sm = 1;
    RS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, GS_WARPS * 32, smem));
    if (per_sm < 1) per_sm = 1;
    int64_t blocks = (int64_t)sms * per_sm;
    const int64_t need = (a.nq * a.n_blk + GS_WARPS - 1) / GS_WARPS;
    if (blocks > need) blocks = need;
    kern<<<(unsigned)blocks, GS_WARPS * 32, smem, h->stream>>>(a);
    return RS_OK;
}

}  // namespace

int32_t rs_given_prepare(rs_knn *h, int32_t n_targets, const int64_t *d_ptr, const int32_t *d_ids,
                         const double *d_vals, int64_t n, rs_given_lists *out) {
    void *hdr, *gp, *flags;
    RS_TRY(rs_scratch_get(h, RS_SCR_GIVEN_HDR, 64, &hdr));
    RS_TRY(rs_scratch_get(h, RS_SCR_GIVEN_PTR, (size_t)(n + 1) * 8, &gp));
    flags = (char *)hdr + 32;
    RS_CUDA(cudaMemsetAsync(hdr, 0, 64, h->stream));
    given_ptr_kernel<<<(unsigned)((n + 1 + 255) / 256), 256, 0, h->stream>>>(d_ptr, n, (int64_t *)gp,
                                                                              (unsigned long long *)hdr);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    unsigned long long hh[4];
    RS_CUDA(cudaMemcpyAsync(hh, hdr, 32, cudaMemcpyDeviceToHost, h->stream));
    RS_CUDA(cudaStreamSynchronize(h->stream));
    const int64_t p0 = (int64_t)hh[0], nnz = (int64_t)hh[1] - p0;
    if (hh[2]) {
        rs_set_error("rs_knn_*_given: ptr must start at >= 0 and be non-decreasing");
        return RS_ERR_INVALID;
    }
    if (nnz >= (1ll << 31)) {
        rs_set_error("rs_knn_*_given: %lld entries (at most 2^31 - 1 per call)", (long long)nnz);
        return RS_ERR_UNSUPPORTED;
    }
    out->ptr = (const int64_t *)gp;
    out->nnz = nnz;
    out->max_len = (int64_t)hh[3];
    out->vals_in = d_vals + p0;
    out->ids = nullptr;
    out->vals = nullptr;
    if (nnz == 0) return RS_OK;
    // sort each list by id (stable; plumbing, not the hot path), then check the sorted entries
    void *s_ids, *s_vals, *tmp;
    RS_TRY(rs_scratch_get(h, RS_SCR_GIVEN_IDS, (size_t)nnz * 4, &s_ids));
    RS_TRY(rs_scratch_get(h, RS_SCR_GIVEN_VALS, (size_t)nnz * 8, &s_vals));
    size_t need = 0;
    RS_CUDA(cub::DeviceSegmentedSort::StableSortPairs(nullptr, need, d_ids + p0, (int32_t *)s_ids, d_vals + p0,
                                                       (double *)s_vals, (int)nnz, (int)n, (const int64_t *)gp,
                                                       (const int64_t *)gp + 1, h->stream));
    RS_TRY(rs_scratch_get(h, RS_SCR_GIVEN_SORT_TMP, need + 256, &tmp));
    RS_CUDA(cub::DeviceSegmentedSort::StableSortPairs(tmp, need, d_ids + p0, (int32_t *)s_ids, d_vals + p0,
                                                       (double *)s_vals, (int)nnz, (int)n, (const int64_t *)gp,
                                                       (const int64_t *)gp + 1, h->stream));
    given_check_kernel<<<(unsigned)n, 128, 0, h->stream>>>((const int64_t *)gp, (const int32_t *)s_ids,
                                                           (const double *)s_vals, n_targets, (int32_t *)flags);
    h->prof.total_launches += 2;
    RS_CUDA(cudaGetLastError());
    int32_t f[2];
    RS_CUDA(cudaMemcpyAsync(f, flags, 8, cudaMemcpyDeviceToHost, h->stream));
    RS_CUDA(cudaStreamSynchronize(h->stream));
    if (f[0]) {
        rs_set_error("rs_knn_*_given: an id outside [0, %d) or a NaN rating", n_targets);
        return RS_ERR_INVALID;
    }
    if (f[1]) {
        rs_set_error("rs_knn_*_given: an id appears twice in one list");
        return RS_ERR_DUPLICATE;
    }
    out->ids = (const int32_t *)s_ids;
    out->vals = (const double *)s_vals;
    return RS_OK;
}

int32_t rs_given_sims_launch(rs_knn *h, const int64_t *ptr, const int32_t *ids, const double *vals,
                             const double *qpmeans, int64_t nq, double *out, int64_t ld, const int32_t *rows,
                             bool own) {
    const int64_t width = own ? h->rows_local : h->n_left;
    if (nq <= 0 || width <= 0) return RS_OK;
    void *counter;
    RS_TRY(rs_scratch_get(h, RS_SCR_GIVEN_COUNTER, 8, &counter));
    RS_CUDA(cudaMemsetAsync(counter, 0, 8, h->stream));
    GivenSimArgs a{};
    a.ptr = ptr; a.ids = ids; a.vals = vals; a.qpmeans = qpmeans; a.rows = rows; a.nq = nq;
    a.r_ptr = h->r_ptr; a.r_col = h->r_col; a.r_val = h->r_val; a.pmeans = h->pmeans;
    a.n_left = (int32_t)width;
    a.n_blk = (int32_t)((width + GS_JC - 1) / GS_JC);
    a.out = out; a.ld = ld;
    a.counter = reinterpret_cast<unsigned long long *>(counter);
    a.cyc_R = h->cyc_R; a.cyc_r = h->cyc_r;
    if (own) a.cyc_div = (uint32_t)(((1ull << 32) + h->cyc_R - 1) / h->cyc_R);
    if (h->p.sim == RS_SIM_COSINE) RS_TRY(launch_given_sims<RS_SIM_COSINE>(h, a, own));
    else if (h->p.sim == RS_SIM_MSD) RS_TRY(launch_given_sims<RS_SIM_MSD>(h, a, own));
    else if (h->p.sim == RS_SIM_PEARSON) RS_TRY(launch_given_sims<RS_SIM_PEARSON>(h, a, own));
    else {
        rs_set_error("rs_knn_*_given: no similarity row for sim %d", h->p.sim);
        return RS_ERR_UNSUPPORTED;
    }
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}
