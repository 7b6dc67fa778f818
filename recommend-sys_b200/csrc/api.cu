// api.cu — the C ABI of include/rs_knn.h: handle lifetime, Fit / Predict orchestration.
// No CPU fallback anywhere: every compute entry point needs a CUDA device.
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>

#include "common.cuh"

static thread_local char g_err[512] = "";

void rs_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

namespace {

int32_t enter(rs_knn *h) {
    if (!h) {
        rs_set_error("null handle");
        return RS_ERR_INVALID;
    }
    // goroutines migrate between OS threads: bind the device on every entry
    RS_CUDA(cudaSetDevice(h->device));
    return RS_OK;
}

// Entry points on ONE handle are serialised: they share the handle's stream, staging buffers and
// event pairs (the reference's Predict is read-only and may be called from several goroutines,
// core/knn.go:75-141).  Recursive because host-pointer entry points call their _device variants.
struct Guard {
    std::unique_lock<std::recursive_mutex> lk;
    explicit Guard(rs_knn *h) { if (h) lk = std::unique_lock<std::recursive_mutex>(h->mu); }
};
#define RS_ENTER(h) Guard guard_(h); RS_TRY(enter(h))

// Forget the fitted state; the arena's chunks are kept for the next Fit.
void free_fit_state(rs_knn *h) {
    h->cur_chunk = 0;
    h->cur_off = 0;
    h->fitted = false;
    h->l_ptr = h->r_ptr = nullptr;
    h->l_col = h->r_col = nullptr;
    h->l_val = h->r_val = h->ld_val = nullptr;
    h->l_code = nullptr;
    h->means = h->stddevs = h->pmeans = h->left_bias = h->right_bias = nullptr;
    h->r_dev = nullptr;
    h->rd_col = nullptr;
    h->right_means = nullptr;
    h->cp = nullptr;
    h->l2r = nullptr;
    h->row_order = nullptr;
    h->row_heavy = nullptr;
    h->n_heavy = 0;
    h->n_pop = h->pop_ld = 0;
    h->rank = h->lab_row = h->pop_items = nullptr;
    h->pop_dense = nullptr;
    h->w_ptr = nullptr;
    h->w_col = nullptr;
    h->w_dev = nullptr;
    h->row_all = nullptr;
    h->n_all_rows = 0;
    h->planes = nullptr;
    h->row_cnt = h->row_sum = nullptr;
    h->sims = nullptr;
    h->topk_idx = nullptr;
    h->topk_sim = nullptr;
    h->thr_key = nullptr;
    h->thr_id = nullptr;
    h->cand_cnt = nullptr;
    h->cand_id = nullptr;
    h->cand_sim = nullptr;
    h->row_flag = nullptr;
    h->d_flags = nullptr;
    rs_update_release(h);
}

int32_t fold_profile(rs_knn *h) {
    RS_CUDA(cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    if (h->prep_pending) {
        RS_CUDA(cudaEventElapsedTime(&ms, h->ev_a, h->ev_b));
        h->prof.prep_ms += ms;
        h->prep_pending = false;
    }
    if (h->sim_pending) {
        RS_CUDA(cudaEventElapsedTime(&ms, h->ev_b, h->ev_c));
        h->prof.sim_kernel_ms += ms;
        h->sim_pending = false;
    }
    if (h->pred_pending) {
        RS_CUDA(cudaEventElapsedTime(&ms, h->ev_d, h->ev_e));
        h->prof.predict_kernel_ms += ms;
        h->pred_pending = false;
    }
    return RS_OK;
}

bool tensor_eligible(const rs_knn *h) {
    if (h->rating_class != RS_CLASS_INT8) return false;
    if (h->p.sim == RS_SIM_COSINE || h->p.sim == RS_SIM_MSD || h->p.sim == RS_SIM_SLOPE_ONE) return true;
    if (h->p.sim == RS_SIM_PEARSON && h->p.pearson_mode == RS_PEARSON_SUMS) return true;
    return false;
}

// Fit path model.  Both paths are bit-exact for Cosine / MSD, so RS_PATH_AUTO takes the faster one.
// The tensor path does dense work, N(N-1)/2 * 2*G*K int8 ops whatever the sparsity; the stream
// path does one step per co-rated triple.  Rates measured on B200 (profiles/r01_path_model.md):
// tensor ~2.0e15 op/s sustained (0.62-0.9 of the int8 roofline), stream 6e10-9e10 triples/s.  Dense
// shapes (MovieLens-1M, 4.5 % filled) go to the tensor cores, sparse ones (MovieLens-20M, 0.5 %)
// are faster as an exact sparse replay.
bool tensor_faster(const rs_knn *h) {
    const double n = (double)h->n_left, rows = (double)(h->row_end - h->row_begin);
    const bool full = h->row_begin == 0 && h->row_end == h->n_left;
    const double g = h->p.sim == RS_SIM_COSINE ? 3.0 : h->p.sim == RS_SIM_MSD ? 4.0 : 6.0;
    const double pairs = full ? n * (n - 1.0) / 2.0 : rows * n;           // a row shard computes full rows
    const double t_tensor = pairs * 2.0 * g * (double)h->n_right / 2.0e15 + 1e-4;
    const double triples = full ? h->triples : 2.0 * h->triples * (rows / n);
    const double t_stream = triples / 6.0e10 + 1e-4;
    return t_tensor <= t_stream;
}

// Peer matrices are mapped once per process and device: estimator copies are created and destroyed per
// fold / per Fit, but their arenas come out of the block cache (devmem.cu), so the same allocations — and
// the same IPC handles — come back; opening a multi-GB mapping costs milliseconds.
struct IpcMap { int device; unsigned char handle[64]; void *base; };
std::mutex g_ipc_mu;
std::vector<IpcMap> g_ipc;

int32_t ipc_open_cached(int device, const unsigned char *hb, void **base) {
    std::lock_guard<std::mutex> lk(g_ipc_mu);
    for (const auto &m : g_ipc)
        if (m.device == device && !std::memcmp(m.handle, hb, 64)) { *base = m.base; return RS_OK; }
    cudaIpcMemHandle_t mh;
    std::memcpy(&mh, hb, 64);
    RS_CUDA(cudaIpcOpenMemHandle(base, mh, cudaIpcMemLazyEnablePeerAccess));
    IpcMap m;
    m.device = device;
    std::memcpy(m.handle, hb, 64);
    m.base = *base;
    g_ipc.push_back(m);
    return RS_OK;
}

int32_t init_handle(rs_knn *h) {
    RS_CUDA(cudaSetDevice(h->device));
    RS_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    RS_CUDA(cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
    RS_CUDA(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
    RS_CUDA(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    RS_CUDA(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    h->stream = h->own_stream;
    RS_CUDA(cudaEventCreate(&h->ev_a));
    RS_CUDA(cudaEventCreate(&h->ev_b));
    RS_CUDA(cudaEventCreate(&h->ev_c));
    RS_CUDA(cudaEventCreate(&h->ev_d));
    RS_CUDA(cudaEventCreate(&h->ev_e));
    return RS_OK;
}

}  // namespace

extern "C" {

const char *rs_last_error(void) { return g_err; }
int32_t rs_knn_abi_version(void) { return 5; }

int32_t rs_knn_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

int32_t rs_knn_params_default(rs_knn_params *p) {
    if (!p) return RS_ERR_INVALID;
    std::memset(p, 0, sizeof(*p));
    p->sim = RS_SIM_MSD;         // core/knn.go:145
    p->knn_type = RS_KNN_BASIC;  // core/knn.go:52
    p->k = 40;                   // core/knn.go:80
    p->min_k = 1;                // core/knn.go:81
    p->device = -1;
    p->pearson_mode = RS_PEARSON_EXACT;
    p->sim_path = RS_PATH_AUTO;
    p->store = RS_STORE_MATRIX;
    p->topk = 40;
    return RS_OK;
}

int32_t rs_knn_create(const rs_knn_params *p, rs_knn **out) {
    if (!p || !out) {
        rs_set_error("rs_knn_create: null argument");
        return RS_ERR_INVALID;
    }
    if (p->sim < RS_SIM_COSINE || p->sim > RS_SIM_SLOPE_ONE || p->knn_type < RS_KNN_BASIC ||
        p->knn_type > RS_KNN_BASELINE || p->k < 1 || p->min_k < 0) {
        rs_set_error("rs_knn_create: invalid sim/knn_type/k/min_k");
        return RS_ERR_INVALID;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        (void)cudaGetLastError();
        rs_set_error("no CUDA device available (%s); this library has no CPU fallback",
                     e == cudaSuccess ? "0 devices" : cudaGetErrorString(e));
        return RS_ERR_CUDA;
    }
    int dev = p->device;
    if (dev < 0) RS_CUDA(cudaGetDevice(&dev));
    if (dev >= ndev) {
        rs_set_error("device %d out of range (%d devices)", dev, ndev);
        return RS_ERR_INVALID;
    }
    int cc_major = 0, cc_minor = 0;   // (cudaGetDeviceProperties costs milliseconds per call)
    RS_CUDA(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, dev));
    RS_CUDA(cudaDeviceGetAttribute(&cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
    if (cc_major != 10) {
        rs_set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", dev, cc_major,
                     cc_minor);
        return RS_ERR_UNSUPPORTED;
    }
    rs_knn *h = new (std::nothrow) rs_knn();
    if (!h) return RS_ERR_OOM;
    h->p = *p;
    h->device = dev;
    const int32_t rc = init_handle(h);
    if (rc != RS_OK) {             // a partially built handle is torn down, not leaked
        rs_knn_destroy(h);
        return rc;
    }
    *out = h;
    return RS_OK;
}

int32_t rs_knn_destroy(rs_knn *h) {
    if (!h) return RS_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    free_fit_state(h);
    for (auto &c : h->chunks) rs_cached_free(h->device, c.p, c.bytes);
    h->chunks.clear();
    if (h->tile_buf) cudaFree(h->tile_buf);
    if (h->band_buf) cudaFree(h->band_buf);
    if (h->ovf) rs_cached_free(h->device, h->ovf, h->ovf_bytes);
    for (size_t i = 0; i < h->scratch.size(); i++) rs_cached_free(h->device, h->scratch[i], h->scratch_bytes[i]);
    if (h->ev_a) cudaEventDestroy(h->ev_a);
    if (h->ev_b) cudaEventDestroy(h->ev_b);
    if (h->ev_c) cudaEventDestroy(h->ev_c);
    if (h->ev_d) cudaEventDestroy(h->ev_d);
    if (h->ev_e) cudaEventDestroy(h->ev_e);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    if (h->aux_stream) cudaStreamDestroy(h->aux_stream);
    if (h->ev_in) cudaEventDestroy(h->ev_in);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    delete h;
    return RS_OK;
}

int32_t rs_knn_set_stream(rs_knn *h, void *cuda_stream, int32_t use_own) {
    RS_ENTER(h);
    RS_CUDA(cudaStreamSynchronize(h->stream));
    // NULL is a real stream (the legacy default stream), so "own" needs its own flag
    h->stream = use_own ? h->own_stream : reinterpret_cast<cudaStream_t>(cuda_stream);
    return RS_OK;
}

int32_t rs_knn_synchronize(rs_knn *h) {
    RS_ENTER(h);
    RS_CUDA(cudaStreamSynchronize(h->stream));
    return RS_OK;
}

int32_t rs_knn_fit_device(rs_knn *h, const int32_t *d_left, const int32_t *d_right, const double *d_rating,
                          int64_t nnz, int32_t n_left, int32_t n_right, double global_mean,
                          const double *d_left_bias, const double *d_right_bias, double global_bias) {
    RS_ENTER(h);
    if (!d_left || !d_right || !d_rating || nnz <= 0 || n_left <= 0 || n_right <= 0) {
        rs_set_error("rs_knn_fit: empty or null input (nnz=%lld n_left=%d n_right=%d)", (long long)nnz, n_left,
                     n_right);
        return RS_ERR_INVALID;
    }
    if (h->p.knn_type == RS_KNN_BASELINE && !d_left_bias) {
        rs_set_error("rs_knn_fit: RS_KNN_BASELINE needs left_bias (core/knn.go:179-187)");
        return RS_ERR_INVALID;
    }
    if (h->p.sim == RS_SIM_PEARSON_BASELINE && (!d_left_bias || !d_right_bias)) {
        rs_set_error("rs_knn_fit: RS_SIM_PEARSON_BASELINE needs both bias vectors");
        return RS_ERR_INVALID;
    }
    RS_TRY(fold_profile(h));
    free_fit_state(h);
    h->nnz = nnz;
    h->n_left = n_left;
    h->n_right = n_right;
    h->global_mean = global_mean;
    h->global_bias = global_bias;
    h->row_begin = h->p.row_begin;
    h->row_end = h->p.row_end;
    if (h->row_begin == 0 && h->row_end == 0) h->row_end = n_left;
    if (h->row_begin < 0 || h->row_end > n_left || h->row_begin > h->row_end) {
        rs_set_error("row shard [%lld,%lld) outside [0,%d)", (long long)h->row_begin, (long long)h->row_end, n_left);
        return RS_ERR_INVALID;
    }
    const int64_t rows = h->row_end - h->row_begin;
    if (h->p.shard_count < 0 || (h->p.shard_count >= 1 && (h->p.shard_index < 0 || h->p.shard_index >= h->p.shard_count))) {
        rs_set_error("shard_index %d outside [0, shard_count=%d)", h->p.shard_index, h->p.shard_count);
        return RS_ERR_INVALID;
    }
    if (h->p.shard_count >= 1 && rows != n_left) {
        rs_set_error("shard_count >= 1 and row_begin/row_end are two different sharding schemes: use one");
        return RS_ERR_INVALID;
    }
    // RS_STORE_MATRIX with shard_count >= 2: CYCLIC ROW SHARDS (see rs_knn_params::shard_count)
    h->cyc_R = (h->p.store == RS_STORE_MATRIX && h->p.shard_count >= 2) ? h->p.shard_count : 0;
    h->cyc_r = h->cyc_R ? h->p.shard_index : 0;
    h->peers_ready = false;
    if (h->cyc_R > RS_MAX_PEERS) {
        rs_set_error("at most %d cyclic row shards", RS_MAX_PEERS);
        return RS_ERR_UNSUPPORTED;
    }
    if (h->cyc_R && h->p.sim == RS_SIM_SLOPE_ONE) {
        rs_set_error("RS_SIM_SLOPE_ONE does not support cyclic row shards (use row_begin/row_end)");
        return RS_ERR_UNSUPPORTED;
    }
    h->rows_local = h->cyc_R ? rs_cyc_rows(n_left, h->cyc_R, h->cyc_r) : rows;

    RS_CUDA(cudaEventRecord(h->ev_a, h->stream));
    int32_t rc = rs_prep_build(h, d_left, d_right, d_rating, d_left_bias, d_right_bias);
    if (rc != RS_OK) { free_fit_state(h); return rc; }

    int path = h->p.sim_path;
    if (const char *force = getenv("RS_KNN_FORCE_PATH")) {  // debugging aid: "stream" | "tensor"
        if (!strcmp(force, "stream")) path = RS_PATH_STREAM;
        else if (!strcmp(force, "tensor")) path = RS_PATH_TENSOR;
    }
    if (h->p.sim == RS_SIM_SLOPE_ONE) {
        // the deviation sums are integer contractions: tensor path only (integer ratings)
        if (!tensor_eligible(h) || path == RS_PATH_STREAM) {
            rs_set_error("RS_SIM_SLOPE_ONE needs integer ratings in [-11,11] (tensor path)");
            free_fit_state(h);
            return RS_ERR_UNSUPPORTED;
        }
        path = RS_PATH_TENSOR;
    }
    if (h->cyc_R) {
        // every pair is computed once by the shard that owns the larger (or smaller) row and the other
        // triangle arrives by rs_knn_mirror: that schedule exists for the exact sparse path only
        if (path == RS_PATH_TENSOR) {
            rs_set_error("cyclic row shards run the stream path; shard the tensor path with row_begin/row_end");
            free_fit_state(h);
            return RS_ERR_UNSUPPORTED;
        }
        path = RS_PATH_STREAM;
    }
    if (path == RS_PATH_AUTO) path = tensor_eligible(h) && tensor_faster(h) ? RS_PATH_TENSOR : RS_PATH_STREAM;
    if (path == RS_PATH_TENSOR && !tensor_eligible(h)) {
        rs_set_error("tensor path needs integer ratings in [-11,11] and Cosine/MSD (or Pearson in SUMS mode)");
        free_fit_state(h);
        return RS_ERR_UNSUPPORTED;
    }
    h->prof.sim_path_used = path;
    h->prof.corated_triples = h->triples;
    rc = (path == RS_PATH_TENSOR) ? rs_prep_planes(h) : rs_prep_rt(h);
    if (rc != RS_OK) { free_fit_state(h); return rc; }

    h->ld_s = ((int64_t)n_left + 15) / 16 * 16;
    if (h->p.store == RS_STORE_MATRIX) {
        rc = rs_alloc(h, &h->sims, (size_t)h->rows_local * (size_t)h->ld_s);
        if (rc != RS_OK) { free_fit_state(h); return rc; }
        RS_CUDA(cudaEventRecord(h->ev_b, h->stream));
        rc = (path == RS_PATH_TENSOR) ? rs_sim_tensor_launch(h, nullptr, 0, 0) : rs_sim_stream_launch(h);
        if (rc != RS_OK) { free_fit_state(h); return rc; }
        RS_CUDA(cudaEventRecord(h->ev_c, h->stream));
        if (path == RS_PATH_STREAM) {
            rc = rs_symmetrize_launch(h);
            if (rc != RS_OK) { free_fit_state(h); return rc; }
        }
    } else if (h->p.shard_count >= 1 && path == RS_PATH_TENSOR && rs_tensor_topk_fused(h)) {
        // top-k only, FUSED: the tensor kernel's epilogue tests every similarity against the current k-th
        // best of its two rows and appends the survivors to per-row candidate buffers; the buffers are merged
        // into the running lists between the waves of the tile schedule (sim_tensor.cu).  No similarity row,
        // slab or transpose is ever written: the only N-proportional buffers are the lists (N x k) and the
        // candidate buffers (N x cap).  Every pair is computed once; a multi-GPU Fit deals the tiles of each
        // wave to the shards, every shard ends with PARTIAL lists for all rows (united after an all-gather).
        const int32_t k = h->p.topk > 0 ? h->p.topk : h->p.k;
        const int64_t n = n_left;
        h->cand_cap = 1792;                          // band 0 brings at most 2 * (512 + 256) entries per row
        if (const char *e = getenv("RS_KNN_TOPK_CAP")) h->cand_cap = atoi(e);   // tests: force the overflow path
        if (k > 256 || h->cand_cap + k > 2048 || h->cand_cap < 1) {
            rs_set_error("fused top-k: k <= 256 and candidate capacity + k <= 2048 (k=%d cap=%d)", k, h->cand_cap);
            free_fit_state(h);
            return RS_ERR_UNSUPPORTED;
        }
        RS_TRY(rs_alloc(h, &h->topk_idx, (size_t)n * k));
        RS_TRY(rs_alloc(h, &h->topk_sim, (size_t)n * k));
        RS_TRY(rs_alloc(h, &h->thr_key, (size_t)n));
        RS_TRY(rs_alloc(h, &h->thr_id, (size_t)n));
        RS_TRY(rs_alloc(h, &h->cand_cnt, (size_t)n));
        RS_TRY(rs_alloc(h, &h->row_flag, (size_t)n));
        RS_TRY(rs_alloc(h, &h->cand_id, (size_t)n * h->cand_cap));
        RS_TRY(rs_alloc(h, &h->cand_sim, (size_t)n * h->cand_cap));
        h->topk_rows = n;
        RS_CUDA(cudaMemsetAsync(h->topk_idx, 0xFF, (size_t)n * k * 4, h->stream));   // -1 = empty
        RS_CUDA(cudaMemsetAsync(h->topk_sim, 0xFF, (size_t)n * k * 8, h->stream));   // NaN
        RS_CUDA(cudaMemsetAsync(h->thr_key, 0, (size_t)n * 8, h->stream));           // accept every valid similarity
        RS_CUDA(cudaMemsetAsync(h->thr_id, 0xFF, (size_t)n * 4, h->stream));
        RS_CUDA(cudaMemsetAsync(h->cand_cnt, 0, (size_t)n * 4, h->stream));
        RS_CUDA(cudaMemsetAsync(h->row_flag, 0, (size_t)n * 4, h->stream));
        int32_t *d_over = h->d_flags + 14;
        RS_CUDA(cudaEventRecord(h->ev_b, h->stream));
        const int n_waves = rs_tensor_band_count(h);
        for (int w = 0; w < n_waves && rc == RS_OK; w++) {
            int rerun = 0;
            for (;;) {
                RS_CUDA(cudaMemsetAsync(d_over, 0, 4, h->stream));
                rc = rs_sim_tensor_band_launch(h, w);
                if (rc == RS_OK) rc = rs_topk_compact_launch(h, k, d_over, rerun);
                if (rc != RS_OK) break;
                int32_t over = 0;
                RS_CUDA(cudaMemcpyAsync(&over, d_over, 4, cudaMemcpyDeviceToHost, h->stream));
                RS_CUDA(cudaStreamSynchronize(h->stream));
                if (rerun) rc = rs_topk_mask_launch(h, k, 1);      // thresholds of the rows that sat the pass out
                if (over == 0 || rc != RS_OK) break;
                rc = rs_topk_mask_launch(h, k, 0);                 // run the band again for the flagged rows only
                rerun = 1;
            }
        }
        if (rc != RS_OK) { free_fit_state(h); return rc; }
        RS_CUDA(cudaEventRecord(h->ev_c, h->stream));
    } else if (h->p.shard_count >= 1) {
        // top-k only, SYMMETRIC SLABS (see rs_knn_params::shard_count): slab s = rows [s*m, s*m+m);
        // of each slab only the part right of the diagonal is computed, the slab feeds the lists of
        // its own rows, its transpose the lists of the rows below it.  Half the similarity work of
        // full rows, and the slabs of a multi-GPU job are dealt round-robin so every rank gets the
        // same share of the triangle.
        const int32_t k = h->p.topk > 0 ? h->p.topk : h->p.k;
        const int64_t n = n_left;
        int64_t m = (int64_t)(6ll << 30) / (h->ld_s * 8);        // ~6 GiB slab + the same for its transpose
        if (h->p.shard_count > 1) {
            // enough slabs for an even deal: at least 4 per shard (down to 1024 rows each)
            int64_t want = (n + 4ll * h->p.shard_count - 1) / (4ll * h->p.shard_count);
            want = (want + 255) / 256 * 256;
            if (want < 1024) want = 1024;
            if (want < m) m = want;
        }
        if (const char *e = getenv("RS_KNN_SLAB_ROWS")) m = atoll(e);   // tests: many slabs on a small matrix
        if (m < 256) m = 256;
        m = m / 256 * 256;
        if (m > n) m = (n + 15) / 16 * 16;
        const int64_t ld_t = m;
        double *tbuf = nullptr;
        RS_TRY(rs_alloc(h, &h->sims, (size_t)m * (size_t)h->ld_s));
        RS_TRY(rs_alloc(h, &tbuf, (size_t)n * (size_t)ld_t));
        RS_TRY(rs_alloc(h, &h->topk_idx, (size_t)n * k));
        RS_TRY(rs_alloc(h, &h->topk_sim, (size_t)n * k));
        h->topk_rows = n;
        RS_CUDA(cudaMemsetAsync(h->topk_idx, 0xFF, (size_t)n * k * 4, h->stream));   // -1 = empty
        RS_CUDA(cudaMemsetAsync(h->topk_sim, 0xFF, (size_t)n * k * 8, h->stream));   // NaN
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
                rc = cudaMemsetAsync(h->sims, 0xFF, (size_t)(r1 - r0) * (size_t)h->ld_s * 8, h->stream) == cudaSuccess
                         ? RS_OK : RS_ERR_CUDA;
                if (rc == RS_OK) rc = rs_sim_stream_launch(h);
            } else {
                rc = rs_sim_tensor_launch(h, nullptr, 0, 0);
            }
            if (rc == RS_OK) rc = rs_topk_slab_launch(h, r0, (int32_t)(r1 - r0), tbuf, ld_t, k);
            if (rc != RS_OK) break;
        }
        h->force_sym = false;
        h->col_begin = 0;
        h->row_begin = 0;
        h->row_end = n;
        if (rc != RS_OK) { free_fit_state(h); return rc; }
        RS_CUDA(cudaEventRecord(h->ev_c, h->stream));
    } else {
        // top-k only: similarity rows are produced slab by slab and reduced to neighbour
        // lists; the N x N matrix never exists in HBM.
        const int32_t k = h->p.topk > 0 ? h->p.topk : h->p.k;
        int64_t slab = (int64_t)(2ull << 30) / ((int64_t)h->ld_s * 8);  // ~2 GiB of rows at a time
        if (slab < 128) slab = 128;
        slab = slab / 128 * 128;
        if (slab > rows) slab = rows;
        RS_TRY(rs_alloc(h, &h->sims, (size_t)slab * (size_t)h->ld_s));
        RS_TRY(rs_alloc(h, &h->topk_idx, (size_t)rows * k));
        RS_TRY(rs_alloc(h, &h->topk_sim, (size_t)rows * k));
        h->topk_rows = rows;
        RS_CUDA(cudaEventRecord(h->ev_b, h->stream));
        const int64_t rb = h->row_begin, re = h->row_end;
        for (int64_t r0 = rb; r0 < re; r0 += slab) {
            h->row_begin = r0;
            h->row_end = r0 + slab < re ? r0 + slab : re;
            rc = (path == RS_PATH_TENSOR) ? rs_sim_tensor_launch(h, nullptr, 0, 0) : rs_sim_stream_launch(h);
            if (rc == RS_OK && path == RS_PATH_STREAM) rc = rs_symmetrize_launch(h);
            if (rc == RS_OK)
                rc = rs_topk_launch(h, k, h->topk_idx + (r0 - rb) * k, h->topk_sim + (r0 - rb) * k);
            if (rc != RS_OK) break;
        }
        h->row_begin = rb;
        h->row_end = re;
        if (rc != RS_OK) { free_fit_state(h); return rc; }
        RS_CUDA(cudaEventRecord(h->ev_c, h->stream));
    }
    h->prep_pending = true;
    h->sim_pending = true;
    h->fitted = true;
    return RS_OK;
}

int32_t rs_scratch_get(rs_knn *h, int slot, size_t bytes, void **out) {
    if (h->scratch.size() <= (size_t)slot) {
        h->scratch.resize(slot + 1, nullptr);
        h->scratch_bytes.resize(slot + 1, 0);
    }
    if (h->scratch_bytes[slot] < bytes) {
        if (h->scratch[slot]) {
            RS_CUDA(cudaStreamSynchronize(h->stream));
            rs_cached_free(h->device, h->scratch[slot], h->scratch_bytes[slot]);
        }
        h->scratch[slot] = nullptr;
        h->scratch_bytes[slot] = 0;
        size_t want = bytes + bytes / 4 + 256, got = 0;
        RS_TRY(rs_cached_malloc(h->device, &h->scratch[slot], want, &got));
        h->scratch_bytes[slot] = got;
    }
    *out = h->scratch[slot];
    return RS_OK;
}

int32_t rs_knn_fit(rs_knn *h, const int32_t *left, const int32_t *right, const double *rating, int64_t nnz,
                   int32_t n_left, int32_t n_right, double global_mean, const double *left_bias,
                   const double *right_bias, double global_bias) {
    RS_ENTER(h);
    if (!left || !right || !rating || nnz <= 0 || n_left <= 0 || n_right <= 0) {
        rs_set_error("rs_knn_fit: empty or null input (nnz=%lld n_left=%d n_right=%d)", (long long)nnz, n_left,
                     n_right);
        return RS_ERR_INVALID;
    }
    // persistent device staging (grow-only): a refit of the same size allocates nothing
    void *d_left, *d_right, *d_rating, *d_lb = nullptr, *d_rb = nullptr;
    RS_TRY(rs_scratch_get(h, RS_SCR_FIT_LEFT, (size_t)nnz * 4, &d_left));
    RS_TRY(rs_scratch_get(h, RS_SCR_FIT_RIGHT, (size_t)nnz * 4, &d_right));
    RS_TRY(rs_scratch_get(h, RS_SCR_FIT_RATING, (size_t)nnz * 8, &d_rating));
    RS_CUDA(cudaMemcpyAsync(d_left, left, (size_t)nnz * 4, cudaMemcpyHostToDevice, h->stream));
    RS_CUDA(cudaMemcpyAsync(d_right, right, (size_t)nnz * 4, cudaMemcpyHostToDevice, h->stream));
    RS_CUDA(cudaMemcpyAsync(d_rating, rating, (size_t)nnz * 8, cudaMemcpyHostToDevice, h->stream));
    if (left_bias) {
        RS_TRY(rs_scratch_get(h, RS_SCR_FIT_LEFT_BIAS, (size_t)n_left * 8, &d_lb));
        RS_CUDA(cudaMemcpyAsync(d_lb, left_bias, (size_t)n_left * 8, cudaMemcpyHostToDevice, h->stream));
    }
    if (right_bias) {
        RS_TRY(rs_scratch_get(h, RS_SCR_FIT_RIGHT_BIAS, (size_t)n_right * 8, &d_rb));
        RS_CUDA(cudaMemcpyAsync(d_rb, right_bias, (size_t)n_right * 8, cudaMemcpyHostToDevice, h->stream));
    }
    RS_CUDA(cudaEventRecord(h->ev_in, h->stream));
    RS_TRY(rs_knn_fit_device(h, (const int32_t *)d_left, (const int32_t *)d_right, (const double *)d_rating, nnz,
                             n_left, n_right, global_mean, (const double *)d_lb, (const double *)d_rb,
                             global_bias));
    // The inputs are borrowed for the duration of the call only: wait until the host->device copies
    // are done (they are — the validation read-backs of the build synchronised after them), NOT for
    // the similarity kernel.  Fit returns while it runs; everything that needs its result
    // (predict, sims_rows, topk, profile) is ordered behind it on the handle's stream, so the
    // caller's next host work (converting the test set's ids, core/data.go:98-105) overlaps it.
    cudaError_t e = cudaEventSynchronize(h->ev_in);
    if (e != cudaSuccess) {
        rs_set_error("rs_knn_fit: %s", cudaGetErrorString(e));
        h->fitted = false;
        return RS_ERR_CUDA;
    }
    return RS_OK;
}

// Every check of rs_knn_update, in the order they fire: the handle is fitted; its model is one that an update can
// extend exactly (a matrix of all rows, no Slope One, no bias of a global fit, the exact Pearson replay); the counts
// do not shrink; the pointers are there when there are ratings.  The ratings themselves are checked on the device.
static int32_t check_update(rs_knn *h, const int32_t *left, const int32_t *right, const double *rating, int64_t nnz,
                            int32_t n_left, int32_t n_right) {
    const char *who = "rs_knn_update";
    if (!h->fitted) {
        rs_set_error("%s: Fit has not been called", who);
        return RS_ERR_INVALID;
    }
    if (h->p.store != RS_STORE_MATRIX) {
        rs_set_error("%s needs RS_STORE_MATRIX (the handle keeps top-k lists only)", who);
        return RS_ERR_UNSUPPORTED;
    }
    if (h->cyc_R > 1 || h->p.shard_count > 1 || h->row_begin != 0 || h->row_end != h->n_left) {
        rs_set_error("%s needs a handle that holds every row (no row_begin/row_end shard, shard_count <= 1)", who);
        return RS_ERR_UNSUPPORTED;
    }
    if (h->p.sim == RS_SIM_SLOPE_ONE) {
        rs_set_error("%s: Slope One is not supported", who);
        return RS_ERR_UNSUPPORTED;
    }
    if (h->p.knn_type == RS_KNN_BASELINE || h->p.sim == RS_SIM_PEARSON_BASELINE) {
        rs_set_error("%s: the baseline biases come from a global fit that every rating changes "
                     "(RS_KNN_BASELINE / RS_SIM_PEARSON_BASELINE): refit", who);
        return RS_ERR_UNSUPPORTED;
    }
    if (h->p.sim == RS_SIM_PEARSON && h->p.pearson_mode == RS_PEARSON_SUMS) {
        rs_set_error("%s: the recomputed rows are the exact Pearson replay (pearson_mode EXACT)", who);
        return RS_ERR_UNSUPPORTED;
    }
    if (n_left < h->n_left || n_right < h->n_right || nnz < 0) {
        rs_set_error("%s: n_left=%d n_right=%d nnz=%lld (the fitted counts are %d x %d)", who, n_left, n_right,
                     (long long)nnz, h->n_left, h->n_right);
        return RS_ERR_INVALID;
    }
    if (nnz > 0 && (!left || !right || !rating)) {
        rs_set_error("%s: null argument", who);
        return RS_ERR_INVALID;
    }
    if (h->nnz + nnz >= (1ll << 31)) {
        rs_set_error("%s: %lld ratings in all exceed the 2^31-1 entries supported", who, (long long)(h->nnz + nnz));
        return RS_ERR_UNSUPPORTED;
    }
    return RS_OK;
}

int32_t rs_knn_update_device(rs_knn *h, const int32_t *d_left, const int32_t *d_right, const double *d_rating,
                             int64_t nnz, int32_t n_left, int32_t n_right, double global_mean) {
    RS_ENTER(h);
    RS_TRY(check_update(h, d_left, d_right, d_rating, nnz, n_left, n_right));
    return rs_update_run(h, d_left, d_right, d_rating, nnz, n_left, n_right, global_mean);
}

int32_t rs_knn_update(rs_knn *h, const int32_t *left, const int32_t *right, const double *rating, int64_t nnz,
                      int32_t n_left, int32_t n_right, double global_mean) {
    RS_ENTER(h);
    RS_TRY(check_update(h, left, right, rating, nnz, n_left, n_right));
    void *d_left = nullptr, *d_right = nullptr, *d_rating = nullptr;
    if (nnz > 0) {
        RS_TRY(rs_scratch_get(h, RS_SCR_FIT_LEFT, (size_t)nnz * 4, &d_left));
        RS_TRY(rs_scratch_get(h, RS_SCR_FIT_RIGHT, (size_t)nnz * 4, &d_right));
        RS_TRY(rs_scratch_get(h, RS_SCR_FIT_RATING, (size_t)nnz * 8, &d_rating));
        RS_CUDA(cudaMemcpyAsync(d_left, left, (size_t)nnz * 4, cudaMemcpyHostToDevice, h->stream));
        RS_CUDA(cudaMemcpyAsync(d_right, right, (size_t)nnz * 4, cudaMemcpyHostToDevice, h->stream));
        RS_CUDA(cudaMemcpyAsync(d_rating, rating, (size_t)nnz * 8, cudaMemcpyHostToDevice, h->stream));
    }
    // the update reads its inputs before its validation read-back: they are consumed when it returns
    return rs_update_run(h, (const int32_t *)d_left, (const int32_t *)d_right, (const double *)d_rating, nnz, n_left,
                         n_right, global_mean);
}

static int32_t require_matrix(rs_knn *h, const char *who) {
    if (!h->fitted) {
        rs_set_error("%s: Fit has not been called", who);
        return RS_ERR_INVALID;
    }
    if (h->p.store != RS_STORE_MATRIX) {
        rs_set_error("%s needs RS_STORE_MATRIX (the handle keeps top-k lists only)", who);
        return RS_ERR_INVALID;
    }
    if (h->cyc_R > 1 && !h->peers_ready) {
        rs_set_error("%s: cyclic row shards hold one triangle of their rows until rs_knn_mirror has run", who);
        return RS_ERR_INVALID;
    }
    return RS_OK;
}

int32_t rs_knn_predict_batch_device(rs_knn *h, const int32_t *d_left, const int32_t *d_right, int64_t n,
                                    double *d_out) {
    RS_ENTER(h);
    RS_TRY(require_matrix(h, "rs_knn_predict_batch"));
    if (n == 0) return RS_OK;
    if (!d_left || !d_right || !d_out || n < 0) {
        rs_set_error("rs_knn_predict_batch: null argument");
        return RS_ERR_INVALID;
    }
    if (h->pred_pending) RS_TRY(fold_profile(h));
    RS_CUDA(cudaEventRecord(h->ev_d, h->stream));
    if (h->p.sim == RS_SIM_SLOPE_ONE) RS_TRY(rs_slope_predict_launch(h, d_left, d_right, n, d_out));
    else RS_TRY(rs_predict_launch(h, d_left, d_right, n, d_out, nullptr, nullptr, nullptr, 0));
    RS_CUDA(cudaEventRecord(h->ev_e, h->stream));
    h->pred_pending = true;
    return RS_OK;
}

int32_t rs_knn_predict_batch_sharded_device(rs_knn *h, const int32_t *d_left, const int32_t *d_right, int64_t n,
                                            double *d_out) {
    RS_ENTER(h);
    RS_TRY(require_matrix(h, "rs_knn_predict_batch_sharded"));
    if (h->cyc_R < 2) {
        rs_set_error("rs_knn_predict_batch_sharded: the handle is not a cyclic row shard");
        return RS_ERR_INVALID;
    }
    if (n == 0) return RS_OK;
    if (!d_left || !d_right || !d_out || n < 0) {
        rs_set_error("rs_knn_predict_batch_sharded: null argument");
        return RS_ERR_INVALID;
    }
    if (h->pred_pending) RS_TRY(fold_profile(h));
    RS_CUDA(cudaEventRecord(h->ev_d, h->stream));
    RS_TRY(rs_predict_launch(h, d_left, d_right, n, d_out, nullptr, nullptr, nullptr, 0, 1));
    RS_CUDA(cudaEventRecord(h->ev_e, h->stream));
    h->pred_pending = true;
    return RS_OK;
}

int32_t rs_knn_predict_batch(rs_knn *h, const int32_t *left, const int32_t *right, int64_t n, double *out) {
    RS_ENTER(h);
    RS_TRY(require_matrix(h, "rs_knn_predict_batch"));
    if (n == 0) return RS_OK;
    if (!left || !right || !out || n < 0) {
        rs_set_error("rs_knn_predict_batch: null argument");
        return RS_ERR_INVALID;
    }
    void *dl, *dr, *dout;
    RS_TRY(rs_scratch_get(h, RS_SCR_PRED_LEFT, (size_t)n * 4, &dl));
    RS_TRY(rs_scratch_get(h, RS_SCR_PRED_RIGHT, (size_t)n * 4, &dr));
    RS_TRY(rs_scratch_get(h, RS_SCR_PRED_OUT, (size_t)n * 8, &dout));
    RS_CUDA(cudaMemcpyAsync(dl, left, (size_t)n * 4, cudaMemcpyHostToDevice, h->stream));
    RS_CUDA(cudaMemcpyAsync(dr, right, (size_t)n * 4, cudaMemcpyHostToDevice, h->stream));
    RS_TRY(rs_knn_predict_batch_device(h, (const int32_t *)dl, (const int32_t *)dr, n, (double *)dout));
    RS_CUDA(cudaMemcpyAsync(out, dout, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    RS_CUDA(cudaStreamSynchronize(h->stream));
    return RS_OK;
}

int32_t rs_knn_predict_neighbors(rs_knn *h, int32_t left, int32_t right, int32_t cap, int32_t *ids, double *sims,
                                 int32_t *n_out) {
    RS_ENTER(h);
    RS_TRY(require_matrix(h, "rs_knn_predict_neighbors"));
    if (!ids || !sims || !n_out || cap < 1) {
        rs_set_error("rs_knn_predict_neighbors: null argument");
        return RS_ERR_INVALID;
    }
    void *dl, *dr, *dout, *dids, *dsims, *dcnt;
    RS_TRY(rs_scratch_get(h, RS_SCR_PRED_LEFT, 4, &dl));
    RS_TRY(rs_scratch_get(h, RS_SCR_PRED_RIGHT, 4, &dr));
    RS_TRY(rs_scratch_get(h, RS_SCR_PRED_OUT, 8, &dout));
    RS_TRY(rs_scratch_get(h, RS_SCR_HOST_IDS, (size_t)cap * 4, &dids));
    RS_TRY(rs_scratch_get(h, RS_SCR_HOST_SIMS, (size_t)cap * 8, &dsims));
    RS_TRY(rs_scratch_get(h, RS_SCR_NB_COUNT, 4, &dcnt));
    RS_CUDA(cudaMemcpyAsync(dl, &left, 4, cudaMemcpyHostToDevice, h->stream));
    RS_CUDA(cudaMemcpyAsync(dr, &right, 4, cudaMemcpyHostToDevice, h->stream));
    RS_CUDA(cudaMemsetAsync(dcnt, 0, 4, h->stream));
    RS_TRY(rs_predict_launch(h, (const int32_t *)dl, (const int32_t *)dr, 1, (double *)dout, (int32_t *)dids,
                             (double *)dsims, (int32_t *)dcnt, cap));
    RS_TRY(rs_nb_cells_launch(h, (const int32_t *)dl, (const int32_t *)dids, (const int32_t *)dcnt, (double *)dsims));
    int32_t cnt = 0;
    RS_CUDA(cudaMemcpyAsync(&cnt, dcnt, 4, cudaMemcpyDeviceToHost, h->stream));
    RS_CUDA(cudaStreamSynchronize(h->stream));
    if (cnt > 0) {
        RS_CUDA(cudaMemcpy(ids, dids, (size_t)cnt * 4, cudaMemcpyDeviceToHost));
        RS_CUDA(cudaMemcpy(sims, dsims, (size_t)cnt * 8, cudaMemcpyDeviceToHost));
    }
    *n_out = cnt;
    return RS_OK;
}

// Every check of the recommendation entry points, in the order they fire: the handle holds the whole matrix (the
// _sharded entry points: a row shard, mirrored if cyclic), the query side exists, k fits, and for lists what
// rs_knn_recommend accepts less top-k-only handles (checked first) and, for left queries, the models that need
// something of the query the lists do not give (a baseline bias) or whose matrix is not the exact replay the lists'
// similarity rows are (Pearson sums).  Pointers are checked only when n > 0.
static int32_t check_recommend(rs_knn *h, const char *who, const rs_rec_call &c) {
    if (c.given && h->fitted && h->p.store == RS_STORE_TOPK) {
        rs_set_error("%s needs RS_STORE_MATRIX (the handle keeps top-k lists only)", who);
        return RS_ERR_UNSUPPORTED;
    }
    if (!h->fitted) {
        rs_set_error("%s: Fit has not been called", who);
        return RS_ERR_INVALID;
    }
    if (h->p.store != RS_STORE_MATRIX) return require_matrix(h, who);
    const bool row_shard = h->cyc_R > 1 || h->p.shard_count > 1 || h->row_begin != 0 || h->row_end != h->n_left;
    if (!c.sharded && row_shard) {
        rs_set_error("%s needs a handle that holds every row (no row_begin/row_end shard, shard_count <= 1)", who);
        return RS_ERR_UNSUPPORTED;
    }
    if (c.sharded && !row_shard) {
        rs_set_error("%s: the handle holds every row, not a row shard (use the plain entry point)", who);
        return RS_ERR_INVALID;
    }
    if (c.sharded) RS_TRY(require_matrix(h, who));
    if (h->p.sim == RS_SIM_SLOPE_ONE) {
        rs_set_error("%s: Slope One is not supported", who);
        return RS_ERR_UNSUPPORTED;
    }
    if (c.side != RS_SIDE_LEFT && c.side != RS_SIDE_RIGHT) {
        rs_set_error("%s: side must be RS_SIDE_LEFT or RS_SIDE_RIGHT (got %d)", who, c.side);
        return RS_ERR_INVALID;
    }
    if (h->p.k > 256) {
        rs_set_error("%s: k=%d exceeds the 256 neighbours the predict kernel supports", who, h->p.k);
        return RS_ERR_UNSUPPORTED;
    }
    if (c.n < 0 || c.n >= (1ll << 31)) {
        rs_set_error("%s: n=%lld outside [0, 2^31)", who, (long long)c.n);
        return RS_ERR_INVALID;
    }
    if (c.given && c.side == RS_SIDE_LEFT) {
        if (h->p.knn_type == RS_KNN_BASELINE || h->p.sim == RS_SIM_PEARSON_BASELINE) {
            rs_set_error("%s: left queries have no baseline bias (RS_KNN_BASELINE / RS_SIM_PEARSON_BASELINE)", who);
            return RS_ERR_UNSUPPORTED;
        }
        if (h->p.sim == RS_SIM_PEARSON && h->p.pearson_mode == RS_PEARSON_SUMS) {
            rs_set_error("%s: left queries need the exact Pearson matrix (pearson_mode EXACT)", who);
            return RS_ERR_UNSUPPORTED;
        }
        if ((int64_t)h->n_left + c.n >= (1ll << 31)) {
            rs_set_error("%s: n_left + n = %lld (at most 2^31 - 1)", who, (long long)h->n_left + c.n);
            return RS_ERR_UNSUPPORTED;
        }
    }
    if (c.lists && (c.n_top < 1 || c.n_top > 512)) {
        rs_set_error("%s: n_top=%d outside [1, 512]", who, c.n_top);
        return RS_ERR_INVALID;
    }
    const bool null_in = c.given ? !c.ptr || !c.ids || !c.vals : !c.queries;
    const bool null_out = c.lists ? !c.top_ids || !c.top_scores : !c.rows;
    if (c.n > 0 && (null_in || null_out)) {
        rs_set_error("%s: null argument", who);
        return RS_ERR_INVALID;
    }
    return RS_OK;
}

// Host variants: the queries to the device.  Ids outside [-1, n_side) are refused (the _device variants score them
// as -1).  Of the lists, ptr is checked only as far as it sizes the copies; the device checks the rest as it does for
// the _device variants.
static int32_t stage_queries(rs_knn *h, const char *who, rs_rec_call &c) {
    if (!c.given) {
        const int32_t n_side = c.side == RS_SIDE_RIGHT ? h->n_right : h->n_left;
        for (int64_t i = 0; i < c.n; i++) {
            if (c.queries[i] < -1 || c.queries[i] >= n_side) {
                rs_set_error("%s: query %lld = %d outside [-1, %d)", who, (long long)i, c.queries[i], n_side);
                return RS_ERR_INVALID;
            }
        }
        void *dq;
        RS_TRY(rs_scratch_get(h, RS_SCR_REC_QUERIES, (size_t)c.n * 4, &dq));
        RS_CUDA(cudaMemcpyAsync(dq, c.queries, (size_t)c.n * 4, cudaMemcpyHostToDevice, h->stream));
        c.queries = (const int32_t *)dq;
        return RS_OK;
    }
    const int64_t p0 = c.ptr[0], nnz = c.ptr[c.n] - p0;
    if (p0 < 0 || nnz < 0) {
        rs_set_error("%s: ptr[0] = %lld, ptr[n] = %lld (need 0 <= ptr[0] <= ptr[n])", who, (long long)p0,
                     (long long)c.ptr[c.n]);
        return RS_ERR_INVALID;
    }
    if (nnz >= (1ll << 31)) {
        rs_set_error("%s: %lld entries (at most 2^31 - 1 per call)", who, (long long)nnz);
        return RS_ERR_UNSUPPORTED;
    }
    void *dp, *di, *dv;
    RS_TRY(rs_scratch_get(h, RS_SCR_REC_PTR, (size_t)(c.n + 1) * 8, &dp));
    RS_TRY(rs_scratch_get(h, RS_SCR_REC_IDS, (size_t)nnz * 4 + 4, &di));
    RS_TRY(rs_scratch_get(h, RS_SCR_REC_VALS, (size_t)nnz * 8 + 8, &dv));
    RS_CUDA(cudaMemcpyAsync(dp, c.ptr, (size_t)(c.n + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    if (nnz > 0) {
        RS_CUDA(cudaMemcpyAsync(di, c.ids + p0, (size_t)nnz * 4, cudaMemcpyHostToDevice, h->stream));
        RS_CUDA(cudaMemcpyAsync(dv, c.vals + p0, (size_t)nnz * 8, cudaMemcpyHostToDevice, h->stream));
    }
    // the device copies hold the entries from ptr[0] on: index them from ptr[0]
    c.ptr = (const int64_t *)dp;
    c.ids = (const int32_t *)di - p0;
    c.vals = (const double *)dv - p0;
    return RS_OK;
}

// The call descriptions of the ten shims.
static rs_rec_call by_id(int32_t side, const int32_t *queries, int64_t n, bool sharded) {
    rs_rec_call c{};
    c.side = side; c.sharded = sharded; c.queries = queries; c.n = n;
    return c;
}

static rs_rec_call by_lists(int32_t side, const int64_t *ptr, const int32_t *ids, const double *vals, int64_t n) {
    rs_rec_call c{};
    c.side = side; c.given = true; c.ptr = ptr; c.ids = ids; c.vals = vals; c.n = n;
    return c;
}

static rs_rec_call with_rows(rs_rec_call c, double *out) {
    c.rows = out;
    return c;
}

static rs_rec_call with_lists(rs_rec_call c, int32_t n_top, int32_t *ids, double *scores) {
    c.lists = true; c.n_top = n_top; c.top_ids = ids; c.top_scores = scores;
    return c;
}

// The one entry of the ten: checks, then the driver; host variants stage their inputs and copy the outputs back.
static int32_t recommend(rs_knn *h, const char *who, rs_rec_call c, bool host) {
    RS_ENTER(h);
    RS_TRY(check_recommend(h, who, c));
    if (c.n == 0) return RS_OK;
    if (!host) return rs_recommend_run(h, c);
    RS_TRY(stage_queries(h, who, c));
    const rs_rec_call caller = c;   // the host outputs
    const size_t cells = c.lists ? (size_t)c.n * c.n_top : (size_t)c.n * rs_n_targets(h, c.side);
    void *d_out, *d_scores = nullptr;
    RS_TRY(rs_scratch_get(h, RS_SCR_REC_OUT, cells * (c.lists ? 4 : 8), &d_out));
    if (c.lists) {
        RS_TRY(rs_scratch_get(h, RS_SCR_REC_SCORES, cells * 8, &d_scores));
        c = with_lists(c, c.n_top, (int32_t *)d_out, (double *)d_scores);
    } else {
        c = with_rows(c, (double *)d_out);
    }
    RS_TRY(rs_recommend_run(h, c));
    if (c.lists) {
        RS_CUDA(cudaMemcpyAsync(caller.top_ids, d_out, cells * 4, cudaMemcpyDeviceToHost, h->stream));
        RS_CUDA(cudaMemcpyAsync(caller.top_scores, d_scores, cells * 8, cudaMemcpyDeviceToHost, h->stream));
    } else {
        RS_CUDA(cudaMemcpyAsync(caller.rows, d_out, cells * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    RS_CUDA(cudaStreamSynchronize(h->stream));
    return RS_OK;
}

int32_t rs_knn_score_all_device(rs_knn *h, int32_t side, const int32_t *d_queries, int64_t n, double *d_out) {
    return recommend(h, "rs_knn_score_all", with_rows(by_id(side, d_queries, n, false), d_out), false);
}

int32_t rs_knn_score_all(rs_knn *h, int32_t side, const int32_t *queries, int64_t n, double *out) {
    return recommend(h, "rs_knn_score_all", with_rows(by_id(side, queries, n, false), out), true);
}

int32_t rs_knn_recommend_device(rs_knn *h, int32_t side, const int32_t *d_queries, int64_t n, int32_t n_top,
                                int32_t *d_ids, double *d_scores) {
    return recommend(h, "rs_knn_recommend", with_lists(by_id(side, d_queries, n, false), n_top, d_ids, d_scores), false);
}

int32_t rs_knn_recommend(rs_knn *h, int32_t side, const int32_t *queries, int64_t n, int32_t n_top, int32_t *ids,
                         double *scores) {
    return recommend(h, "rs_knn_recommend", with_lists(by_id(side, queries, n, false), n_top, ids, scores), true);
}

int32_t rs_knn_score_all_sharded_device(rs_knn *h, int32_t side, const int32_t *d_queries, int64_t n,
                                        double *d_out) {
    return recommend(h, "rs_knn_score_all_sharded", with_rows(by_id(side, d_queries, n, true), d_out), false);
}

int32_t rs_knn_recommend_sharded_device(rs_knn *h, int32_t side, const int32_t *d_queries, int64_t n, int32_t n_top,
                                        int32_t *d_ids, double *d_scores) {
    return recommend(h, "rs_knn_recommend_sharded", with_lists(by_id(side, d_queries, n, true), n_top, d_ids, d_scores),
                     false);
}

int32_t rs_knn_score_all_given_device(rs_knn *h, int32_t side, const int64_t *d_ptr, const int32_t *d_ids,
                                      const double *d_vals, int64_t n, double *d_out) {
    return recommend(h, "rs_knn_score_all_given", with_rows(by_lists(side, d_ptr, d_ids, d_vals, n), d_out), false);
}

int32_t rs_knn_recommend_given_device(rs_knn *h, int32_t side, const int64_t *d_ptr, const int32_t *d_ids,
                                      const double *d_vals, int64_t n, int32_t n_top, int32_t *d_top_ids,
                                      double *d_top_scores) {
    return recommend(h, "rs_knn_recommend_given",
                     with_lists(by_lists(side, d_ptr, d_ids, d_vals, n), n_top, d_top_ids, d_top_scores), false);
}

int32_t rs_knn_score_all_given(rs_knn *h, int32_t side, const int64_t *ptr, const int32_t *ids, const double *vals,
                               int64_t n, double *out) {
    return recommend(h, "rs_knn_score_all_given", with_rows(by_lists(side, ptr, ids, vals, n), out), true);
}

int32_t rs_knn_recommend_given(rs_knn *h, int32_t side, const int64_t *ptr, const int32_t *ids, const double *vals,
                               int64_t n, int32_t n_top, int32_t *top_ids, double *top_scores) {
    return recommend(h, "rs_knn_recommend_given", with_lists(by_lists(side, ptr, ids, vals, n), n_top, top_ids, top_scores),
                     true);
}

int32_t rs_knn_sims_rows(rs_knn *h, int64_t row0, int64_t nrows, double *out) {
    RS_ENTER(h);
    RS_TRY(require_matrix(h, "rs_knn_sims_rows"));
    if (!out || nrows < 0 || row0 < h->row_begin || row0 + nrows > h->row_end) {
        rs_set_error("rs_knn_sims_rows: rows [%lld,%lld) outside the shard [%lld,%lld)", (long long)row0,
                     (long long)(row0 + nrows), (long long)h->row_begin, (long long)h->row_end);
        return RS_ERR_INVALID;
    }
    if (nrows == 0) return RS_OK;
    int64_t local0 = row0 - h->row_begin;
    if (h->cyc_R > 1) {
        // cyclic shards: the rows asked for must lie in ONE block of RS_CYC_B rows this shard owns
        if (!rs_cyc_owns(row0, h->cyc_R, h->cyc_r) || row0 / RS_CYC_B != (row0 + nrows - 1) / RS_CYC_B) {
            rs_set_error("rs_knn_sims_rows: rows [%lld,%lld) are not inside one %d-row block of shard %d of %d",
                         (long long)row0, (long long)(row0 + nrows), RS_CYC_B, h->cyc_r, h->cyc_R);
            return RS_ERR_INVALID;
        }
        local0 = rs_cyc_local(row0, h->cyc_R);
    }
    RS_CUDA(cudaMemcpy2DAsync(out, (size_t)h->n_left * 8, h->sims + local0 * h->ld_s,
                              (size_t)h->ld_s * 8, (size_t)h->n_left * 8, (size_t)nrows, cudaMemcpyDeviceToHost,
                              h->stream));
    RS_CUDA(cudaStreamSynchronize(h->stream));
    return RS_OK;
}

int32_t rs_knn_topk_device(rs_knn *h, int32_t k, int32_t *d_idx, double *d_sim) {
    RS_ENTER(h);
    if (!h->fitted || !d_idx || !d_sim) {
        rs_set_error("rs_knn_topk: not fitted or null argument");
        return RS_ERR_INVALID;
    }
    const int64_t rows = h->p.store == RS_STORE_TOPK ? h->topk_rows : h->rows_local;
    if (h->p.store == RS_STORE_MATRIX) RS_TRY(require_matrix(h, "rs_knn_topk"));
    if (h->p.store == RS_STORE_TOPK) {
        const int32_t kk = h->p.topk > 0 ? h->p.topk : h->p.k;
        if (k != kk) {
            rs_set_error("rs_knn_topk: handle holds top-%d lists, asked for %d", kk, k);
            return RS_ERR_INVALID;
        }
        RS_CUDA(cudaMemcpyAsync(d_idx, h->topk_idx, (size_t)rows * k * 4, cudaMemcpyDeviceToDevice, h->stream));
        RS_CUDA(cudaMemcpyAsync(d_sim, h->topk_sim, (size_t)rows * k * 8, cudaMemcpyDeviceToDevice, h->stream));
        return RS_OK;
    }
    return rs_topk_launch(h, k, d_idx, d_sim);
}

int32_t rs_knn_topk(rs_knn *h, int32_t k, int32_t *idx, double *sim) {
    RS_ENTER(h);
    if (!h->fitted || !idx || !sim || k < 1) {
        rs_set_error("rs_knn_topk: not fitted or bad argument");
        return RS_ERR_INVALID;
    }
    const int64_t rows = h->p.store == RS_STORE_TOPK ? h->topk_rows : h->rows_local;
    void *di, *ds;
    RS_TRY(rs_scratch_get(h, RS_SCR_HOST_IDS, (size_t)rows * k * 4, &di));
    RS_TRY(rs_scratch_get(h, RS_SCR_HOST_SIMS, (size_t)rows * k * 8, &ds));
    RS_TRY(rs_knn_topk_device(h, k, (int32_t *)di, (double *)ds));
    RS_CUDA(cudaMemcpyAsync(idx, di, (size_t)rows * k * 4, cudaMemcpyDeviceToHost, h->stream));
    RS_CUDA(cudaMemcpyAsync(sim, ds, (size_t)rows * k * 8, cudaMemcpyDeviceToHost, h->stream));
    RS_CUDA(cudaStreamSynchronize(h->stream));
    return RS_OK;
}

int32_t rs_knn_cosums(rs_knn *h, int64_t row0, int64_t nrows, int32_t *out) {
    RS_ENTER(h);
    if (!h->fitted || !out || nrows < 0 || row0 < 0 || row0 + nrows > h->n_left) {
        rs_set_error("rs_knn_cosums: not fitted or bad argument");
        return RS_ERR_INVALID;
    }
    if (h->rating_class != RS_CLASS_INT8) {
        rs_set_error("rs_knn_cosums: integer co-rating sums need integer ratings in [-11,11]");
        return RS_ERR_UNSUPPORTED;
    }
    if (nrows == 0) return RS_OK;
    if (!h->planes) RS_TRY(rs_prep_planes(h));
    void *d;
    const size_t bytes = (size_t)nrows * (size_t)h->n_left * 6 * 4;
    RS_TRY(rs_scratch_get(h, RS_SCR_COSUMS, bytes, &d));
    RS_TRY(rs_sim_tensor_launch(h, (int32_t *)d, row0, nrows));
    RS_CUDA(cudaMemcpyAsync(out, d, bytes, cudaMemcpyDeviceToHost, h->stream));
    RS_CUDA(cudaStreamSynchronize(h->stream));
    return RS_OK;
}

static int32_t copy_vec(rs_knn *h, const double *d, double *out, const char *who) {
    RS_ENTER(h);
    if (!h->fitted || !out || !d) {
        rs_set_error("%s: not fitted or null argument", who);
        return RS_ERR_INVALID;
    }
    // row statistics are final when Fit returns (the build ends with a synchronisation): read them on
    // the auxiliary stream so that the read-back does not queue behind the similarity kernel
    RS_CUDA(cudaMemcpyAsync(out, d, (size_t)h->n_left * 8, cudaMemcpyDeviceToHost, h->aux_stream));
    RS_CUDA(cudaStreamSynchronize(h->aux_stream));
    return RS_OK;
}

int32_t rs_knn_means(rs_knn *h, double *out) { return copy_vec(h, h ? h->means : nullptr, out, "rs_knn_means"); }
int32_t rs_knn_stddevs(rs_knn *h, double *out) {
    if (h && h->p.knn_type != RS_KNN_ZSCORE) {
        rs_set_error("rs_knn_stddevs: only the z-score KNN keeps StdDevs (core/knn.go:167)");
        return RS_ERR_INVALID;
    }
    return copy_vec(h, h ? h->stddevs : nullptr, out, "rs_knn_stddevs");
}

int32_t rs_knn_set_k(rs_knn *h, int32_t k, int32_t min_k) {
    RS_ENTER(h);
    if (k < 1 || min_k < 0) {
        rs_set_error("rs_knn_set_k: k >= 1 and min_k >= 0 required");
        return RS_ERR_INVALID;
    }
    h->p.k = k;
    h->p.min_k = min_k;
    return RS_OK;
}

int32_t rs_knn_peer_export(rs_knn *h, unsigned char *handle64, int64_t *offset) {
    RS_ENTER(h);
    if (!h->fitted || h->cyc_R < 2 || !handle64 || !offset) {
        rs_set_error("rs_knn_peer_export: the handle is not a fitted cyclic row shard");
        return RS_ERR_INVALID;
    }
    for (const auto &c : h->chunks) {
        const char *s0 = reinterpret_cast<const char *>(h->sims);
        if (s0 >= c.p && s0 < c.p + c.bytes) {
            cudaIpcMemHandle_t mh;
            RS_CUDA(cudaIpcGetMemHandle(&mh, c.p));
            static_assert(sizeof(mh) == 64, "cudaIpcMemHandle_t is 64 bytes");
            std::memcpy(handle64, &mh, 64);
            *offset = (int64_t)(s0 - c.p);
            return RS_OK;
        }
    }
    rs_set_error("rs_knn_peer_export: the matrix is not in the handle's arena");
    return RS_ERR_INVALID;
}

int32_t rs_knn_peer_import(rs_knn *h, int32_t n_peers, const unsigned char *handles, const int64_t *offsets) {
    RS_ENTER(h);
    if (!h->fitted || h->cyc_R < 2 || n_peers != h->cyc_R || !handles || !offsets) {
        rs_set_error("rs_knn_peer_import: needs a fitted cyclic row shard and one (handle, offset) per shard");
        return RS_ERR_INVALID;
    }
    for (int q = 0; q < n_peers; q++) {
        if (q == h->cyc_r) { h->peer_sims[q] = h->sims; continue; }
        const unsigned char *hb = handles + (size_t)q * 64;
        void *base = nullptr;
        RS_TRY(ipc_open_cached(h->device, hb, &base));
        h->peer_sims[q] = reinterpret_cast<const double *>(static_cast<const char *>(base) + offsets[q]);
    }
    return RS_OK;
}

int32_t rs_knn_peer_import_local(rs_knn *h, int32_t n_peers, rs_knn *const *peers) {
    RS_ENTER(h);
    if (!h->fitted || h->cyc_R < 2 || n_peers != h->cyc_R || !peers) {
        rs_set_error("rs_knn_peer_import_local: needs a fitted cyclic row shard and one handle per shard");
        return RS_ERR_INVALID;
    }
    for (int q = 0; q < n_peers; q++) {
        const rs_knn *o = peers[q];
        if (!o || !o->fitted || o->cyc_R != h->cyc_R || o->cyc_r != q || o->n_left != h->n_left || o->ld_s != h->ld_s) {
            rs_set_error("rs_knn_peer_import_local: peer %d is not shard %d of the same Fit", q, q);
            return RS_ERR_INVALID;
        }
        if (o->device != h->device) {
            int can = 0;
            RS_CUDA(cudaDeviceCanAccessPeer(&can, h->device, o->device));
            if (!can) {
                rs_set_error("device %d cannot access device %d", h->device, o->device);
                return RS_ERR_UNSUPPORTED;
            }
            cudaError_t e = cudaDeviceEnablePeerAccess(o->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) RS_CUDA(e);
            (void)cudaGetLastError();
        }
        h->peer_sims[q] = o->sims;
    }
    return RS_OK;
}

int32_t rs_knn_mirror(rs_knn *h) {
    RS_ENTER(h);
    if (!h->fitted || h->cyc_R < 2) {
        rs_set_error("rs_knn_mirror: the handle is not a fitted cyclic row shard");
        return RS_ERR_INVALID;
    }
    for (int q = 0; q < h->cyc_R; q++)
        if (q != h->cyc_r && !h->peer_sims[q]) {
            rs_set_error("rs_knn_mirror: shard %d has not been attached (rs_knn_peer_import)", q);
            return RS_ERR_INVALID;
        }
    RS_TRY(rs_mirror_launch(h));
    h->peers_ready = true;
    return RS_OK;
}

int32_t rs_knn_profile_get(rs_knn *h, rs_knn_profile *out) {
    RS_ENTER(h);
    if (!out) return RS_ERR_INVALID;
    RS_TRY(fold_profile(h));
    *out = h->prof;
    return RS_OK;
}

// ---- page-locked host blocks, cached per process ----
namespace {
struct HostBlock { void *p; size_t bytes; bool used; };
std::mutex g_host_mu;
std::vector<HostBlock> g_host;
}  // namespace

int32_t rs_knn_host_alloc(size_t bytes, void **out) {
    if (!out) { rs_set_error("rs_knn_host_alloc: null argument"); return RS_ERR_INVALID; }
    if (bytes == 0) bytes = 1;
    std::lock_guard<std::mutex> lk(g_host_mu);
    HostBlock *best = nullptr;
    for (auto &b : g_host)                                   // the smallest free block that fits without wasting half of it
        if (!b.used && b.bytes >= bytes && b.bytes <= 2 * bytes + 4096 && (!best || b.bytes < best->bytes)) best = &b;
    if (best) { best->used = true; *out = best->p; return RS_OK; }
    void *p = nullptr;
    RS_CUDA(cudaHostAlloc(&p, bytes, cudaHostAllocPortable));
    g_host.push_back({p, bytes, true});
    *out = p;
    return RS_OK;
}

int32_t rs_knn_host_free(void *p) {
    if (!p) return RS_OK;
    std::lock_guard<std::mutex> lk(g_host_mu);
    for (auto &b : g_host)
        if (b.p == p && b.used) { b.used = false; return RS_OK; }
    rs_set_error("rs_knn_host_free: not a block of rs_knn_host_alloc");
    return RS_ERR_INVALID;
}

int32_t rs_knn_trim_cache(void) {
    rs_cache_trim();
    {
        std::lock_guard<std::mutex> lk(g_host_mu);
        size_t kept = 0;
        for (auto &b : g_host) {
            if (b.used) g_host[kept++] = b;
            else cudaFreeHost(b.p);
        }
        g_host.resize(kept);
    }
    std::lock_guard<std::mutex> lk(g_ipc_mu);
    int cur = 0;
    cudaGetDevice(&cur);
    for (const auto &m : g_ipc) {
        cudaSetDevice(m.device);
        cudaIpcCloseMemHandle(m.base);
    }
    g_ipc.clear();
    cudaSetDevice(cur);
    return RS_OK;
}

int32_t rs_knn_profile_reset(rs_knn *h) {
    RS_ENTER(h);
    RS_TRY(fold_profile(h));
    int32_t path = h->prof.sim_path_used;
    h->prof = rs_knn_profile{};
    h->prof.sim_path_used = path;
    h->prof.corated_triples = h->triples;
    return RS_OK;
}

}  // extern "C"
