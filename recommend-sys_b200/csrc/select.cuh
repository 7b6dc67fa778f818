// select.cuh — the neighbour selection and weighted sum of ONE prediction (core/knn.go:93-141), shared by the
// batched Predict kernel (predict.cu) and the recommend kernels (recommend.cu), so that a recommendation score is
// the same computation as the prediction of the same pair, bit for bit.
//
// One warp per prediction:
//   pass A  gather the similarity of every candidate ONCE (4 independent gathers per lane in
//           flight), map it to an order-preserving 64-bit key (0 = NaN, core/knn.go:95-99), park
//           the keys in shared memory, count the valid ones and find the key range;
//   pass B  (only when more candidates than the register capacity CAP = 32*R) radix selection:
//           256-bucket histogram of (key - lo) >> shift in shared memory, suffix scan -> boundary
//           bucket: everything above it is certainly in the top k, everything below certainly
//           not; the window shrinks to the boundary bucket (8 more key bits per level) while it
//           is too full; a one-value bucket that is still too full is a genuine tie and is taken
//           in scan order = ascending inner id (canonical).  Integer compares only;
//   pass C  compaction of the surviving <= CAP candidates into registers (R per lane);
//   sort    one warp-wide bitonic network over CAP (key,pos) records in registers
//           (strides < R in-register, >= R via __shfl_xor);
//   reduce  the first min(k,valid) neighbours are accumulated sequentially in sorted order,
//           exactly as core/knn.go:116-130 does.
#pragma once

#include "common.cuh"

namespace {

constexpr int PRED_CAP = 512;   // k <= PRED_CAP / 2 (register capacity of predict_select_kernel<8>)

struct Rec {
    uint64_t key;
    uint32_t pos;
};

// a ranks before b: larger key first, then smaller position (= smaller id)
__device__ __forceinline__ bool rec_before(uint64_t ka, uint32_t pa, uint64_t kb, uint32_t pb) {
    return ka > kb || (ka == kb && pa < pb);
}

struct PredArgs {
    const int32_t *perm;   // optional processing order (test pairs grouped by left row), else identity
    unsigned long long *work;   // dynamic work counter: warps grab PRED_GRAB consecutive positions
    const int32_t *left, *right;
    int64_t n;
    double *out;
    const int64_t *r_ptr;
    const int32_t *r_col;
    const double *r_val;
    const double *sims;
    int64_t ld_s;
    int64_t row_begin, row_end;
    int32_t cyc_R, cyc_r;       // cyclic row shards (cyc_R >= 2): the handle holds the rows it owns
    const double *means, *stddevs, *bias;
    double global_mean;
    int32_t n_right;
    int32_t k, min_k, knn_type;
    int32_t *nb_ids;
    double *nb_sims;
    int32_t *nb_count;
    int32_t nb_cap;
    const long long *n_dev; // when set: only the first *n_dev positions of `perm` are processed (the shard's own pairs)
    int32_t foreign_zero;   // cyclic shards: pairs of another shard's rows yield +0.0 (not NaN) and a cold-start pair is answered by
                            // ONE shard, so that an integer all-reduce (sum) of the bit patterns assembles the full vector
    uint64_t *gstage;       // per-warp spill of the staged keys beyond the shared-memory capacity
    int64_t gcap;           // keys per warp in gstage
};

constexpr int SEL_WARPS = 8;
constexpr int PRED_GRAB = 1;   // positions a warp takes per visit to the work counter (1 / 4 / 16 measured: 28.9 / 31.3 / 36.7 ms at the
                               // ML-20M shape; a CTA sharing chunks of 64 / 256 consecutive positions: +20 % / +7 % — rejected)

template <int R>
__device__ __forceinline__ void ce_regs(uint64_t (&key)[R], uint32_t (&pos)[R], int i, int j, bool up) {
    const bool j_before_i = rec_before(key[j], pos[j], key[i], pos[i]);
    if (j_before_i == up) {
        const uint64_t tk = key[i]; key[i] = key[j]; key[j] = tk;
        const uint32_t tp = pos[i]; pos[i] = pos[j]; pos[j] = tp;
    }
}

template <int R, int STRIDE>
__device__ __forceinline__ void stage_regs(uint64_t (&key)[R], uint32_t (&pos)[R], int lane, int size) {
#pragma unroll
    for (int x = 0; x < R; x++) {
        if ((x & STRIDE) == 0) {
            const bool up = (((lane * R + x) & size) == 0);
            ce_regs<R>(key, pos, x, x | STRIDE, up);
        }
    }
}

// blocked layout: element e = lane*R + x
template <int R>
__device__ __forceinline__ void warp_sort_regs(uint64_t (&key)[R], uint32_t (&pos)[R], int lane) {
#pragma unroll 1
    for (int size = 2; size <= 32 * R; size <<= 1) {
#pragma unroll 1
        for (int stride = size >> 1; stride >= R; stride >>= 1) {
            const int lm = stride / R;
            const bool lower = (lane & lm) == 0;
#pragma unroll
            for (int x = 0; x < R; x++) {
                const bool up = (((lane * R + x) & size) == 0);
                const uint64_t ok = __shfl_xor_sync(0xffffffffu, key[x], lm);
                const uint32_t op = __shfl_xor_sync(0xffffffffu, pos[x], lm);
                const bool other_before = rec_before(ok, op, key[x], pos[x]);
                if (other_before == (up == lower)) { key[x] = ok; pos[x] = op; }
            }
        }
        if (R >= 16 && size >= 16) stage_regs<R, (R >= 16 ? 8 : 0)>(key, pos, lane, size);
        if (R >= 8 && size >= 8) stage_regs<R, (R >= 8 ? 4 : 0)>(key, pos, lane, size);
        if (R >= 4 && size >= 4) stage_regs<R, (R >= 4 ? 2 : 0)>(key, pos, lane, size);
        if (R >= 2) stage_regs<R, (R >= 2 ? 1 : 0)>(key, pos, lane, size);
    }
}

// order-preserving key of a similarity, 0 for NaN (rs_sim_key of any real value is >= 2^52 - 1)

// Top 32 bits of the order-preserving key (sign, exponent, 20 mantissa bits): monotone — a larger key32
// means a larger similarity, equal key32 says nothing —, 0 for NaN.  The selection passes work on these
// (half the staging bytes, single-instruction compares and warp reductions); only a boundary bucket that
// is still too full at full 32-bit resolution sends the prediction to the exact 64-bit passes.
__device__ __forceinline__ uint32_t sim_key32(double s) {
    if (!(s == s)) return 0u;
    const uint32_t hi = (uint32_t)__double2hiint(s + 0.0);        // -0.0 -> +0.0
    return (hi & 0x80000000u) ? ~hi : (hi | 0x80000000u);
}

// One prediction: its candidates are the entries of a right row — `cnt` left ids a.r_col[cb ..] (ascending) with
// ratings a.r_val[cb ..] —, their similarities to the predicted left row `l` are row[id] (row l of the matrix), and
// lane 0 writes the prediction to *dst.
struct PredItem {
    int32_t l;
    int64_t cb;
    int cnt;
    const double *row;
    double *dst;
};

// The warp loop of the selection kernels: a warp takes positions w < n_eff from `work` one at a time; item(w, c)
// fills the prediction to make (returns false when it has already answered position w itself) and the warp runs
// the selection and the weighted sum on it.  Scratch per warp: hist[256], ckey / cpos / w_a [32 * R] and
// sbuf [scap] in shared memory, gbuf [scap, scap + a.gcap) in global memory.
template <int R, class Item>
__device__ __forceinline__ void select_loop(const PredArgs &a, unsigned long long *work, int64_t n_eff, const Item &item,
                                            int lane, uint32_t *hist, uint64_t *ckey, uint32_t *cpos, double *w_a,
                                            uint64_t *sbuf, uint64_t *gbuf, int scap) {
    constexpr int CAP = 32 * R;
    const double nan_v = __longlong_as_double(0x7ff8000000000001ll);
    const uint32_t lt_mask = (1u << lane) - 1u;
    for (;;) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(work, (unsigned long long)PRED_GRAB);
        base = __shfl_sync(0xffffffffu, base, 0);
        if ((int64_t)base >= n_eff) break;
        const int64_t w_end = (int64_t)base + PRED_GRAB < n_eff ? (int64_t)base + PRED_GRAB : n_eff;
        for (int64_t w = (int64_t)base; w < w_end; w++) {
            PredItem c;
            if (!item(w, c)) continue;
            const int32_t l = c.l;
            const int64_t cb = c.cb;
            const int cnt = c.cnt;
            const double *row = c.row;
            double *dst = c.dst;
            const int32_t *ids = a.r_col + cb;
            int num = 0;
            uint64_t key[R];
            uint32_t pos[R];
            bool fast_done = false;
            // ================= fast path: selection on 32-bit keys =================
            // pass A gathers every candidate's similarity ONCE and stages its key32 (4 B: shared memory for the
            // first 2*scap candidates, the per-warp global slice beyond); a radix selection on the staged key32
            // finds a threshold with num <= #{key32 >= thr} <= CAP; those survivors are gathered again (<= CAP
            // exact values, L2 hits) and sorted under the exact order (key64 desc, position asc).  Exact: a larger
            // key32 implies a larger key64, so the survivors contain the true top `num`.
            {
                uint32_t *s32 = reinterpret_cast<uint32_t *>(sbuf);
                const int cap32 = 2 * scap;
                uint32_t *g32 = reinterpret_cast<uint32_t *>(gbuf + scap) - cap32;     // g32[e], e >= cap32, lives in the warp's slice
                uint32_t kmax = 0u, kmin = 0xffffffffu;
                int valid = 0;
                __syncwarp();   // the previous prediction has finished with the stage
                for (int e0 = 0; e0 < cnt; e0 += 128) {
                    int32_t idv[4];
                    double sv4[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int e = e0 + u * 32 + lane;
                        idv[u] = e < cnt ? ids[e] : -1;
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) sv4[u] = idv[u] >= 0 ? row[idv[u]] : nan_v;
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int e = e0 + u * 32 + lane;
                        const uint32_t k32 = sim_key32(sv4[u]);
                        if (e < cap32) s32[e] = k32;
                        else if (e < cnt) g32[e] = k32;
                        valid += k32 != 0u;
                        kmax = k32 > kmax ? k32 : kmax;
                        kmin = (k32 != 0u && k32 < kmin) ? k32 : kmin;
                    }
                }
                valid = __reduce_add_sync(0xffffffffu, valid);
                kmax = __reduce_max_sync(0xffffffffu, kmax);
                kmin = __reduce_min_sync(0xffffffffu, kmin);
                __syncwarp();
                if (valid <= a.min_k) {                            // core/knn.go:102-104 (note <=)
                    if (lane == 0) *dst = a.global_mean;
                    continue;
                }
                num = a.k < valid ? a.k : valid;                   // core/knn.go:111-114
                uint32_t thr32 = 1u;                               // every valid key32 is >= 0x000fffff
                bool ok = true;
                if (valid > CAP) {
                    // windows of <= 256 equal buckets; the first one is the top binade (2^20 key32 units, value-linear)
                    uint32_t wlo = kmin, whi = kmax;
                    if (whi - wlo > (1u << 20)) wlo = whi - (1u << 20);
                    int sure = 0;
                    for (;;) {
                        const uint32_t width = whi - wlo;
                        const int sh = width < 256u ? 0 : (32 - __clz(width)) - 8;
                        for (int x = lane; x < 256; x += 32) hist[x] = 0;
                        __syncwarp();
                        for (int e = lane; e < cnt; e += 32) {
                            const uint32_t k32 = e < cap32 ? s32[e] : g32[e];
                            if (k32 >= wlo && k32 <= whi) atomicAdd(&hist[(k32 - wlo) >> sh], 1u);
                        }
                        __syncwarp();
                        uint32_t h[8], mine = 0;
#pragma unroll
                        for (int x = 0; x < 8; x++) { h[x] = hist[8 * lane + x]; mine += h[x]; }
                        uint32_t above = mine;   // inclusive suffix over lanes
#pragma unroll
                        for (int o = 1; o < 32; o <<= 1) {
                            const uint32_t v = __shfl_down_sync(0xffffffffu, above, o);
                            if (lane + o < 32) above += v;
                        }
                        const int in_window = (int)__shfl_sync(0xffffffffu, above, 0);
                        above -= mine;           // candidates in buckets of higher lanes
                        const int need = num - sure;
                        if (in_window < need) {  // the whole window is selected; continue below it
                            sure += in_window;
                            whi = wlo - 1u;
                            wlo = kmin;
                            continue;
                        }
                        int myT = -1;
                        uint32_t run = above, sure_here = 0, bd_here = 0;
#pragma unroll
                        for (int x = 7; x >= 0; x--) {
                            if (myT < 0 && run + h[x] >= (uint32_t)need) { myT = 8 * lane + x; sure_here = run; bd_here = h[x]; }
                            run += h[x];
                        }
                        const uint32_t has = __ballot_sync(0xffffffffu, myT >= 0);
                        const int src = 31 - __clz(has);           // highest lane that found it
                        const int T = __shfl_sync(0xffffffffu, myT, src);
                        const int sure_lvl = (int)__shfl_sync(0xffffffffu, sure_here, src);
                        const int bd = (int)__shfl_sync(0xffffffffu, bd_here, src);
                        const uint32_t b_lo = wlo + ((uint32_t)T << sh);
                        if (sure + sure_lvl + bd <= CAP) { thr32 = b_lo; break; }
                        sure += sure_lvl;
                        if (sh == 0) { ok = false; break; }        // one key32 value fills the bucket: exact passes
                        const uint32_t b_hi = b_lo + ((1u << sh) - 1u);
                        wlo = b_lo;
                        whi = b_hi < whi ? b_hi : whi;
                    }
                }
                if (ok) {
                    // compaction of the survivors' positions (scan order = ascending inner id)
                    int have = 0;
                    for (int base = 0; base < cnt; base += 32) {
                        const int e = base + lane;
                        uint32_t k32 = 0u;
                        if (e < cnt) k32 = e < cap32 ? s32[e] : g32[e];
                        const bool take = k32 >= thr32;
                        const uint32_t m = __ballot_sync(0xffffffffu, take);
                        if (take) cpos[have + __popc(m & lt_mask)] = (uint32_t)e;
                        have += __popc(m);
                    }
                    __syncwarp();
#pragma unroll
                    for (int x = 0; x < R; x++) {
                        const int e = lane * R + x;
                        key[x] = 0ull;
                        pos[x] = 0xffffffffu;
                        if (e < have) {
                            pos[x] = cpos[e];
                            key[x] = rs_sim_key(row[ids[pos[x]]]);   // survivors are never NaN
                        }
                    }
                    __syncwarp();
                    warp_sort_regs<R>(key, pos, lane);
                    fast_done = true;
                }
            }
            if (!fast_done) {
                // ---- pass A: gather once -> order-preserving 64-bit keys (0 = NaN / absent), count + range ----
                uint64_t klo = ~0ull, khi = 0ull;
                int valid = 0;
                __syncwarp();   // the previous prediction has finished reading sbuf
                for (int e0 = 0; e0 < cnt; e0 += 128) {
                    int32_t idv[4];
                    double sv4[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int e = e0 + u * 32 + lane;
                        idv[u] = e < cnt ? ids[e] : -1;
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) sv4[u] = idv[u] >= 0 ? row[idv[u]] : nan_v;
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int e = e0 + u * 32 + lane;
                        const double sv = sv4[u];
                        const uint64_t key = (sv == sv) ? rs_sim_key(sv) : 0ull;
                        if (e < scap) sbuf[e] = key;
                        else if (e < cnt) gbuf[e] = key;
                        if (key) { valid++; klo = key < klo ? key : klo; khi = key > khi ? key : khi; }
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    valid += __shfl_xor_sync(0xffffffffu, valid, o);
                    const uint64_t ol = __shfl_xor_sync(0xffffffffu, klo, o), oh = __shfl_xor_sync(0xffffffffu, khi, o);
                    klo = ol < klo ? ol : klo;
                    khi = oh > khi ? oh : khi;
                }
                __syncwarp();
                if (valid <= a.min_k) {                            // core/knn.go:102-104 (note <=)
                    if (lane == 0) *dst = a.global_mean;
                    continue;
                }
                num = a.k < valid ? a.k : valid;                   // core/knn.go:111-114

                // ---- pass B: radix selection on the keys: narrow to <= CAP candidates holding the top `num` ----
                // The window [klo, khi] is cut into <= 256 equal buckets ((key - klo) >> sh); the boundary
                // bucket is the highest T with count(bucket >= T) >= need.  If everything from T upwards
                // fits the register capacity the threshold is klo + (T << sh) and ONE compare selects;
                // otherwise the window shrinks to bucket T (8 more key bits per level, so it terminates: a
                // bucket of one key value that still does not fit is a genuine tie and is taken in scan
                // order = ascending inner id, the canonical policy).
                uint64_t thr = 1ull;       // take every key >= thr ...
                uint64_t tie_key = 0ull;   // ... and, when tie_take >= 0, the first tie_take keys == tie_key (< thr)
                int tie_take = -1;
                if (valid > CAP) {
                    int sure = 0;          // candidates above the window, already known to be in the top `num`
                    bool top_binade = true;
                    for (;;) {
                        // Keys are linear in the similarity inside one binade and logarithmic across binades,
                        // so the first window is the top binade only ([max/2, max], 2^52 key units): the top k
                        // of a neighbourhood almost always lie there and get 256 value-linear buckets.  If the
                        // window holds fewer than `need` they are all selected and the search goes on below it.
                        uint64_t wlo = klo;
                        if (top_binade && khi - klo > (1ull << 52)) wlo = khi - (1ull << 52);
                        top_binade = false;
                        const uint64_t width = khi - wlo;
                        const int sh = width < 256ull ? 0 : (64 - __clzll((long long)width)) - 8;
                        for (int x = lane; x < 256; x += 32) hist[x] = 0;
                        __syncwarp();
                        for (int e = lane; e < cnt; e += 32) {
                            const uint64_t key = e < scap ? sbuf[e] : gbuf[e];
                            if (key >= wlo && key <= khi) atomicAdd(&hist[(uint32_t)((key - wlo) >> sh)], 1u);
                        }
                        __syncwarp();
                        // suffix counts: lane owns buckets [8*lane, 8*lane+8)
                        uint32_t h[8], mine = 0;
#pragma unroll
                        for (int x = 0; x < 8; x++) { h[x] = hist[8 * lane + x]; mine += h[x]; }
                        uint32_t above = mine;   // inclusive suffix over lanes
#pragma unroll
                        for (int o = 1; o < 32; o <<= 1) {
                            const uint32_t v = __shfl_down_sync(0xffffffffu, above, o);
                            if (lane + o < 32) above += v;
                        }
                        const int in_window = (int)__shfl_sync(0xffffffffu, above, 0);
                        above -= mine;           // candidates in buckets of higher lanes
                        const int need = num - sure;
                        if (in_window < need) {  // the whole window is selected; continue below it
                            sure += in_window;
                            khi = wlo - 1ull;
                            continue;
                        }
                        int myT = -1;
                        uint32_t run = above, sure_here = 0, bd_here = 0;
#pragma unroll
                        for (int x = 7; x >= 0; x--) {
                            if (myT < 0 && run + h[x] >= (uint32_t)need) { myT = 8 * lane + x; sure_here = run; bd_here = h[x]; }
                            run += h[x];
                        }
                        const uint32_t has = __ballot_sync(0xffffffffu, myT >= 0);
                        const int src = 31 - __clz(has);           // highest lane that found it
                        const int T = __shfl_sync(0xffffffffu, myT, src);
                        const int sure_lvl = (int)__shfl_sync(0xffffffffu, sure_here, src);
                        const int bd = (int)__shfl_sync(0xffffffffu, bd_here, src);
                        const uint64_t b_lo = wlo + ((uint64_t)T << sh);
                        if (sure + sure_lvl + bd <= CAP) { thr = b_lo; break; }      // compaction fits
                        sure += sure_lvl;
                        if (sh == 0) {             // one key value fills the bucket: genuine ties
                            tie_key = b_lo;
                            tie_take = num - sure;
                            thr = b_lo + 1ull;
                            break;
                        }
                        // shrink the window to the keys actually present in the boundary bucket: similarity
                        // data is full of exact ties (27 % of the item-item Pearson values are +-1.0), and a
                        // bucket holding one repeated value is recognised here in ONE pass instead of being
                        // narrowed 8 key bits at a time
                        const uint64_t b_hi = b_lo + ((1ull << sh) - 1ull);
                        uint64_t nlo = ~0ull, nhi = 0ull;
                        for (int e = lane; e < cnt; e += 32) {
                            const uint64_t key = e < scap ? sbuf[e] : gbuf[e];
                            if (key >= b_lo && key <= b_hi && key <= khi) { nlo = key < nlo ? key : nlo; nhi = key > nhi ? key : nhi; }
                        }
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            const uint64_t ol = __shfl_xor_sync(0xffffffffu, nlo, o), oh = __shfl_xor_sync(0xffffffffu, nhi, o);
                            nlo = ol < nlo ? ol : nlo;
                            nhi = oh > nhi ? oh : nhi;
                        }
                        klo = nlo;
                        khi = nhi;
                        if (nlo == nhi) {          // one key value fills the bucket: genuine ties
                            tie_key = nlo;
                            tie_take = num - sure;
                            thr = nlo + 1ull;
                            break;
                        }
                    }
                }

                // ---- pass C: compaction (scan order = ascending inner id) ----
                int have = 0, ties_taken = 0;
                for (int base = 0; base < cnt; base += 32) {
                    const int e = base + lane;
                    uint64_t key = 0ull;
                    if (e < cnt) key = e < scap ? sbuf[e] : gbuf[e];
                    bool take = key >= thr;
                    if (tie_take >= 0) {
                        const bool tie = key == tie_key;
                        const uint32_t tm = __ballot_sync(0xffffffffu, tie);
                        if (tie && ties_taken + __popc(tm & lt_mask) < tie_take) take = true;
                        ties_taken += __popc(tm);
                    }
                    const uint32_t m = __ballot_sync(0xffffffffu, take);
                    if (take) {
                        const int slot = have + __popc(m & lt_mask);
                        ckey[slot] = key;
                        cpos[slot] = (uint32_t)e;
                    }
                    have += __popc(m);
                }
                __syncwarp();

                // ---- sort the survivors in registers ----
#pragma unroll
                for (int x = 0; x < R; x++) {
                    const int e = lane * R + x;
                    key[x] = e < have ? ckey[e] : 0ull;
                    pos[x] = e < have ? cpos[e] : 0xffffffffu;
                }
                __syncwarp();
                warp_sort_regs<R>(key, pos, lane);

            }

            // ---- weighted mean over the first `num`, sequential in sorted order ----
            // the sorted (similarity, adjusted rating) pairs go through shared memory so that the
            // serial accumulation is two broadcast loads and three FP64 operations per neighbour
            double *w_s = reinterpret_cast<double *>(ckey);
#pragma unroll
            for (int x = 0; x < R; x++) {
                const int e = lane * R + x;
                if (e < num) {
                    const int32_t id = ids[pos[x]];
                    const double s = rs_key_sim(key[x]);          // the exact similarity the record was sorted by
                    double rating = a.r_val[cb + pos[x]];
                    if (a.knn_type == RS_KNN_CENTERED) rating -= a.means[id];                       // core/knn.go:121
                    else if (a.knn_type == RS_KNN_ZSCORE) rating = (rating - a.means[id]) / a.stddevs[id];
                    else if (a.knn_type == RS_KNN_BASELINE) rating -= a.bias[id];
                    w_s[e] = s;
                    w_a[e] = rating;
                    if (a.nb_ids && e < a.nb_cap) { a.nb_ids[e] = id; a.nb_sims[e] = s; }   // +-0 as +0: see nb_cells_kernel
                }
            }
            __syncwarp();
            double wsum = 0.0, wrat = 0.0;
#pragma unroll 4
            for (int e = 0; e < num; e++) {
                const double sq = w_s[e], aq = w_a[e];
                wsum += sq;                                        // core/knn.go:117
                wrat += sq * aq;                                   // core/knn.go:127
            }
            __syncwarp();
            if (lane == 0) {
                double pred = wrat / wsum;                         // core/knn.go:131
                if (a.knn_type == RS_KNN_CENTERED) pred += a.means[l];
                else if (a.knn_type == RS_KNN_BASELINE) pred += a.bias[l];
                else if (a.knn_type == RS_KNN_ZSCORE) { pred *= a.stddevs[l]; pred += a.means[l]; }
                *dst = pred;
                if (a.nb_count) *a.nb_count = num < a.nb_cap ? num : a.nb_cap;
            }
        }
    }
}

}  // namespace
