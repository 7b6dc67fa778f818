// sim_stream.cu — exact-order FP64 similarity kernel ("stream" path).
//
// Reproduces core/sim.go (Cosine :10-25, MSD :28-44, Pearson :47-81) bit for bit.  For a left
// row i the reference walks i's entries in ascending right id c and, for every other left row
// j that also rated c, adds one term to each of three running sums — in that order.
//
// Mapping ("column walk"): one WARP owns a work item (row i, chunk of JC = 128 or 256 consecutive columns j)
// and keeps that chunk's accumulators in shared memory.  It walks row i's entries in ascending
// c; for each c the raters of c that fall in the chunk are a CONTIGUOUS slice of c's id-sorted
// list in the right CSR (chunk pointers `cp`, precomputed), so the lanes read (j, b-side term)
// coalesced and update acc[j] — every j at most once per c, and c strictly in order, so each
// accumulator receives exactly the reference's terms in the reference's order with the same
// IEEE operations (the library is built with --fmad=false).  With the full matrix only j > i
// is visited (the slice starts right after i's own position in c's list, `l2r`); the mirror
// pass fills j < i.  Work = the co-rated triples; no N x nnz term anywhere.
//
// Bound: shared-memory RMW bandwidth (6 accesses per triple, random banks) and L2 reads of
// 12 B per triple; see DESIGN.md and profiles/.
//
// The longest rows ("popular columns") are taken out of that walk: their pairs are dense work items of the same
// kernel and queue (pop_item below: lane = column, accumulators in registers), see the comment there.
#include "common.cuh"
#include "sim_terms.cuh"

namespace {

constexpr int SW = RS_STREAM_WARPS;        // warps per CTA, each an independent work item

struct StreamArgs {
    const int64_t *l_ptr;
    const int32_t *l_col;
    const double *l_val;
    const int64_t *l2r;       // left-CSR entry (i,c) -> index of (c,i) in the right CSR
    const int64_t *r_ptr;
    const int32_t *r_col;
    const double *r_dev;      // b-side term per right-CSR entry (rating, or rating - row mean, ...)
    const int32_t *row_order; // left rows of the shard, longest first (load balance)
    const int32_t *cp;        // [n_right][Q+1] offsets (relative to r_ptr[c]) of the chunk boundaries
    int32_t n_chunks;         // Q
    const double *pmeans;
    const double *left_bias, *right_bias;
    double global_bias, shrinkage;
    double *sims;
    int64_t ld_s;
    int32_t n_left;
    int64_t row_begin, row_end;
    int64_t n_rows;           // rows of row_order to walk
    int cyc_R;                // >= 2: cyclic row shards, the output row is rs_cyc_local(i)
    int symmetric;            // 0: full rows; 1: only columns j > i are computed; 2: only j < i (the mirror pass fills the rest)
    // popular columns split off (else null): the CSR this walk reads holds the other rows under their labels
    // (rank - n_pop), so chunks, triangles and the diagonal are in label space and lab_row maps a label back
    const int32_t *rank;
    const int32_t *lab_row;
    int32_t n_pop;
    unsigned long long *counter;
};

constexpr int G = 8;   // columns whose first 32 raters are loaded together (must divide 32)

// ---------------------------------------------------------------------------------------------
// Popular columns.  The column walk below serialises a row's entries in ONE warp, so the few rows that a large
// part of the right ids rated (78 k of 138 k on the MovieLens-20M shape) are chains of tens of thousands of
// dependent steps, and as COLUMNS they fill the other rows' runs with most of the triples (the 312 longest of
// 26,744 rows hold 34 % of the ratings and take part in 56 % of the co-rated triples).  rs_prep_rt takes their
// ratings out of the CSR the walk reads and lays them out as a dense table D[right id][popular column]; every
// pair with a popular column is computed from it by a second kind of work item of the same kernel:
//   (row i, block of 32 popular columns), one warp; LANE = column, accumulators in registers; the warp walks
//   row i's entries in ascending right id c — the reference's order (core/sim.go:14-22) —, each step is ONE
//   coalesced load of D[c][block] (independent of the accumulators: 16 or 8 in flight) and, in the lanes whose column c
//   rated, the reference's IEEE operations on the lane's own sums.
// No lookups, no gathers, no shared-memory read-modify-writes, and no item depends on another: a row of 78 k
// entries is 10 items of 78 k pipelined steps.  Who computes which pair (the mirror passes copy the transposed
// cell): a popular column's pairs with every other row belong to THAT row; two popular rows: to the one further
// down the popular list (the shorter one); two other rows: the triangle rule of the column walk over their labels.

struct PopArgs {
    const int32_t *rows;      // the shard's rows, longest first: the popular ones come first
    int64_t n_rows;
    const int32_t *rank;      // [n_left] position in the longest-first order: < n_pop is the index in the popular list
    int32_t n_pop;
    const int32_t *pop_items; // [32 * n_blk] row id, -1 beyond the list
    int32_t n_blk, ld;        // blocks of 32 popular columns; row stride of the table
    const void *dense;
    int64_t n_first;          // dense items of the shard's popular rows: they open the work queue (longest chains)
};

__device__ __forceinline__ void pop_cp_async16(void *dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void pop_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void pop_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// One dense item.  `scratch`: 3 KB of the warp's shared memory (its accumulator area): per batch of 32 entries the
// a-side terms {ra, ra^2} [32][2], the right rows' biases [32], the right ids [32], and — byte table — two buffers
// of 32 x 32 table bytes filled by cp.async one batch ahead (two 16-byte copies per lane and batch; the right ids
// are loaded two batches ahead), so the chain of a long row is bound by its own arithmetic, not by memory latency.
// The per-entry arithmetic is branch-free: every lane computes its b-side term and products, only the three
// additions are predicated on "this column was rated" — the unrolled entries overlap in the FP64 pipe.
template <int SIM, bool SHRINK, typename DT>
__device__ __forceinline__ void pop_item(const StreamArgs &a, const PopArgs &pa, int64_t item, double *scratch, int lane) {
    constexpr bool U8 = sizeof(DT) == 1;
    double2 *s_a = reinterpret_cast<double2 *>(scratch);                          // {ra, ra * ra}
    double *s_rbias = scratch + 64;
    int32_t *s_c = reinterpret_cast<int32_t *>(scratch + 96);
    uint8_t *s_d = reinterpret_cast<uint8_t *>(scratch + 112);                    // [2][32][32]
    const DT *__restrict__ dense = static_cast<const DT *>(pa.dense);
    const double nan_v = __longlong_as_double(0x7ff8000000000001ll);
    const int32_t i = pa.rows[item / pa.n_blk];
    const int b = (int)(item % pa.n_blk);
    const int pi = pa.rank[i] < pa.n_pop ? pa.rank[i] : -1;
    if (pi >= 0 && 32 * b > pi) return;                       // a popular row: only the columns above it in the list
    const int col = 32 * b + lane;
    const int32_t hcol = pa.pop_items[col];
    const bool want = hcol >= 0 && (pi < 0 || col < pi);
    double bh = 0.0;                                          // what is subtracted from the column's ratings
    if (want && SIM == RS_SIM_PEARSON) bh = a.pmeans[hcol];
    if (want && SIM == RS_SIM_PEARSON_BASELINE) bh = a.global_bias + a.left_bias[hcol];
    double ai = 0.0;
    if (SIM == RS_SIM_PEARSON) ai = a.pmeans[i];
    if (SIM == RS_SIM_PEARSON_BASELINE) ai = a.global_bias + a.left_bias[i];
    double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
    const int64_t eb = a.l_ptr[i], ee = a.l_ptr[i + 1];

    // the reference's operations on the lane's sums for one entry; `rated` predicates the additions only
    auto apply = [&](bool rated, double rb, const double2 aa, double rbias_u) {
        (void)rbias_u;
        if (SIM == RS_SIM_MSD) {
            const double dd = aa.x - rb;
            const double t = dd * dd;
            if (rated) { acc0 += t; acc1 += 1.0; }                                // core/sim.go:37-38
        } else {
            const double t1 = rb * rb, t2 = aa.x * rb;
            if (rated) {
                acc0 += aa.y;                                                     // core/sim.go:19 / :75
                acc1 += t1;                                                       // core/sim.go:20 / :76
                acc2 += t2;                                                       // core/sim.go:21 / :77
                if (SHRINK) acc3 += 1.0;
            }
        }
    };

    if (__any_sync(0xffffffffu, want)) {
        // batch k: entries [eb + 32 k, ...); (c, v) in registers for batches k and k + 1, loads of k + 2 in flight
        int32_t c_0 = 0, c_1 = 0;
        double v_0 = 0.0, v_1 = 0.0;
        if (eb + lane < ee) { c_0 = a.l_col[eb + lane]; v_0 = a.l_val[eb + lane]; }
        if (eb + 32 + lane < ee) { c_1 = a.l_col[eb + 32 + lane]; v_1 = a.l_val[eb + 32 + lane]; }
        // copies of one batch: piece p = lane, lane + 32 is half (p & 1) of entry p >> 1
        auto issue = [&](int32_t c_l, int64_t x0, int buf) {
            if constexpr (U8) {
#pragma unroll
                for (int h2 = 0; h2 < 2; h2++) {
                    const int p = lane + 32 * h2, u = p >> 1;
                    const int32_t c_u = __shfl_sync(0xffffffffu, c_l, u);
                    if (x0 + u < ee)
                        pop_cp_async16(s_d + buf * 1024 + 32 * u + 16 * (p & 1),
                                       reinterpret_cast<const uint8_t *>(dense) + (int64_t)c_u * pa.ld + 32 * b + 16 * (p & 1));
                }
            }
            pop_commit();
        };
        __syncwarp();
        issue(c_0, eb, 0);
        int buf = 0;
        for (int64_t x0 = eb; x0 < ee; x0 += 32, buf ^= 1) {
            const int32_t c = c_0;
            const double v = v_0;
            c_0 = c_1; v_0 = v_1;
            c_1 = 0; v_1 = 0.0;
            if (x0 + 64 + lane < ee) { c_1 = a.l_col[x0 + 64 + lane]; v_1 = a.l_val[x0 + 64 + lane]; }
            double ra = 0.0, rbias = 0.0;
            if (x0 + lane < ee) {
                if (SIM == RS_SIM_PEARSON) ra = v - ai;                           // core/sim.go:73
                else if (SIM == RS_SIM_PEARSON_BASELINE) { rbias = a.right_bias[c]; const double bb = ai + rbias; ra = v - bb; }
                else ra = v;
            }
            s_a[lane] = make_double2(ra, ra * ra);                                // core/sim.go:19 / :75
            if (SIM == RS_SIM_PEARSON_BASELINE) s_rbias[lane] = rbias;
            if (!U8) s_c[lane] = c;
            issue(c_0, x0 + 32, buf ^ 1);                     // the next batch, into the buffer the previous one left
            pop_wait<1>();                                    // this batch has landed (this lane's copies) ...
            __syncwarp();                                     // ... and every lane's; the staged terms are visible
            const int lim = (ee - x0) < 32 ? (int)(ee - x0) : 32;
            if constexpr (U8) {
                const uint8_t *sd = s_d + buf * 1024 + lane;
#pragma unroll 8
                for (int u = 0; u < lim; u++) {
                    const int code = want ? (int)sd[32 * u] : 0;
                    // code -> rating without a conversion: 2^52 + 2^51 + code as a double, minus 2^52 + 2^51 + bias (exact)
                    const double y = __hiloint2double(0x43380000, code) - (6755399441055744.0 + (double)RS_INT8_BIAS);
                    const double2 aa = s_a[u];
                    double rb;                                                    // the b-side term, as build_rdev_kernel (prep.cu)
                    double rbias_u = 0.0;
                    if (SIM == RS_SIM_PEARSON) rb = y - bh;                       // core/sim.go:74
                    else if (SIM == RS_SIM_PEARSON_BASELINE) { rbias_u = s_rbias[u]; const double bb = bh + rbias_u; rb = y - bb; }
                    else rb = y;
                    apply(code != 0, rb, aa, rbias_u);
                }
            } else {
                constexpr int PU = 8;                                             // table loads in flight
                for (int u0 = 0; u0 < lim; u0 += PU) {
                    double d[PU];
#pragma unroll
                    for (int g = 0; g < PU; g++) {
                        d[g] = nan_v;
                        if (want && u0 + g < lim) d[g] = dense[(int64_t)s_c[u0 + g] * pa.ld + col];
                    }
#pragma unroll
                    for (int g = 0; g < PU; g++) {
                        const int u = (u0 + g) & 31;
                        apply(d[g] == d[g], d[g], s_a[u], 0.0);
                    }
                }
            }
            __syncwarp();                                     // the batch has been read: its buffer and the staged terms are free
        }
        pop_wait<0>();
    }

    if (hcol >= 0) {
        double *out = a.sims + (a.cyc_R > 1 ? rs_cyc_local(i, a.cyc_R) : (int64_t)(i - a.row_begin)) * a.ld_s;
        if (pi >= 0 && col == pi) {
            out[hcol] = nan_v;                                                    // diagonal stays NaN
        } else if (want) {
            const double acc_r[4] = {acc0, acc1, acc2, acc3};
            out[hcol] = sim_value<SIM, SHRINK>(acc_r, 1, a.shrinkage);                        // core/sim.go:43 / :24 / :80
        }
    }
}

// SYM = 1: the full matrix is being computed, only columns j > i are visited (the run starts right
// after i's own position in c's list) and the mirror pass fills j < i.  SYM = 2: only columns j < i
// (the run ends at i's own position).  Which triangle is cheaper depends on how the row lengths
// correlate with the ids: a row pays one lookup per (entry, chunk) it visits, so long rows should
// visit few chunks — with first-appearance ids the popular rows have the LOW ids and the lower
// triangle costs 3.5x fewer lookups on the MovieLens-20M shape (rs_prep_rt picks per Fit).
// SYM = 0 (row shard): the whole run is visited and the diagonal pair (i,i) is skipped by index.
// Indices into the right CSR are kept in 32 bits inside the loop (nnz < 2^32 is checked at launch)
// and the per-entry a-side terms are staged in shared memory, which halves the instructions per
// column against the first version of this kernel (profiles/r01_stream_notes.md).
// POP = 1 / 2: popular columns were split off (table of bytes / of doubles): the queue holds the dense items of the
// shard's popular rows (the longest chains) first, then the column-walk items, then the dense items of the other rows.
// The walk's columns are then the LABELS of the other rows, longest first (rs_knn::rank): chunk q covers labels
// [q JC, (q + 1) JC), the triangle is taken in label space, so the lower one visits few chunks for the long rows,
// and the epilogue scatters the chunk's cells to the rows lab_row[label].
template <int SIM, bool SHRINK, int SYM, int JC, int POP>
__global__ void __launch_bounds__(SW * 32, 4) sim_stream_kernel(StreamArgs a, PopArgs pa) {
    constexpr int NACC = SHRINK ? 4 : 3;
    extern __shared__ double s_acc_all[];                    // [SW][NACC][JC] accumulators, then [SW][32] a-side terms
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *acc = s_acc_all + (size_t)warp * NACC * JC;
    double *s_ra = s_acc_all + (size_t)SW * NACC * JC + warp * 32;
    const int64_t Q = a.n_chunks;
    const int64_t n_items = a.n_rows * Q;
    const double nan_v = __longlong_as_double(0x7ff8000000000001ll);
    const int32_t *__restrict__ r_col = a.r_col;
    const double *__restrict__ r_dev = a.r_dev;

    for (;;) {
        unsigned long long item = 0;
        if (lane == 0) item = atomicAdd(a.counter, 1ull);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (POP) {
            int64_t d = (int64_t)item;
            if (d >= pa.n_first) d = d >= pa.n_first + n_items ? d - n_items : -1;
            if (d >= pa.n_rows * pa.n_blk) break;
            if (d >= 0) {
                __syncwarp();
                if (POP == 1) pop_item<SIM, SHRINK, uint8_t>(a, pa, d, acc, lane);
                else pop_item<SIM, SHRINK, double>(a, pa, d, acc, lane);
                __syncwarp();
                continue;
            }
            item -= (unsigned long long)pa.n_first;
        } else if ((int64_t)item >= n_items) break;
        // items are ordered longest row first, so the critical path starts early
        const int64_t q = (int64_t)item % Q;
        const int32_t i = a.row_order[(int64_t)item / Q];
        const int32_t li = POP ? a.rank[i] - a.n_pop : i;   // i's own column
        const int j0 = (int)(q * JC);
        if (SYM == 1 && j0 + JC <= li) continue;  // every column of the chunk is < li
        if (SYM == 2 && j0 > li) continue;        // every column of the chunk is > li

        for (int x = lane; x < NACC * JC; x += 32) acc[x] = 0.0;

        double ai = 0.0;
        if (SIM == RS_SIM_PEARSON) ai = a.pmeans[i];
        if (SIM == RS_SIM_PEARSON_BASELINE) ai = a.global_bias + a.left_bias[i];

        const int64_t eb = a.l_ptr[i], ee = a.l_ptr[i + 1];
        for (int64_t x0 = eb; x0 < ee; x0 += 32) {
            // each lane prepares one entry (c, x) of row i: its a-side term and its run of c's list
            const int64_t e = x0 + lane;
            double ra = 0.0;
            uint32_t lo = 0, self = 0xffffffffu;
            int n = 0;
            if (e < ee) {
                const int32_t c = a.l_col[e];
                const double v = a.l_val[e];
                if (SIM == RS_SIM_PEARSON) ra = v - ai;                           // core/sim.go:73
                else if (SIM == RS_SIM_PEARSON_BASELINE) { const double bb = ai + a.right_bias[c]; ra = v - bb; }
                else ra = v;
                const int64_t rp = a.r_ptr[c];
                const int32_t *cpc = a.cp + (int64_t)c * (Q + 1) + q;
                int64_t lo64 = rp + cpc[0];
                int64_t hi = rp + cpc[1];
                const int64_t self64 = a.l2r[e];
                if (SYM == 1) { if (self64 + 1 > lo64) lo64 = self64 + 1; }       // only j > i
                else if (SYM == 2) { if (self64 < hi) hi = self64; }              // only j < i
                else self = (uint32_t)self64;
                n = hi > lo64 ? (int)(hi - lo64) : 0;
                lo = (uint32_t)lo64;
            }
            __syncwarp();           // the previous batch has finished with acc and s_ra
            s_ra[lane] = ra;
            __syncwarp();
            const int lim = (ee - x0) < 32 ? (int)(ee - x0) : 32;
            // Columns are processed in order, G at a time: the (j, b-side) pairs of the first 32
            // raters of G consecutive columns are loaded up front (independent L2 requests in
            // flight), then applied column by column.
            for (int u0 = 0; u0 < lim; u0 += G) {
                int jj[G], nn[G];
                double rbv[G];
#pragma unroll
                for (int g = 0; g < G; g++) {
                    const int u = u0 + g;                                           // < 32 always (G divides 32)
                    nn[g] = __shfl_sync(0xffffffffu, n, u);                         // 0 for u >= lim
                    const uint32_t lo_u = __shfl_sync(0xffffffffu, lo, u);
                    uint32_t self_u = 0xffffffffu;
                    if (!SYM) self_u = __shfl_sync(0xffffffffu, self, u);
                    jj[g] = -1;
                    rbv[g] = 0.0;
                    if (lane < nn[g]) {
                        const uint32_t idx = lo_u + (uint32_t)lane;
                        if (SYM || idx != self_u) {                                 // the diagonal pair (i,i)
                            jj[g] = r_col[idx] - j0;
                            rbv[g] = r_dev[idx];                                    // jr | jr - meanB (core/sim.go:74)
                        }
                    }
                }
#pragma unroll
                for (int g = 0; g < G; g++) {
                    if (nn[g] == 0) continue;                                       // warp-uniform
                    const double ra_u = s_ra[u0 + g];
                    const double raa_u = ra_u * ra_u;                               // core/sim.go:19 / :75
                    if (jj[g] >= 0) stream_update<SIM, SHRINK, JC>(acc, jj[g], ra_u, raa_u, rbv[g]);
                    if (nn[g] > 32) {                                               // long run: remaining raters
                        const uint32_t lo_u = __shfl_sync(0xffffffffu, lo, u0 + g);
                        uint32_t self_u = 0xffffffffu;
                        if (!SYM) self_u = __shfl_sync(0xffffffffu, self, u0 + g);
                        for (int t = lane + 32; t < nn[g]; t += 32) {
                            const uint32_t idx = lo_u + (uint32_t)t;
                            if (!SYM && idx == self_u) continue;
                            stream_update<SIM, SHRINK, JC>(acc, r_col[idx] - j0, ra_u, raa_u, r_dev[idx]);
                        }
                    }
                    __syncwarp();   // column c is complete before column c+1 touches the same j
                }
            }
        }
        __syncwarp();

        // epilogue: the chunk's similarities of row i, coalesced (scattered by label with popular columns): the
        // columns below n_cols and > li (SYM 1) or <= li (SYM 2).  The POP kernels test them per column, the others
        // hoist the bounds: fewer spills in each (profiles/r03_walk_labels.md)
        double *out = a.sims + (a.cyc_R > 1 ? rs_cyc_local(i, a.cyc_R) : (int64_t)(i - a.row_begin)) * a.ld_s + (POP ? 0 : j0);
        auto emit = [&](int j, int64_t col) {
            double s = sim_value<SIM, SHRINK>(acc + j, JC, a.shrinkage);                 // core/sim.go:43 / :24 / :80
            if (col == (int64_t)li) s = nan_v;                                    // diagonal stays NaN
            out[POP ? a.lab_row[col] : j] = s;
        };
        if (POP) {
            for (int j = lane; j < JC; j += 32) {
                const int64_t col = (int64_t)j0 + j;
                if (col >= a.n_left - a.n_pop) break;
                if (SYM == 1 && col < li) continue;                                   // mirror pass writes it
                if (SYM == 2 && col > li) break;
                emit(j, col);
            }
        } else {
            int j_end = a.n_left - j0;
            if (SYM == 2 && li - j0 + 1 < j_end) j_end = li - j0 + 1;
            if (j_end > JC) j_end = JC;
            const int j_beg = SYM == 1 && li > j0 ? li - j0 : 0;
            for (int j = j_beg + lane; j < j_end; j += 32) emit(j, j0 + j);
        }
        __syncwarp();
    }
}

// does row r's own pass (its column-walk or dense items in sim_stream_kernel) compute cell (r, c)?  rr / rc: the
// rows' ranks.  The row further down the longest-first order owns the pair; with the upper triangle two walked rows
// swap.
__device__ __forceinline__ bool pop_owns(int32_t rr, int32_t rc, int32_t n_pop, int lower) {
    if (!lower && rr >= n_pop && rc >= n_pop) return rr < rc;
    return rr > rc;
}

// Mirror the computed upper block-triangle into the lower one: the three similarities are
// bit-symmetric (sums and products commute), which is why the reference can write
// Sims[j][i] = Sims[i][j] (core/knn.go:205-208).  32x32 tiles through shared memory,
// coalesced on both sides.  `chunk` is the column-chunk width the producer skipped by.
// lower = 1: the producer computed j < i, the destinations are the cells right of the diagonal.
__global__ void symmetrize_kernel(double *__restrict__ s, int64_t ld, int32_t n, int lower) {
    __shared__ double tile[32][33];
    int64_t bi = blockIdx.y, bj = blockIdx.x;                // destination tile (rows bi, cols bj)
    if (bj > bi) return;                                     // one block per unordered tile pair
    if (lower) { const int64_t t = bi; bi = bj; bj = t; }
    const int64_t r0 = bi * 32, c0 = bj * 32;
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        int64_t sr = c0 + y, sc = r0 + threadIdx.x;          // source = transposed position
        tile[y][threadIdx.x] = (sr < n && sc < n) ? s[sr * ld + sc] : 0.0;
    }
    __syncthreads();
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        int64_t r = r0 + y, c = c0 + threadIdx.x;
        if (r < n && c < n && (lower ? c > r : c < r)) s[r * ld + c] = tile[threadIdx.x][y];
    }
}

// Cyclic row shards: every shard computed one triangle of ITS rows (lower = 1: the cells j < i); the
// other triangle of a row is the transpose of cells that live in the rows of other shards.  One CTA
// moves one 32 x 32 tile: it reads the source tile from the owner's matrix — peer memory over NVLink
// when the owner is another GPU, 256 contiguous bytes per row —, transposes it in shared memory and
// writes it into this shard's rows.  This is the one exchange step of the sharded Fit: half the
// matrix crosses the links once, pulled by the consumers (no staging buffer, no pack / unpack).
struct MirrorArgs {
    double *self;
    const double *peer[RS_MAX_PEERS];
    int64_t ld;
    int32_t n;
    int32_t count, index, lower;
};
__global__ void mirror_kernel(MirrorArgs a) {
    __shared__ double tile[32][33];
    const int64_t bI = blockIdx.y;                           // own block (local index)
    const int64_t gI = bI * a.count + a.index, gJ = blockIdx.x;
    if (a.lower ? gJ < gI : gJ > gI) return;                 // destination tiles: right of (left of) the diagonal
    const double *src = a.peer[gJ % a.count];
    const int64_t sJ = (gJ / a.count) * RS_CYC_B;            // first local row of block gJ at its owner
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int64_t sr = gJ * 32 + y, sc = gI * 32 + threadIdx.x;   // global (row, col) of the source cell
        tile[y][threadIdx.x] = (sr < a.n && sc < a.n) ? src[(sJ + y) * a.ld + sc] : 0.0;
    }
    __syncthreads();
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int64_t r = gI * 32 + y, c = gJ * 32 + threadIdx.x;
        if (r < a.n && c < a.n && (a.lower ? c > r : c < r)) a.self[(bI * 32 + y) * a.ld + c] = tile[threadIdx.x][y];
    }
}

// The same two passes when popular columns were split off: which of the cells (r, c) / (c, r) was computed is
// pop_owns() of the rows' ranks, cell by cell, so a pair of transposed tiles exchanges cells in both directions.
__global__ void symmetrize_pop_kernel(double *__restrict__ s, int64_t ld, int32_t n, int lower,
                                      const int32_t *__restrict__ rank, int32_t n_pop) {
    __shared__ double ta[32][33], tb[32][33];
    __shared__ int32_t rk_a[32], rk_b[32];
    const int64_t bi = blockIdx.y, bj = blockIdx.x;
    if (bj > bi) return;                                     // one block per unordered tile pair
    const int64_t r0 = bi * 32, c0 = bj * 32;                // tile A = rows r0.., cols c0..; tile B = rows c0.., cols r0..
    if (threadIdx.y == 0) {
        rk_a[threadIdx.x] = r0 + threadIdx.x < n ? rank[r0 + threadIdx.x] : 0;
        rk_b[threadIdx.x] = c0 + threadIdx.x < n ? rank[c0 + threadIdx.x] : 0;
    }
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int64_t ar = r0 + y, ac = c0 + threadIdx.x, br = c0 + y, bc = r0 + threadIdx.x;
        ta[y][threadIdx.x] = (ar < n && ac < n) ? s[ar * ld + ac] : 0.0;
        tb[y][threadIdx.x] = (br < n && bc < n) ? s[br * ld + bc] : 0.0;
    }
    __syncthreads();
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        int64_t r = r0 + y, c = c0 + threadIdx.x;            // a cell of A takes B's transposed cell (c, r)
        if (r < n && c < n && r != c && !pop_owns(rk_a[y], rk_b[threadIdx.x], n_pop, lower)) s[r * ld + c] = tb[threadIdx.x][y];
        if (bi == bj) continue;
        r = c0 + y; c = r0 + threadIdx.x;                    // a cell of B takes A's transposed cell
        if (r < n && c < n && !pop_owns(rk_b[y], rk_a[threadIdx.x], n_pop, lower)) s[r * ld + c] = ta[threadIdx.x][y];
    }
}

__global__ void mirror_pop_kernel(MirrorArgs a, const int32_t *__restrict__ rank, int32_t n_pop) {
    __shared__ double tile[32][33];
    const int64_t bI = blockIdx.y;                           // own block (local index)
    const int64_t gI = bI * a.count + a.index, gJ = blockIdx.x;
    bool need[4];                                            // blockDim.y == 8: four cells per thread
    bool any = false;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int y = threadIdx.y + 8 * k;
        const int64_t r = gI * 32 + y, c = gJ * 32 + threadIdx.x;
        need[k] = r < a.n && c < a.n && r != c && !pop_owns(rank[r], rank[c], n_pop, a.lower);
        any = any || need[k];
    }
    if (!__syncthreads_or(any)) return;                      // every cell of the tile is this shard's own work
    const double *src = a.peer[gJ % a.count];
    const int64_t sJ = (gJ / a.count) * RS_CYC_B;            // first local row of block gJ at its owner
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int64_t sr = gJ * 32 + y, sc = gI * 32 + threadIdx.x;   // global (row, col) of the source cell
        tile[y][threadIdx.x] = (sr < a.n && sc < a.n) ? src[(sJ + y) * a.ld + sc] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int y = threadIdx.y + 8 * k;
        if (need[k]) a.self[(bI * 32 + y) * a.ld + gJ * 32 + threadIdx.x] = tile[threadIdx.x][y];
    }
}

}  // namespace

template <int SIM, bool SHRINK, int SYM, int JC, int POP>
static int32_t launch_stream_pop(rs_knn *h, const StreamArgs &s, const PopArgs &pa, int grid) {
    const int smem = SW * ((SHRINK ? 4 : 3) * JC + 32) * (int)sizeof(double);
    auto kern = sim_stream_kernel<SIM, SHRINK, SYM, JC, POP>;
    RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<grid, SW * 32, smem, h->stream>>>(s, pa);
    return RS_OK;
}
template <int SIM, bool SHRINK, int SYM, int JC>
static int32_t launch_stream_jc(rs_knn *h, const StreamArgs &s, const PopArgs &pa, int grid) {
    if (SYM != 0 && s.rank) {                              // popular columns exist only where a triangle is computed
        if (h->pop_u8) return launch_stream_pop<SIM, SHRINK, SYM ? SYM : 1, JC, 1>(h, s, pa, grid);
        return launch_stream_pop<SIM, SHRINK, SYM ? SYM : 1, JC, 2>(h, s, pa, grid);
    }
    return launch_stream_pop<SIM, SHRINK, SYM, JC, 0>(h, s, pa, grid);
}
template <int SIM, bool SHRINK, int SYM>
static int32_t launch_stream_sym(rs_knn *h, const StreamArgs &s, const PopArgs &pa, int grid) {
    if (h->stream_jc == 128) return launch_stream_jc<SIM, SHRINK, SYM, 128>(h, s, pa, grid);
    return launch_stream_jc<SIM, SHRINK, SYM, 256>(h, s, pa, grid);
}
template <int SIM, bool SHRINK>
static int32_t launch_stream(rs_knn *h, const StreamArgs &s, const PopArgs &pa, int grid) {
    if (h->nnz >= (int64_t)0xffffffffll) {
        rs_set_error("stream path indexes the ratings with 32 bits (nnz=%lld)", (long long)h->nnz);
        return RS_ERR_UNSUPPORTED;
    }
    if (s.symmetric == 2) return launch_stream_sym<SIM, SHRINK, 2>(h, s, pa, grid);
    return s.symmetric ? launch_stream_sym<SIM, SHRINK, 1>(h, s, pa, grid) : launch_stream_sym<SIM, SHRINK, 0>(h, s, pa, grid);
}

int32_t rs_sim_stream_launch(rs_knn *h) {
    StreamArgs a{};
    a.l_ptr = h->l_ptr; a.l_col = h->l_col; a.l_val = h->l_val; a.l2r = h->l2r;
    a.r_ptr = h->r_ptr; a.r_col = h->r_col; a.r_dev = h->r_dev; a.cp = h->cp; a.n_chunks = h->n_chunks;
    const bool cyc = h->cyc_R > 1;
    // rs_prep_rt leaves the rows to walk (longest first) in row_order; in top-k-only
    // mode (n_work_rows < 0) it is the natural order and the current slab is a slice of it
    a.row_order = h->n_work_rows >= 0 ? h->row_order : h->row_order + h->row_begin;
    a.n_rows = h->n_work_rows >= 0 ? h->n_work_rows : h->row_end - h->row_begin;
    a.cyc_R = h->cyc_R;
    a.pmeans = h->pmeans; a.left_bias = h->left_bias; a.right_bias = h->right_bias;
    a.global_bias = h->global_bias; a.shrinkage = h->p.shrinkage;
    a.sims = h->sims; a.ld_s = h->ld_s; a.n_left = h->n_left;
    a.row_begin = h->row_begin; a.row_end = h->row_end;
    a.symmetric = h->force_sym ? 1 : ((h->row_begin == 0 && h->row_end == h->n_left) || cyc) ? (h->stream_lower ? 2 : 1) : 0;
    a.counter = reinterpret_cast<unsigned long long *>(h->d_flags + 2);
    RS_CUDA(cudaMemsetAsync(a.counter, 0, 8, h->stream));
    // popular columns (rs_prep_rt split them off: the walk reads the CSR without them): their pairs are dense work
    // items of the same kernel
    const bool pop = h->n_pop > 0;
    PopArgs pa{};
    if (pop) {
        if (a.symmetric == 0 || h->force_sym) {
            rs_set_error("popular columns were split off, but this Fit does not compute a triangle of the full matrix");
            return RS_ERR_INVALID;
        }
        a.r_ptr = h->w_ptr; a.r_col = h->w_col; a.r_dev = h->w_dev;
        a.rank = h->rank; a.lab_row = h->lab_row; a.n_pop = h->n_pop;
        pa.rows = h->row_all; pa.n_rows = h->n_all_rows;
        pa.rank = h->rank; pa.n_pop = h->n_pop; pa.pop_items = h->pop_items;
        pa.n_blk = h->pop_ld / 32; pa.ld = h->pop_ld;
        pa.dense = h->pop_dense;
        pa.n_first = (h->n_all_rows - a.n_rows) * pa.n_blk;
    }
    if (a.n_rows <= 0 && !(pop && pa.n_rows > 0)) return RS_OK;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    const int64_t items = a.n_rows * (int64_t)h->n_chunks + (pop ? pa.n_rows * pa.n_blk : 0);
    int64_t grid = (int64_t)sms * 4;          // resident CTAs; warps pull work items from the counter
    if (grid > (items + SW - 1) / SW) grid = (items + SW - 1) / SW;
    switch (h->p.sim) {
    case RS_SIM_COSINE: RS_TRY((launch_stream<RS_SIM_COSINE, false>(h, a, pa, (int)grid))); break;
    case RS_SIM_MSD: RS_TRY((launch_stream<RS_SIM_MSD, false>(h, a, pa, (int)grid))); break;
    case RS_SIM_PEARSON: RS_TRY((launch_stream<RS_SIM_PEARSON, false>(h, a, pa, (int)grid))); break;
    case RS_SIM_PEARSON_BASELINE:
        if (h->p.shrinkage > 0.0) RS_TRY((launch_stream<RS_SIM_PEARSON_BASELINE, true>(h, a, pa, (int)grid)));
        else RS_TRY((launch_stream<RS_SIM_PEARSON_BASELINE, false>(h, a, pa, (int)grid)));
        break;
    default: rs_set_error("unknown similarity %d", h->p.sim); return RS_ERR_INVALID;
    }
    h->prof.sim_launches++;
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

int32_t rs_mirror_launch(rs_knn *h) {
    MirrorArgs a{};
    a.self = h->sims;
    for (int q = 0; q < h->cyc_R; q++) a.peer[q] = h->peer_sims[q];
    a.peer[h->cyc_r] = h->sims;
    a.ld = h->ld_s; a.n = h->n_left; a.count = h->cyc_R; a.index = h->cyc_r; a.lower = h->stream_lower ? 1 : 0;
    const int64_t nblk = ((int64_t)h->n_left + RS_CYC_B - 1) / RS_CYC_B;
    const int64_t own = (nblk - h->cyc_r + h->cyc_R - 1) / h->cyc_R;
    if (own <= 0) return RS_OK;
    dim3 grid((unsigned)nblk, (unsigned)own), block(32, 8);
    if (h->n_pop > 0) mirror_pop_kernel<<<grid, block, 0, h->stream>>>(a, h->rank, h->n_pop);
    else mirror_kernel<<<grid, block, 0, h->stream>>>(a);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

int32_t rs_symmetrize_launch(rs_knn *h) {
    if (h->cyc_R > 1) return RS_OK;                          // cyclic shards: rs_knn_mirror after the peers are attached
    if (!(h->row_begin == 0 && h->row_end == h->n_left)) return RS_OK;
    const unsigned t = (unsigned)((h->n_left + 31) / 32);
    dim3 grid(t, t), block(32, 8);
    if (h->n_pop > 0) symmetrize_pop_kernel<<<grid, block, 0, h->stream>>>(h->sims, h->ld_s, h->n_left, h->stream_lower ? 1 : 0, h->rank, h->n_pop);
    else symmetrize_kernel<<<grid, block, 0, h->stream>>>(h->sims, h->ld_s, h->n_left, h->stream_lower ? 1 : 0);
    h->prof.total_launches++;
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}
