// sim_tensor.cu — the co-rated similarity as masked integer contractions on the 5th-gen
// tensor cores (tcgen05.mma.kind::i8, int32 accumulators in TMEM), sm_100a only.
//
// For integer ratings every sum core/sim.go accumulates over the co-rated entries of two left
// rows a, b is a dot product of int8 planes of the left matrix (X = rating, X2 = rating^2,
// M = 1 where rated):
//     count = M_a.M_b   Sx = X_a.M_b   Sy = M_a.X_b   Sxx = X2_a.M_b   Syy = M_a.X2_b   Sxy = X_a.X_b
// The int32 accumulation is exact while no sum leaves int32: with m = the largest |rating| and n2 = the
// second-longest left row (a pair is co-rated over at most its shorter row), 4 m^2 n2 for MSD (its epilogue
// forms Sxx + Syy - 2 Sxy in int32), m^2 n2 for Cosine and Pearson, 2 m n2 for Slope One (Sx - Sy); tensor_eligible
// (api.cu) refuses a Fit beyond them.  Inside them the FP64 epilogue reproduces the reference bit for bit
// for Cosine (core/sim.go:10-25) and MSD (core/sim.go:28-44), whose Go sums are sums of small
// integers.  Pearson from the sums is exact integer arithmetic followed by four roundings (see
// pearson_from_sums): within 4 ulps of the exact value (6 once an integer passes 2^53), but NOT the
// reference's rounding sequence; the
// bit-exact Pearson is the stream path (sim_stream.cu).
//
// Kernel shape (one CTA per SM, persistent over a static tile list):
//   tile      = 128 left rows (MMA M, TMEM lanes) x BN left rows (MMA N) x all K;
//               BN = 128 for Cosine / MSD, 64 for Pearson (six accumulators), see Cfg<>
//   operands  = planes laid out K-blocked, [plane][K / 256][row][256] int8 (see tma_load_box);
//               TMA 4-D boxes (BK bytes of K x rows, one plane per instruction) land one pipeline
//               stage with SWIZZLE_128B (BK = 128, Pearson: 3 stages x 72 KB) or SWIZZLE_64B
//               (BK = 64, Cosine / MSD / Slope One: 4 stages x 48 KB)
//   pipeline  = mbarrier full/empty ring; warp 0 lane 0 issues TMA, warp 1 lane 0 issues
//               tcgen05.mma, warps 2-9 run the epilogue (tcgen05.ld -> FP64 -> HBM)
//   MMAs      = the B planes of a stage are adjacent in shared memory in the order (X2, M, X), so
//               products that share an A plane are ONE instruction with a wider N:
//                 Pearson: M_I x [X2|M|X]_J (N=192), X_I x [M|X]_J (N=128), X2_I x M_J (N=64)
//                 MSD    : M_I x [X2|M]_J (N=256), then X2_I x M_J accumulated INTO the Syy columns
//                          (only Sxx+Syy is needed), X_I x X_J (N=128)
//                 Cosine : M_I x X2_J, X_I x X_J, X2_I x M_J (N=128 each)
//                 Slope  : M_I x [M|X]_J (N=256: count, Sy), X_I x M_J (Sx)   (core/slope_one.go)
//   TMEM      = 384 accumulator columns in every mode
//   large Cosine / MSD / Slope One problems run the CTA-pair variant below (namespace pair:
//   tcgen05 cta_group::2, 256 x 128 tiles, each SM stages its 128 A rows and half of the B rows)
//   schedule  = block-triangular: a tile runs iff it holds a pair (i, j) with j >= i and writes both
//               S[i][j] and S[j][i] (the similarities are bit-symmetric, core/knn.go:205-208); a
//               row-sharded handle runs every bj for its own row blocks and writes S[i][j] only.
//               Tiles are rasterised in 1024 x 1024 supertiles and the CTAs stream K in lockstep
//               (throttle in the TMA producer) so that shared operand rows hit in L2.
#include <cuda.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "common.cuh"

namespace {

constexpr int BM = RS_TC_BM;   // 128 left rows per tile (MMA M, TMEM lanes)
// warp 0 TMA, warp 1 MMA + TMEM alloc, warps 2..9 epilogue.  Eight epilogue warps: a warp can only read the
// TMEM lane quarter (warp % 4), so two warps share each quarter and take half of the tile's columns each —
// with single-buffered accumulators the epilogue is exposed, and on short contractions (K of a few
// thousand) its FP64 divisions and square roots cost more than the MMAs of the tile.
constexpr int NUM_THREADS = 320;
constexpr int EPI_THREADS = 256;
constexpr int TMEM_COLS = 512;

// plane order in global and shared memory
constexpr int PL_X2 = 0, PL_M = 1, PL_X = 2;

// TC_PEARSON128: Pearson with the __int128 epilogue (pearson_from_sums), for rows too long for the int64 one
enum { TC_COSINE = 0, TC_MSD = 1, TC_PEARSON = 2, TC_COSUMS = 3, TC_SLOPE = 4, TC_PEARSON128 = 5 };

// Per-mode tile shape.  Every tcgen05.mma reads its A slab (128 x 32 B) and B slab (N x 32 B) from
// shared memory, so narrow instructions are shared-memory bound: 3 x N=64 (the first Cosine
// kernel) measured 52 % of the MMA rate with the loads switched off, the wide Pearson mix 97 %
// (profiles/r01_tensor_calibration.md).  Cosine and MSD therefore use BN = 128 (instructions of
// N = 128 / 256) with 64-byte K blocks (SWIZZLE_64B) to keep four 48 KB stages in flight;
// Pearson keeps BN = 64 (six accumulators = 384 TMEM columns) with 128-byte K blocks.
template <int MODE> struct Cfg;
template <> struct Cfg<TC_COSINE> {
    static constexpr int BN = 128, BK = 64, STAGES = 4;
    static constexpr int ACC_COLS = 384, ACC_STAGES = 1;
    static constexpr int C_SYY = 0, C_SXY = 128, C_SXX = 256, C_CNT = -1, C_SX = -1, C_SY = -1;
};
template <> struct Cfg<TC_MSD> {
    // C_SYY holds Sxx + Syy: both products accumulate into the same columns (only the sum is needed)
    static constexpr int BN = 128, BK = 64, STAGES = 4;
    static constexpr int ACC_COLS = 384, ACC_STAGES = 1;
    static constexpr int C_SYY = 0, C_CNT = 128, C_SXY = 256, C_SXX = -1, C_SX = -1, C_SY = -1;
};
template <> struct Cfg<TC_PEARSON> {
    static constexpr int BN = 64, BK = 128, STAGES = 3;
    static constexpr int ACC_COLS = 384, ACC_STAGES = 1;
    static constexpr int C_SYY = 0, C_CNT = 64, C_SY = 128, C_SX = 192, C_SXY = 256, C_SXX = 320;
};
template <> struct Cfg<TC_COSUMS> : Cfg<TC_PEARSON> {};
template <> struct Cfg<TC_PEARSON128> : Cfg<TC_PEARSON> {};
template <> struct Cfg<TC_SLOPE> {
    // Slope One deviations (core/slope_one.go:71-90): count, Sy = M_I x [M|X]_J (N = 256), Sx = X_I x M_J
    static constexpr int BN = 128, BK = 64, STAGES = 4;
    static constexpr int ACC_COLS = 384, ACC_STAGES = 1;
    static constexpr int C_CNT = 0, C_SY = 128, C_SX = 256, C_SYY = -1, C_SXY = -1, C_SXX = -1;
};

template <int MODE> struct Geo {
    using C = Cfg<MODE>;
    static constexpr int BN = C::BN, BK = C::BK, STAGES = C::STAGES;
    static constexpr int A_PLANE_BYTES = BM * BK;
    static constexpr int B_PLANE_BYTES = BN * BK;
    static constexpr int A_STAGE_BYTES = 3 * A_PLANE_BYTES;
    static constexpr int B_STAGE_BYTES = 3 * B_PLANE_BYTES;
    static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
    static_assert(SMEM_BYTES <= 227 * 1024, "pipeline does not fit in shared memory");
    static_assert(C::ACC_COLS * C::ACC_STAGES <= TMEM_COLS, "accumulators do not fit in TMEM");
};

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a pipeline bug must trap loudly instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int who) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000ll) {  // ~2 s at 1.9 GHz
            printf("sim_tensor_kernel: mbarrier timeout (role %d, block %d, thread %d)\n", who, blockIdx.x,
                   threadIdx.x);
            __trap();
        }
    }
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// Operand boxes: the planes are stored K-BLOCKED, [plane][K / 256][row][256 bytes of K] (RS_TC_KBLK), so
// the rows of a tile are contiguous 256-byte pieces (one DRAM page / TLB entry serves a tile's rows
// instead of one per row: +30 % on the Netflix shape, whose rows are 480 KB apart otherwise) while a
// row piece still holds the next K blocks of the same row, which the 256-byte L2 promotion of the
// tensor map prefetches.  Tensor map dims {256, rows, K / 256, planes}; a box is BK bytes x rows at
// coordinates {k % 256, row, k / 256, plane}.
__device__ __forceinline__ void tma_load_box(uint32_t dst, const CUtensorMap *map, int row, int k, int plane,
                                             uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], "
        "[%6];" ::"r"(dst),
        "l"(map), "r"(k & (RS_TC_KBLK - 1)), "r"(row), "r"(k / RS_TC_KBLK), "r"(plane), "r"(bar)
        : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, int8 x int8 -> int32
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                        uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrive once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t addr, int32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(addr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major shared-memory matrix descriptor, sm_100 descriptor version 1.  One swizzle atom along K
// (BK = 128 B -> SWIZZLE_128B, BK = 64 B -> SWIZZLE_64B); 8-row groups are 8*BK bytes apart.
template <int BK_>
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
    static_assert(BK_ == 128 || BK_ == 64, "one swizzle atom per K block");
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);            // start address      bits [0,14)
    d |= (uint64_t)0 << 16;                                  // leading byte offset (unused: one atom along K)
    d |= (uint64_t)((8u * BK_) >> 4) << 32;                  // stride byte offset  bits [32,46)
    d |= (uint64_t)1 << 46;                                  // descriptor version  bits [46,48)
    d |= (uint64_t)(BK_ == 128 ? 2 : 4) << 61;               // SWIZZLE_128B / SWIZZLE_64B  bits [61,64)
    return d;
}
// kind::i8 instruction descriptor: D=S32, A=B=signed int8, both K-major, M=128, N=n
__host__ __device__ constexpr uint32_t make_idesc(int n) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

struct TcArgs {
    const int2 *tiles;      // (bi, bj) per tile
    int32_t num_tiles;
    int32_t k_blocks;       // K / 128
    int32_t n_left;
    int64_t row_begin, row_end;
    int mirror;
    double *sims;
    int64_t ld_s;
    const int32_t *row_cnt; // Pearson: ratings per left row, and their integer sum
    const int32_t *row_sum;
    int32_t *cosums;        // TC_COSUMS: raw sums of rows [cos_row0, cos_row0+cos_nrows)
    int64_t cos_row0, cos_nrows;
    // K-lockstep throttle (performance hint only, see the TMA producer): chunks of `sync_chunk` K
    // blocks, a CTA may run at most `sync_slack` chunks ahead of the grid's average progress.
    unsigned long long *progress;
    int sync_chunk, sync_slack, sync_timeout;
    // Fused top-k (pair kernel, RS_STORE_TOPK): no similarity is stored.  Every pair {i, j}, j > i, is tested
    // against the current k-th best of row i and of row j (thr_*; key 0 = list not full, accept) and the
    // survivors are appended to the rows' candidate buffers, merged between waves (topk.cu).
    int topk_mode;
    const unsigned long long *thr_key;
    const int32_t *thr_id;
    int32_t *cand_cnt;
    int32_t *cand_id;
    double *cand_sim;
    int32_t cand_cap;
};

__device__ __forceinline__ unsigned long long ld_relaxed_gpu(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// Pearson from exact integer sums.  With a-row count ca and sum sa (b: cb, sb) and n co-ratings:
//   m  = sum (x-sa/ca)^2 = Mi/ca^2,  Mi = ca^2*Sxx - 2*ca*sa*Sx + n*sa^2          (integers)
//   nn = Ni/cb^2,                    Ni = cb^2*Syy - 2*cb*sb*Sy + n*sb^2
//   l  = L/(ca*cb),                  L  = ca*cb*Sxy - ca*sb*Sx - cb*sa*Sy + n*sa*sb
//   l/(sqrt(m)*sqrt(nn)) = L/(sqrt(Mi)*sqrt(Ni))   — the counts cancel; Mi==0 <=> m==0 exactly,
// so NaN-ness matches the reference's 0/0 (core/sim.go:80) with no cancellation noise.
// Range: Mi = ca^2 * sum (x - sa/ca)^2 over the co-rated x, and every partial term and partial sum of the three
// integers is at most 4 m^2 n1^3 for ratings |x| <= m and rows of at most n1 ratings (ca*ca*sxx, 2*ca*sa*sx up to
// 242 ca^3 for +-11).  Two instantiations (the host picks one per Fit, rs_sim_tensor_launch):
//   I128 = false  int64, exact and free of signed overflow while 4 m^2 n1^3 < 2^63 (rows of up to ~2.67e5 ratings of
//                 +-11, ~4.5e5 of 1..5: every MovieLens shape);
//   I128 = true   __int128 beyond: with the co-rated sums and the row sums inside int32 (tensor_eligible in api.cu)
//                 and rows of fewer than 2^31 ratings every term is below 2^100.
// Rounding: L, Mi and Ni convert exactly below 2^53 and correctly rounded (to nearest) above; then two square roots,
// a product and a quotient, each correctly rounded.  Relative error below 4 * 2^-53 (to first order) while |L|, Mi
// and Ni are below 2^53, i.e. within 4 ulps of the exact L / sqrt(Mi * Ni); past 2^53 the conversion of L adds
// 2^-53 and those of Mi and Ni 2^-53 each, halved by the square root: 6 ulps.  It is not the correctly rounded value,
// and not the reference's rounding sequence.
// (double) of a __int128 is lowered in software without a documented rounding; this one rounds to nearest: below
// 2^63 cvt.rn.f64.s64, above a right shift to 62 bits that ORs the dropped bits into the last one (the sticky bit
// lies below the rounding position, so rounding the shifted value to 53 bits rounds the original), then an exact
// power-of-two scaling.
__device__ __forceinline__ double i128_to_double_rn(__int128 v) {
    const long long lo = (long long)v;
    if ((__int128)lo == v) return (double)lo;
    const unsigned __int128 u = v < 0 ? (unsigned __int128)(-v) : (unsigned __int128)v;   // >= 2^63
    const unsigned long long uh = (unsigned long long)(u >> 64);
    const int bits = uh ? 128 - __clzll((long long)uh) : 64;
    const int shift = bits - 62;
    const unsigned long long w = (unsigned long long)(u >> shift) | ((u & (((unsigned __int128)1 << shift) - 1)) != 0);
    const double d = ldexp((double)(long long)w, shift);
    return v < 0 ? -d : d;
}

template <bool I128>
__device__ __forceinline__ double pearson_from_sums(long long n, long long sx, long long sy, long long sxx,
                                                    long long syy, long long sxy, long long ca, long long sa,
                                                    long long cb, long long sb) {
    if constexpr (!I128) {
        const long long Mi = ca * ca * sxx - 2 * ca * sa * sx + n * sa * sa;
        const long long Ni = cb * cb * syy - 2 * cb * sb * sy + n * sb * sb;
        const long long L = ca * cb * sxy - ca * sb * sx - cb * sa * sy + n * sa * sb;
        return (double)L / (sqrt((double)Mi) * sqrt((double)Ni));
    } else {
        using i128 = __int128;
        const i128 Mi = (i128)ca * ca * sxx - (i128)(2 * ca) * sa * sx + (i128)n * sa * sa;
        const i128 Ni = (i128)cb * cb * syy - (i128)(2 * cb) * sb * sy + (i128)n * sb * sb;
        const i128 L = (i128)ca * cb * sxy - (i128)ca * sb * sx - (i128)cb * sa * sy + (i128)n * sa * sb;
        return i128_to_double_rn(L) / (sqrt(i128_to_double_rn(Mi)) * sqrt(i128_to_double_rn(Ni)));
    }
}

// K-lockstep throttle of the TMA producers.  Tiles that run at the same time share operand rows (supertile
// rasterisation), but a row block is tens of MB long in K, so the sharing only hits in L2 while the CTAs stream
// through K at the same position; left alone they drift apart and the DRAM traffic is 3-4x the ideal
// (profiles/r01_tensor_cos_v2_summary.txt).  Every producer counts the K chunks it has issued in one global
// counter and does not start chunk g before the grid as a whole has issued (g - slack) chunks per CTA.  The wait
// is bounded and carries no data dependence: on a timeout the CTA just proceeds.
// throttle_wait runs before K block kb; g counts the chunks this CTA has started.
__device__ __forceinline__ void throttle_wait(const TcArgs &a, int kb, long long &g) {
    const int chunk = a.sync_chunk;
    if (chunk > 0 && kb % chunk == 0) {
        if (g > 0) atomicAdd(a.progress, 1ull);          // chunk g-1 is issued
        const long long need = (g - a.sync_slack) * (long long)gridDim.x;
        if (need > 0 && (long long)ld_relaxed_gpu(a.progress) < need) {
            const long long t0 = clock64();
            while ((long long)ld_relaxed_gpu(a.progress) < need && clock64() - t0 < a.sync_timeout) {}
        }
        g++;
    }
}
// Done: credit every chunk a CTA with the longest tile list would still issue.  The grid takes one tile per
// cluster of CS CTAs.
template <int CS>
__device__ __forceinline__ void throttle_credit(const TcArgs &a, long long g) {
    if (a.sync_chunk > 0) {
        const int n_units = (int)(gridDim.x / CS);
        const long long cpt = (a.k_blocks + a.sync_chunk - 1) / a.sync_chunk;
        const long long max_chunks = (long long)((a.num_tiles + n_units - 1) / n_units) * cpt;
        atomicAdd(a.progress, (unsigned long long)(max_chunks - g + 1));
    }
}

// A thread's integer sums against 8 consecutive columns, read from the accumulator columns Cfg<MODE> assigns;
// the sums a mode does not accumulate are left unset.
struct Sums8 {
    int32_t syy[8], sxy[8], sxx[8], cnt[8], sx[8], sy[8];
};
template <int MODE>
__device__ __forceinline__ void tmem_ld_sums(uint32_t taddr, Sums8 &v) {
    using C = Cfg<MODE>;
    if constexpr (C::C_SYY >= 0) tmem_ld8(taddr + C::C_SYY, v.syy);
    if constexpr (C::C_SXY >= 0) tmem_ld8(taddr + C::C_SXY, v.sxy);
    if constexpr (C::C_SXX >= 0) tmem_ld8(taddr + C::C_SXX, v.sxx);
    if constexpr (C::C_CNT >= 0) tmem_ld8(taddr + C::C_CNT, v.cnt);
    if constexpr (C::C_SX >= 0) tmem_ld8(taddr + C::C_SX, v.sx);
    if constexpr (C::C_SY >= 0) tmem_ld8(taddr + C::C_SY, v.sy);
    tmem_ld_wait();
}

// S[i][j] from the sums of column c, for Cosine, MSD and Slope One (Pearson: pearson_from_sums)
template <int MODE>
__device__ __forceinline__ double sim_from_sums(const Sums8 &v, int c, int64_t i, int64_t j) {
    if constexpr (MODE == TC_SLOPE) {
        // core/slope_one.go:74-88: for i > j  dev[i][j] = sum(r_i - r_j) / count and
        // dev[j][i] = -dev[i][j]; untouched cells (no co-rating, the diagonal) stay +0
        const int32_t dbig = i > j ? v.sx[c] - v.sy[c] : v.sy[c] - v.sx[c];   // larger index minus smaller
        const double q = (double)dbig / (double)v.cnt[c];
        return (v.cnt[c] == 0 || i == j) ? 0.0 : (i > j ? q : -q);
    } else {
        static_assert(MODE == TC_COSINE || MODE == TC_MSD, "sim_from_sums: Cosine / MSD / Slope One");
        double s;
        if constexpr (MODE == TC_COSINE) {
            // core/sim.go:24  l / (sqrt(m) * sqrt(n)),  m = Sxx, n = Syy, l = Sxy
            s = (double)v.sxy[c] / (sqrt((double)v.sxx[c]) * sqrt((double)v.syy[c]));
        } else {
            // core/sim.go:43  1 / (sum/count + 1),  sum = (Sxx + Syy) - 2 Sxy (exact integer)
            const int32_t sum = v.syy[c] - 2 * v.sxy[c];
            s = 1.0 / ((double)sum / (double)v.cnt[c] + 1.0);
        }
        return j == i ? __longlong_as_double(0x7ff8000000000001ll) : s;   // diagonal stays unset (core/knn.go:202)
    }
}

// Stores a thread's 8 similarities S[i][j0 .. j0+8): 64 contiguous bytes, if the handle holds row i (row_ok).
// With a.mirror it also stores the mirrored S[j][i]: for a fixed j the 32 lanes write 32 consecutive doubles.
template <int MODE>
__device__ __forceinline__ void store8(const TcArgs &a, int64_t i, int64_t j0, bool row_ok, const double (&s)[8],
                                       const Sums8 &v) {
    if (row_ok) {
        double *o = a.sims + (i - a.row_begin) * a.ld_s + j0;
        if (j0 + 8 <= a.n_left) {
#pragma unroll
            for (int c = 0; c < 8; c += 2) *reinterpret_cast<double2 *>(o + c) = make_double2(s[c], s[c + 1]);
        } else {
#pragma unroll
            for (int c = 0; c < 8; c++) if (j0 + c < a.n_left) o[c] = s[c];
        }
    }
    if (a.mirror && i < a.n_left) {
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const int64_t j = j0 + c;
            // Slope One is antisymmetric: dev[j][i] = -dev[i][j], signed zeros included, but cells
            // that were never assigned (no co-rating) stay +0 on both sides
            double sm = s[c];
            if constexpr (MODE == TC_SLOPE) { if (v.cnt[c] != 0 && i != j) sm = -s[c]; }
            if (j < a.n_left) a.sims[j * a.ld_s + i] = sm;
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(NUM_THREADS, 1)
sim_tensor_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, TcArgs a) {
    using C = Cfg<MODE>;
    using G = Geo<MODE>;
    constexpr int BN = G::BN, BK = G::BK, STAGES = G::STAGES;
    constexpr int A_PLANE_BYTES = G::A_PLANE_BYTES, B_PLANE_BYTES = G::B_PLANE_BYTES;
    constexpr int A_STAGE_BYTES = G::A_STAGE_BYTES, STAGE_BYTES = G::STAGE_BYTES;
    const int cta_id = blockIdx.x, n_ctas = gridDim.x;
    extern __shared__ uint8_t smem_raw[];
    // SWIZZLE_128B needs 1024-byte aligned tiles
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = smem_base + STAGES * STAGE_BYTES;
    const uint32_t full_bar = bars;                    // STAGES x 8 B
    const uint32_t empty_bar = bars + 8 * STAGES;      // STAGES x 8 B
    const uint32_t tfull_bar = bars + 16 * STAGES;     // 2 x 8 B   accumulator ready
    const uint32_t tempty_bar = tfull_bar + 16;        // 2 x 8 B   accumulator drained
    const uint32_t tmem_slot = tempty_bar + 16;        // 4 B       TMEM base address
    uint8_t *smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    volatile uint32_t *tmem_slot_ptr = reinterpret_cast<volatile uint32_t *>(smem_gen + STAGES * STAGE_BYTES +
                                                                              16 * STAGES + 32);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&map_a);
        tma_prefetch_desc(&map_b);
        for (int s = 0; s < STAGES; s++) {
            mbar_init(full_bar + 8 * s, 1);
            mbar_init(empty_bar + 8 * s, 1);
        }
        for (int s = 0; s < 2; s++) {
            mbar_init(tfull_bar + 8 * s, 1);
            mbar_init(tempty_bar + 8 * s, EPI_THREADS);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp == 0) {
        // ======================= TMA producer =======================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            long long g = 0;
            for (int t = cta_id; t < a.num_tiles; t += n_ctas) {
                const int2 tile = a.tiles[t];
                const int row_a = tile.x * BM;
                const int row_b = tile.y * BN;
                for (int kb = 0; kb < a.k_blocks; kb++) {
                    throttle_wait(a, kb, g);
                    mbar_wait(empty_bar + 8 * stage, phase ^ 1u, 0);   // the MMAs freed the stage
                    const uint32_t sa = smem_base + stage * STAGE_BYTES;
                    const uint32_t sb = sa + A_STAGE_BYTES;
                    const uint32_t fb = full_bar + 8 * stage;
                    mbar_arrive_expect_tx(fb, STAGE_BYTES);
#pragma unroll
                    for (int p = 0; p < 3; p++) {
                        tma_load_box(sa + p * A_PLANE_BYTES, &map_a, row_a, kb * BK, p, fb);
                        tma_load_box(sb + p * B_PLANE_BYTES, &map_b, row_b, kb * BK, p, fb);
                    }
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
            }
            throttle_credit<1>(a, g);
        }
    } else if (warp == 1) {
        // ======================= MMA issuer =======================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int t = cta_id; t < a.num_tiles; t += n_ctas) {
                mbar_wait(tempty_bar + 8 * acc, acc_phase ^ 1u, 1);   // epilogue drained this buffer
                tc_fence_after();
                const uint32_t d0 = tmem_base + (uint32_t)(acc * C::ACC_COLS);
                for (int kb = 0; kb < a.k_blocks; kb++) {
                    mbar_wait(full_bar + 8 * stage, phase, 2);        // TMA bytes have landed
                    tc_fence_after();
                    const uint32_t sa = smem_base + stage * STAGE_BYTES;
                    const uint32_t sb = sa + A_STAGE_BYTES;
#pragma unroll
                    for (int k = 0; k < BK / 32; k++) {
                        const uint32_t accum = (kb > 0 || k > 0) ? 1u : 0u;
                        const uint32_t ko = (uint32_t)k * 32u;
                        const uint64_t a_x2 = make_desc<BK>(sa + PL_X2 * A_PLANE_BYTES + ko);
                        const uint64_t a_m = make_desc<BK>(sa + PL_M * A_PLANE_BYTES + ko);
                        const uint64_t a_x = make_desc<BK>(sa + PL_X * A_PLANE_BYTES + ko);
                        const uint64_t b_x2 = make_desc<BK>(sb + PL_X2 * B_PLANE_BYTES + ko);
                        const uint64_t b_m = make_desc<BK>(sb + PL_M * B_PLANE_BYTES + ko);
                        const uint64_t b_x = make_desc<BK>(sb + PL_X * B_PLANE_BYTES + ko);
                        if constexpr (MODE == TC_COSINE) {
                            umma_i8(d0 + C::C_SYY, a_m, b_x2, make_idesc(BN), accum);
                            umma_i8(d0 + C::C_SXY, a_x, b_x, make_idesc(BN), accum);
                            umma_i8(d0 + C::C_SXX, a_x2, b_m, make_idesc(BN), accum);
                        } else if constexpr (MODE == TC_SLOPE) {
                            umma_i8(d0 + C::C_CNT, a_m, b_m, make_idesc(2 * BN), accum);    // [count | Sy]
                            umma_i8(d0 + C::C_SX, a_x, b_m, make_idesc(BN), accum);         // Sx
                        } else if constexpr (MODE == TC_MSD) {
                            umma_i8(d0 + C::C_SYY, a_m, b_x2, make_idesc(2 * BN), accum);   // [Syy | count]
                            umma_i8(d0 + C::C_SYY, a_x2, b_m, make_idesc(BN), 1u);          // Syy += Sxx
                            umma_i8(d0 + C::C_SXY, a_x, b_x, make_idesc(BN), accum);
                        } else {
                            umma_i8(d0 + C::C_SYY, a_m, b_x2, make_idesc(3 * BN), accum);   // [Syy | count | Sy]
                            umma_i8(d0 + C::C_SX, a_x, b_m, make_idesc(2 * BN), accum);     // [Sx | Sxy]
                            umma_i8(d0 + C::C_SXX, a_x2, b_m, make_idesc(BN), accum);
                        }
                    }
                    umma_commit(empty_bar + 8 * stage);               // frees the smem stage once the MMAs are done
                    if (kb == a.k_blocks - 1) umma_commit(tfull_bar + 8 * acc);
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
                if (++acc == C::ACC_STAGES) { acc = 0; acc_phase ^= 1u; }
            }
        }
    } else {
        // ======================= epilogue (8 warps: TMEM lane quarter = warp % 4, column half = (warp-2)/4) =======================
        const int q = warp & 3;
        const int chalf = (warp - 2) >> 2;          // which half of the tile's columns this warp converts
        const int r_in_tile = q * 32 + lane;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int t = cta_id; t < a.num_tiles; t += n_ctas) {
            const int2 tile = a.tiles[t];
            const int64_t i = (int64_t)tile.x * BM + r_in_tile;
            const int64_t j0 = (int64_t)tile.y * BN;
            mbar_wait(tfull_bar + 8 * acc, acc_phase, 3);
            tc_fence_after();
            const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * C::ACC_COLS);
            long long ca = 0, sa = 0;
            if ((MODE == TC_PEARSON || MODE == TC_PEARSON128) && i < a.n_left) { ca = a.row_cnt[i]; sa = a.row_sum[i]; }
            const bool row_ok = (i < a.n_left) && (i >= a.row_begin) && (i < a.row_end);
#pragma unroll 1
            for (int c0 = chalf * (BN / 2); c0 < (chalf + 1) * (BN / 2); c0 += 8) {
                Sums8 v;
                tmem_ld_sums<MODE>(tbase + c0, v);
                if constexpr (MODE == TC_COSUMS) {
                    const int64_t r = i - a.cos_row0;
                    if (i < a.n_left && r >= 0 && r < a.cos_nrows) {
#pragma unroll
                        for (int c = 0; c < 8; c++) {
                            const int64_t j = j0 + c0 + c;
                            if (j < a.n_left) {
                                int32_t *o = a.cosums + (r * a.n_left + j) * 6;
                                o[0] = v.cnt[c]; o[1] = v.sx[c]; o[2] = v.sy[c];
                                o[3] = v.sxx[c]; o[4] = v.syy[c]; o[5] = v.sxy[c];
                            }
                        }
                    }
                } else {
                    double s[8];
#pragma unroll
                    for (int c = 0; c < 8; c++) {
                        const int64_t j = j0 + c0 + c;
                        if constexpr (MODE == TC_PEARSON || MODE == TC_PEARSON128) {
                            long long cb = 0, sb = 0;
                            if (j < a.n_left) { cb = a.row_cnt[j]; sb = a.row_sum[j]; }
                            s[c] = pearson_from_sums<MODE == TC_PEARSON128>(v.cnt[c], v.sx[c], v.sy[c], v.sxx[c],
                                                                            v.syy[c], v.sxy[c], ca, sa, cb, sb);
                            if (j == i) s[c] = __longlong_as_double(0x7ff8000000000001ll);   // diagonal stays unset
                        } else {
                            s[c] = sim_from_sums<MODE>(v, c, i, j);
                        }
                    }
                    store8<MODE>(a, i, j0 + c0, row_ok, s, v);
                }
            }
            tc_fence_before();
            mbar_arrive(tempty_bar + 8 * acc);     // 256 arrivals release the accumulator buffer
            if (++acc == C::ACC_STAGES) { acc = 0; acc_phase ^= 1u; }
        }
    }

    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) {
        __syncwarp();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// =================================================================================================
// CTA-pair variant (tcgen05 cta_group::2) for Cosine / MSD.
//
// The single-CTA kernel above is bound by operand delivery for Cosine / MSD: a 128 x 128 tile needs
// 128 A rows + 128 B rows (x 3 planes) per K block.  Here the two CTAs of a cluster (two SMs of one
// TPC) compute ONE 256 x 128 tile with M = 256 instructions issued by the even CTA: each SM stages
// its own 128 A rows and only HALF of the B rows (64) — the tensor cores read the other half from
// the peer's shared memory — i.e. 192 instead of 256 operand rows per 128 x 128 outputs and half
// the B shared-memory reads per SM.  Stages are 36 KB, six of them in flight.
//   barriers  full[s]  : lives in the even CTA; both CTAs' TMA loads complete_tx on it, the even
//                        CTA's producer posts the expected bytes of both
//             empty[s] : one per CTA; tcgen05.commit.cta_group::2 multicast to both
//             tfull    : one per CTA (commit multicast) -> each CTA's epilogue reads ITS 128 TMEM lanes
//             tempty   : even CTA only, 512 arrivals (both epilogues; the odd one arrives remotely)
// Accumulator columns are those of Cfg<MODE>: Cosine [Syy | Sxy | Sxx], MSD [Syy+Sxx | count | Sxy], Slope One
// [count | Sy | Sx] (N = 128 each; the wide N = 256 combination of the single-CTA kernel is not available because
// the pair splits B by rows).
namespace pair {

constexpr int P_BN = 128, P_BK = 64, P_STAGES = 6;
constexpr int P_A_PLANE = BM * P_BK;              // 8 KB  (128 rows of this CTA)
constexpr int P_B_PLANE = (P_BN / 2) * P_BK;      // 4 KB  (this CTA's 64 of the 128 B rows)
constexpr int P_A_STAGE = 3 * P_A_PLANE, P_B_STAGE = 3 * P_B_PLANE;
constexpr int P_STAGE = P_A_STAGE + P_B_STAGE;    // 36 KB
constexpr int P_THR_BYTES = 2 * P_BN * 12;          // double-buffered (key, id) thresholds of a tile's columns
constexpr int P_SMEM = P_STAGES * P_STAGE + 1024 + 256 + P_THR_BYTES;
static_assert(P_SMEM <= 227 * 1024, "pair pipeline does not fit in shared memory");
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;       // shared::cluster address of the same offset in the even CTA

__device__ __forceinline__ void tma_load_box_2sm(uint32_t dst, const CUtensorMap *map, int row, int k, int plane,
                                                 uint32_t leader_bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, "
        "%4, %5}], [%6];" ::"r"(dst),
        "l"(map), "r"(k & (RS_TC_KBLK - 1)), "r"(row), "r"(k / RS_TC_KBLK), "r"(plane), "r"(leader_bar)
        : "memory");
}
__device__ __forceinline__ void umma_i8_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {   // arrives on `bar` in BOTH CTAs
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
        "h"((uint16_t)3)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// kind::i8 instruction descriptor for the pair: D=S32, A=B=signed int8, K-major, M=256, N=n
__host__ __device__ constexpr uint32_t make_idesc_2sm(int n) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
}

template <int MODE>
__global__ void __launch_bounds__(NUM_THREADS, 1)
sim_tensor_pair_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, TcArgs a) {
    static_assert(MODE == TC_COSINE || MODE == TC_MSD || MODE == TC_SLOPE, "pair kernel: Cosine / MSD / Slope One");
    using C = Cfg<MODE>;
    const int rank = (int)cluster_ctarank();         // 0 = even CTA = MMA issuer
    const int pair_id = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = smem_base + P_STAGES * P_STAGE;
    const uint32_t full_bar = bars;                      // P_STAGES x 8 B (used in the even CTA)
    const uint32_t empty_bar = bars + 8 * P_STAGES;      // P_STAGES x 8 B
    const uint32_t tfull_bar = bars + 16 * P_STAGES;     // 8 B
    const uint32_t tempty_bar = tfull_bar + 8;           // 8 B (used in the even CTA)
    const uint32_t tmem_slot = tempty_bar + 8;
    uint8_t *smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    volatile uint32_t *tmem_slot_ptr =
        reinterpret_cast<volatile uint32_t *>(smem_gen + P_STAGES * P_STAGE + 16 * P_STAGES + 16);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&map_a);
        tma_prefetch_desc(&map_b);
        for (int s = 0; s < P_STAGES; s++) {
            mbar_init(full_bar + 8 * s, 1);
            mbar_init(empty_bar + 8 * s, 1);
        }
        mbar_init(tfull_bar, 1);
        mbar_init(tempty_bar, 2 * EPI_THREADS);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc_2sm(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();   // both CTAs' barriers and TMEM exist before anyone signals or issues
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp == 0) {
        // ======================= TMA producer (both CTAs) =======================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            long long g = 0;
            for (int t = pair_id; t < a.num_tiles; t += n_pairs) {
                const int2 tile = a.tiles[t];
                const int row_a = (tile.x * 2 + rank) * BM;                  // my 128 of the tile's 256 A rows
                const int row_b = tile.y * P_BN + rank * (P_BN / 2);          // my 64 of the tile's 128 B rows
                for (int kb = 0; kb < a.k_blocks; kb++) {
                    throttle_wait(a, kb, g);
                    mbar_wait(empty_bar + 8 * stage, phase ^ 1u, 0);
                    const uint32_t sa = smem_base + stage * P_STAGE;
                    const uint32_t sb = sa + P_A_STAGE;
                    const uint32_t fb = (full_bar + 8 * stage) & PEER_MASK;    // the even CTA's barrier
                    if (rank == 0) mbar_arrive_expect_tx(full_bar + 8 * stage, 2 * P_STAGE);
#pragma unroll
                    for (int p = 0; p < 3; p++) {
                        tma_load_box_2sm(sa + p * P_A_PLANE, &map_a, row_a, kb * P_BK, p, fb);
                        tma_load_box_2sm(sb + p * P_B_PLANE, &map_b, row_b, kb * P_BK, p, fb);
                    }
                    if (++stage == P_STAGES) { stage = 0; phase ^= 1u; }
                }
            }
            throttle_credit<2>(a, g);
        }
    } else if (warp == 1) {
        // ======================= MMA issuer (even CTA only) =======================
        if (lane == 0 && rank == 0) {
            int stage = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (int t = pair_id; t < a.num_tiles; t += n_pairs) {
                mbar_wait(tempty_bar, acc_phase ^ 1u, 1);            // both epilogues drained the accumulators
                tc_fence_after();
                const uint32_t d0 = tmem_base;
                for (int kb = 0; kb < a.k_blocks; kb++) {
                    mbar_wait(full_bar + 8 * stage, phase, 2);       // both CTAs' bytes have landed
                    tc_fence_after();
                    const uint32_t sa = smem_base + stage * P_STAGE;
                    const uint32_t sb = sa + P_A_STAGE;
#pragma unroll
                    for (int k = 0; k < P_BK / 32; k++) {
                        const uint32_t accum = (kb > 0 || k > 0) ? 1u : 0u;
                        const uint32_t ko = (uint32_t)k * 32u;
                        const uint64_t a_x2 = make_desc<P_BK>(sa + PL_X2 * P_A_PLANE + ko);
                        const uint64_t a_m = make_desc<P_BK>(sa + PL_M * P_A_PLANE + ko);
                        const uint64_t a_x = make_desc<P_BK>(sa + PL_X * P_A_PLANE + ko);
                        const uint64_t b_x2 = make_desc<P_BK>(sb + PL_X2 * P_B_PLANE + ko);
                        const uint64_t b_m = make_desc<P_BK>(sb + PL_M * P_B_PLANE + ko);
                        const uint64_t b_x = make_desc<P_BK>(sb + PL_X * P_B_PLANE + ko);
                        if constexpr (MODE == TC_SLOPE) {
                            umma_i8_2sm(d0 + C::C_CNT, a_m, b_m, make_idesc_2sm(P_BN), accum);
                            umma_i8_2sm(d0 + C::C_SY, a_m, b_x, make_idesc_2sm(P_BN), accum);
                            umma_i8_2sm(d0 + C::C_SX, a_x, b_m, make_idesc_2sm(P_BN), accum);
                        } else if constexpr (MODE == TC_COSINE) {
                            umma_i8_2sm(d0 + C::C_SYY, a_m, b_x2, make_idesc_2sm(P_BN), accum);
                            umma_i8_2sm(d0 + C::C_SXY, a_x, b_x, make_idesc_2sm(P_BN), accum);
                            umma_i8_2sm(d0 + C::C_SXX, a_x2, b_m, make_idesc_2sm(P_BN), accum);
                        } else {
                            umma_i8_2sm(d0 + C::C_SYY, a_m, b_x2, make_idesc_2sm(P_BN), accum);
                            umma_i8_2sm(d0 + C::C_SYY, a_x2, b_m, make_idesc_2sm(P_BN), 1u);   // Syy += Sxx
                            umma_i8_2sm(d0 + C::C_CNT, a_m, b_m, make_idesc_2sm(P_BN), accum);
                            umma_i8_2sm(d0 + C::C_SXY, a_x, b_x, make_idesc_2sm(P_BN), accum);
                        }
                    }
                    umma_commit_2sm(empty_bar + 8 * stage);          // frees the stage in both CTAs
                    if (kb == a.k_blocks - 1) umma_commit_2sm(tfull_bar);
                    if (++stage == P_STAGES) { stage = 0; phase ^= 1u; }
                }
                acc_phase ^= 1u;
            }
        }
    } else {
        // ======================= epilogue (both CTAs: own 128 TMEM lanes) =======================
        const int q = warp & 3;
        const int chalf = (warp - 2) >> 2;          // which half of the tile's columns this warp converts
        const int r_in_tile = q * 32 + lane;
        uint32_t acc_phase = 0;
        const uint32_t tempty_leader = tempty_bar & PEER_MASK;
        unsigned long long *s_thrk = reinterpret_cast<unsigned long long *>(smem_gen + P_STAGES * P_STAGE + 256);
        uint32_t *s_thri = reinterpret_cast<uint32_t *>(s_thrk + 2 * P_BN);
        int tbuf = 0;
        for (int t = pair_id; t < a.num_tiles; t += n_pairs) {
            const int2 tile = a.tiles[t];
            const int64_t i = ((int64_t)tile.x * 2 + rank) * BM + r_in_tile;
            const int64_t j0 = (int64_t)tile.y * P_BN;
            unsigned long long trk_i = ~0ull;
            uint32_t tri_i = 0u;
            if (a.topk_mode) {
                // thresholds of the tile's 128 columns -> shared memory (while the MMAs of the tile run), of
                // this thread's row -> registers.  Stale values only admit extra candidates.
                const int e = (int)threadIdx.x - 64;
                if (e < P_BN) {
                    const int64_t jc = j0 + e;
                    s_thrk[tbuf * P_BN + e] = jc < a.n_left ? a.thr_key[jc] : ~0ull;
                    s_thri[tbuf * P_BN + e] = jc < a.n_left ? (uint32_t)a.thr_id[jc] : 0u;
                }
                if (i < a.n_left) { trk_i = a.thr_key[i]; tri_i = (uint32_t)a.thr_id[i]; }
                asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
            }
            mbar_wait(tfull_bar, acc_phase, 3);
            tc_fence_after();
            const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16);
            const bool row_ok = (i < a.n_left) && (i >= a.row_begin) && (i < a.row_end);
#pragma unroll 1
            for (int c0 = chalf * (P_BN / 2); c0 < (chalf + 1) * (P_BN / 2); c0 += 8) {
                Sums8 v;
                tmem_ld_sums<MODE>(tbase + c0, v);
                double s[8];
#pragma unroll
                for (int c = 0; c < 8; c++) s[c] = sim_from_sums<MODE>(v, c, i, j0 + c0 + c);
                if (a.topk_mode) {
                    // selection fused into the epilogue: one compare against each of the two rows' thresholds,
                    // the rare survivor is appended to that row's candidate buffer
#pragma unroll
                    for (int c = 0; c < 8; c++) {
                        const int64_t j = j0 + c0 + c;
                        const double sv = s[c];
                        if (i < a.n_left && j < a.n_left && j > i && sv == sv) {
                            const unsigned long long key = rs_sim_key(sv);
                            if (key > trk_i || (key == trk_i && (uint32_t)j < tri_i)) {
                                const int slot = atomicAdd(a.cand_cnt + i, 1);
                                if (slot < a.cand_cap) {
                                    a.cand_id[i * a.cand_cap + slot] = (int32_t)j;
                                    a.cand_sim[i * a.cand_cap + slot] = sv;
                                }
                            }
                            const unsigned long long tk = s_thrk[tbuf * P_BN + c0 + c];
                            if (key > tk || (key == tk && (uint32_t)i < s_thri[tbuf * P_BN + c0 + c])) {
                                const int slot = atomicAdd(a.cand_cnt + j, 1);
                                if (slot < a.cand_cap) {
                                    a.cand_id[j * a.cand_cap + slot] = (int32_t)i;
                                    a.cand_sim[j * a.cand_cap + slot] = sv;
                                }
                            }
                        }
                    }
                    continue;
                }
                store8<MODE>(a, i, j0 + c0, row_ok, s, v);
            }
            tc_fence_before();
            mbar_arrive_cluster(tempty_leader);    // 2 x 256 arrivals release the accumulators of the pair
            acc_phase ^= 1u;
            tbuf ^= 1;
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();   // no CTA leaves while its peer may still read its shared memory / signal it
    tc_fence_after();
    if (warp == 1) {
        __syncwarp();
        tmem_dealloc_2sm(tmem_base, TMEM_COLS);
    }
}

}  // namespace pair

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int32_t get_encode_fn(EncodeTiledFn *out) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        RS_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !p) {
            rs_set_error("cuTensorMapEncodeTiled is not available from the driver");
            return RS_ERR_CUDA;
        }
        fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    *out = fn;
    return RS_OK;
}

int32_t make_map(const rs_knn *h, int box_k, int box_rows, CUtensorMap *map) {
    EncodeTiledFn enc;
    RS_TRY(get_encode_fn(&enc));
    // [plane][K / 256][row][256 bytes of K]
    const cuuint64_t dims[4] = {(cuuint64_t)RS_TC_KBLK, (cuuint64_t)h->tc_npad, (cuuint64_t)(h->tc_kpad / RS_TC_KBLK), 3};
    const cuuint64_t strides[3] = {(cuuint64_t)RS_TC_KBLK, (cuuint64_t)h->tc_npad * (cuuint64_t)RS_TC_KBLK,
                                   (cuuint64_t)h->tc_kpad * (cuuint64_t)h->tc_npad};
    const cuuint32_t box[4] = {(cuuint32_t)box_k, (cuuint32_t)box_rows, 1, 1};   // one plane, one K block per instruction
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, h->planes, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, box_k == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        rs_set_error("cuTensorMapEncodeTiled failed with CUresult %d (npad=%lld kpad=%lld)", (int)r,
                     (long long)h->tc_npad, (long long)h->tc_kpad);
        return RS_ERR_CUDA;
    }
    return RS_OK;
}

typedef void (*TcKernel)(CUtensorMap, CUtensorMap, TcArgs);

// Launches one persistent wave of `kern` (`smem` bytes of dynamic shared memory) in clusters of `cs` CTAs: 1, or 2
// for the CTA pair.  Each CTA loads operand boxes of bk bytes of K by a_rows rows of A and b_rows rows of B.
int32_t launch_tc(rs_knn *h, TcKernel kern, int smem, int cs, int bk, int a_rows, int b_rows, TcArgs a) {
    a.k_blocks = (int32_t)(h->tc_kpad / bk);
    // K-lockstep throttle: only worth it when a row block does not fit in L2 many times over
    a.progress = reinterpret_cast<unsigned long long *>(h->d_flags + 4);
    a.sync_chunk = (a.k_blocks >= 256 && a.num_tiles > 148) ? 32 : 0;
    a.sync_slack = 1;
    a.sync_timeout = 40000;   // clocks (~20 us): a hint, never a dependence
    if (a.sync_chunk > 0) RS_CUDA(cudaMemsetAsync(a.progress, 0, 8, h->stream));
    CUtensorMap ma, mb;
    RS_TRY(make_map(h, bk, a_rows, &ma));
    RS_TRY(make_map(h, bk, b_rows, &mb));
    RS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = h->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cs;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n_clusters = sms / cs;
    if (cs > 1) {
        cfg.gridDim = dim3((unsigned)(n_clusters * cs));
        int max_clusters = 0;
        RS_CUDA(cudaOccupancyMaxActiveClusters(&max_clusters, kern, &cfg));
        if (max_clusters < 1) {
            rs_set_error("a CTA pair of the tensor kernel does not fit on this device");
            return RS_ERR_CUDA;
        }
        if (n_clusters > max_clusters) n_clusters = max_clusters;   // persistent: one resident wave
    }
    if (n_clusters > a.num_tiles) n_clusters = a.num_tiles;
    cfg.gridDim = dim3((unsigned)(n_clusters * cs));
    RS_CUDA(cudaLaunchKernelEx(&cfg, kern, ma, mb, a));
    RS_CUDA(cudaGetLastError());
    return RS_OK;
}

template <int MODE>
int32_t launch_single(rs_knn *h, const TcArgs &a) {
    using G = Geo<MODE>;
    return launch_tc(h, sim_tensor_kernel<MODE>, G::SMEM_BYTES, 1, G::BK, BM, G::BN, a);
}

template <int MODE>
int32_t launch_pair(rs_knn *h, const TcArgs &a) {
    return launch_tc(h, pair::sim_tensor_pair_kernel<MODE>, pair::P_SMEM, 2, pair::P_BK, BM, pair::P_BN / 2, a);
}

// Copies a tile list into the grow-only device buffer *buf of *cap bytes.  Returns once the copy is done:
// `tiles` is a pageable temporary.
int32_t upload_tiles(rs_knn *h, const std::vector<int2> &tiles, void **buf, size_t *cap) {
    const size_t bytes = tiles.size() * sizeof(int2);
    if (bytes > *cap) {
        RS_CUDA(cudaStreamSynchronize(h->stream));
        if (*buf) cudaFree(*buf);
        *buf = nullptr;
        *cap = 0;
        RS_CUDA(cudaMalloc(buf, bytes + 256));
        *cap = bytes + 256;
    }
    if (bytes) {
        RS_CUDA(cudaMemcpyAsync(*buf, tiles.data(), bytes, cudaMemcpyHostToDevice, h->stream));
        RS_CUDA(cudaStreamSynchronize(h->stream));
    }
    return RS_OK;
}

// Pearson: the int64 epilogue is exact and free of signed overflow while every term of pearson_from_sums, at most
// 4 m^2 n1^3 (m = the largest |rating|, n1 = the longest left row), is below 2^63; past that the __int128 one runs.
// RS_KNN_PEARSON_I128=1 forces the __int128 epilogue (tests: both are exact integers, so both give the same bits).
bool pearson_i128(const rs_knn *h) {
    if (const char *e = getenv("RS_KNN_PEARSON_I128")) if (atoi(e) != 0) return true;
    const unsigned __int128 m = (unsigned __int128)h->int_abs_max, n1 = (unsigned __int128)h->row_len1;
    return 4 * m * m * n1 * n1 * n1 >= ((unsigned __int128)1 << 63);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// Fused top-k (RS_STORE_TOPK on the tensor path, large problems): the pair kernel tests every similarity
// against thresholds that are refreshed only BETWEEN launches, so the block-triangular tile set is cut into
// waves that keep the number of survivors per row small:
//   wave 0      the tiles within 512 columns of the diagonal: every row meets ~1.5 k columns, all of them
//               candidates (there is no threshold yet) — the bootstrap sample;
//   waves 1..W  all other tiles, grouped in supertiles of 4 x 8 cluster tiles (1024 x 1024 similarities, the
//               unit of L2 sharing) taken in a PSEUDO-RANDOM order, wave w ending at the fraction 2^(w-W) of
//               them: a wave brings a row about as many new columns as it has seen before, in an order that
//               is independent of the ids — of which ~k beat the row's current k-th best.
// The order matters because ties are broken by id: user-based MSD is 1.0 for thousands of pairs per row (one
// co-rated item, equal ratings), and a schedule that feeds a row ids in DESCENDING order (plain bands by distance
// did, for the columns left of the diagonal) makes every one of those ties a survivor.
// The N x N matrix, or any slab of it, never exists.  The supertiles of each wave are dealt round-robin to the
// shards of a multi-GPU Fit (equal cost per tile).
static int32_t band_waves(int64_t n_left) {
    // two extra small waves at the start: the thresholds of the bootstrap band are weak for rows with thousands
    // of tied similarities, and a re-run of a small wave is cheap but not free (13 ms each on config 4)
    int w = 0;
    for (int64_t seen = 1536; seen < n_left; seen *= 2) w++;
    return w < 1 ? 1 : w + 2;
}
int32_t rs_tensor_band_count(const rs_knn *h) { return 1 + band_waves(h->n_left); }

static inline uint64_t mix64(uint64_t x) {     // splitmix64 finaliser
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

int32_t rs_sim_tensor_band_launch(rs_knn *h, int32_t wave) {
    if (!h->planes) {
        rs_set_error("tensor path: int8 planes were not built");
        return RS_ERR_INVALID;
    }
    const int mode = h->p.sim == RS_SIM_COSINE ? TC_COSINE : TC_MSD;
    const int n_waves = rs_tensor_band_count(h);
    const int shard_count = h->p.shard_count > 1 ? h->p.shard_count : 1, shard_index = h->p.shard_count > 1 ? h->p.shard_index : 0;
    const int64_t key[4] = {h->n_left, shard_count, shard_index, n_waves};
    if (memcmp(key, h->band_key, sizeof(key)) != 0) {
        // cluster tiles: cbi = 256 rows, cbj = 128 columns; needed iff the tile holds a pair with j > i
        const int ncbi = (int)((h->n_left + 2 * BM - 1) / (2 * BM)), ncbj = (int)((h->n_left + pair::P_BN - 1) / pair::P_BN);
        const int W = n_waves - 1;
        std::vector<std::vector<int2>> bands(n_waves);
        constexpr int SI = 4, SJ = 8;
        auto tile_dist = [&](int cbi, int cbj) { return (int64_t)cbj * pair::P_BN - (int64_t)cbi * 2 * BM; };
        struct Sup { uint64_t h; int sbi, sbj; };
        std::vector<Sup> sups;
        int64_t dealt0 = 0;
        for (int sbi = 0; sbi < ncbi; sbi += SI)
            for (int sbj = 0; sbj < ncbj; sbj += SJ) {
                bool any0 = false, any1 = false;
                for (int cbi = sbi; cbi < sbi + SI && cbi < ncbi; cbi++)
                    for (int cbj = sbj; cbj < sbj + SJ && cbj < ncbj; cbj++) {
                        const int64_t d = tile_dist(cbi, cbj);
                        if (d + pair::P_BN <= 0) continue;                                     // every column <= every row
                        if (d < 512) any0 = true; else any1 = true;
                    }
                if (any0) {     // wave 0: the diagonal band, whole supertile shares dealt to one shard
                    const bool mine = dealt0++ % shard_count == shard_index;
                    for (int cbi = sbi; cbi < sbi + SI && cbi < ncbi; cbi++)
                        for (int cbj = sbj; cbj < sbj + SJ && cbj < ncbj; cbj++) {
                            const int64_t d = tile_dist(cbi, cbj);
                            if (d + pair::P_BN > 0 && d < 512 && mine) bands[0].push_back(make_int2(cbi, cbj));
                        }
                }
                if (any1) sups.push_back({mix64(((uint64_t)sbi << 32) | (uint64_t)sbj), sbi, sbj});
            }
        std::sort(sups.begin(), sups.end(), [](const Sup &x, const Sup &y) { return x.h < y.h; });
        for (size_t q = 0; q < sups.size(); q++) {
            // wave w (1..W) ends at the fraction 2^(w-W) of the shuffled supertiles
            int w = 1;
            while (w < W && (double)(q + 1) > (double)sups.size() * std::ldexp(1.0, w - W)) w++;
            if ((int64_t)q % shard_count != shard_index) continue;
            for (int cbi = sups[q].sbi; cbi < sups[q].sbi + SI && cbi < ncbi; cbi++)
                for (int cbj = sups[q].sbj; cbj < sups[q].sbj + SJ && cbj < ncbj; cbj++) {
                    const int64_t d = tile_dist(cbi, cbj);
                    if (d >= 512) bands[w].push_back(make_int2(cbi, cbj));
                }
        }
        std::vector<int2> flat;
        h->band_off.assign(n_waves + 1, 0);
        for (int w = 0; w < n_waves; w++) {
            h->band_off[w] = (int64_t)flat.size();
            flat.insert(flat.end(), bands[w].begin(), bands[w].end());
        }
        h->band_off[n_waves] = (int64_t)flat.size();
        RS_TRY(upload_tiles(h, flat, &h->band_buf, &h->band_buf_bytes));
        memcpy(h->band_key, key, sizeof(key));
    }
    const int64_t t0 = h->band_off[wave], t1 = h->band_off[wave + 1];
    if (t1 <= t0) return RS_OK;
    TcArgs a{};
    a.tiles = reinterpret_cast<const int2 *>(h->band_buf) + t0;
    a.num_tiles = (int32_t)(t1 - t0);
    a.n_left = h->n_left;
    a.row_begin = 0;
    a.row_end = h->n_left;
    a.mirror = 0;
    a.sims = nullptr;
    a.ld_s = 0;
    a.topk_mode = 1;
    a.thr_key = h->thr_key;
    a.thr_id = h->thr_id;
    a.cand_cnt = h->cand_cnt;
    a.cand_id = h->cand_id;
    a.cand_sim = h->cand_sim;
    a.cand_cap = h->cand_cap;
    RS_TRY(mode == TC_COSINE ? launch_pair<TC_COSINE>(h, a) : launch_pair<TC_MSD>(h, a));
    h->prof.sim_launches++;
    h->prof.total_launches++;
    return RS_OK;
}

// Is the fused top-k path available for this Fit?  (Cosine / MSD on integer ratings, large enough for the
// pair kernel; everything else reduces bounded slabs of similarity rows, see topk.cu.)
bool rs_tensor_topk_fused(const rs_knn *h) {
    if (h->p.sim != RS_SIM_COSINE && h->p.sim != RS_SIM_MSD) return false;
    if (const char *e = getenv("RS_KNN_TOPK_FUSED")) return atoi(e) != 0;
    const int64_t plain_tiles = (((int64_t)h->n_left + BM - 1) / BM) * (((int64_t)h->n_left + pair::P_BN - 1) / pair::P_BN) / 2;
    return plain_tiles >= 4 * 148;
}

int32_t rs_sim_tensor_launch(rs_knn *h, int32_t *d_cosums, int64_t cos_row0, int64_t cos_nrows) {
    if (!h->planes) {
        rs_set_error("tensor path: int8 planes were not built");
        return RS_ERR_INVALID;
    }
    const bool cosums = d_cosums != nullptr;
    const int64_t rb = cosums ? cos_row0 : h->row_begin;
    const int64_t re = cosums ? cos_row0 + cos_nrows : h->row_end;
    if (re <= rb) return RS_OK;
    const bool mirror = !cosums && rb == 0 && re == h->n_left;
    const int mode = cosums ? TC_COSUMS
                            : h->p.sim == RS_SIM_COSINE ? TC_COSINE
                            : h->p.sim == RS_SIM_MSD ? TC_MSD
                            : h->p.sim == RS_SIM_SLOPE_ONE ? TC_SLOPE
                            : h->p.sim == RS_SIM_PEARSON ? TC_PEARSON : -1;
    if (mode < 0) {
        rs_set_error("tensor path supports Cosine, MSD and Pearson (sums mode) only");
        return RS_ERR_UNSUPPORTED;
    }
    const bool wide = mode == TC_COSINE || mode == TC_MSD || mode == TC_SLOPE;       // 128 x 128 tiles, 64-byte K blocks
    const int BN = wide ? Cfg<TC_COSINE>::BN : Cfg<TC_PEARSON>::BN;
    static_assert(Cfg<TC_COSINE>::BN == Cfg<TC_MSD>::BN && Cfg<TC_COSINE>::BN == Cfg<TC_SLOPE>::BN, "host tile geometry");
    const int64_t plain_tiles = ((re - rb + BM - 1) / BM) * ((h->n_left + BN - 1) / BN) / (mirror ? 2 : 1);
    // Which kernel: Cosine / MSD / Slope One problems of at least four tiles per SM run the cta_group::2 pair kernel
    // (256 x 128 tiles; measured on the ML-20M item shape in profiles/r01_tensor_calibration.md), everything else the
    // single-CTA kernel, so that small problems give every SM a tile.  RS_KNN_TC_PAIR=0|1 overrides.
    bool use_pair = wide && plain_tiles >= 4 * 148;
    if (const char *e = getenv("RS_KNN_TC_PAIR")) use_pair = wide && atoi(e) != 0;
    const int ci = use_pair ? 2 : 1;   // row blocks per tile: the pair kernel's tiles are 256 x 128
    const int nbj = (int)((h->n_left + BN - 1) / BN);
    const int bi0 = (int)(rb / BM), bi1 = (int)((re + BM - 1) / BM);
    const int64_t key[5] = {h->n_left, rb, re, (mirror ? 1 : 0) + (use_pair ? 2 : 0) + 4 * (int64_t)BN,
                            cosums ? 0 : h->col_begin};
    if (memcmp(key, h->tile_key, sizeof(key)) != 0) {
        // Rasterised in supertiles of 1024 x 1024 similarities so concurrently running CTAs touch few
        // distinct row blocks.
        const int SUP_I = 8 / ci, SUP_J = 1024 / BN;
        const int cbi0 = bi0 / ci, cbi1 = (bi1 + ci - 1) / ci;
        std::vector<int2> tiles;
        auto needed = [&](int cbi, int bj) {
            // mirror mode keeps a tile iff it holds a pair (i, j) with j >= i; a symmetric slab
            // (col_begin > 0) needs nothing left of its first row
            if (!cosums && (int64_t)(bj + 1) * BN <= h->col_begin) return false;
            return !mirror || (int64_t)(bj + 1) * BN > (int64_t)(cbi * ci) * BM;
        };
        for (int sbi = cbi0; sbi < cbi1; sbi += SUP_I)
            for (int sbj = 0; sbj < nbj; sbj += SUP_J)
                for (int cbi = sbi; cbi < sbi + SUP_I && cbi < cbi1; cbi++)
                    for (int bj = sbj; bj < sbj + SUP_J && bj < nbj; bj++)
                        if (needed(cbi, bj)) tiles.push_back(make_int2(cbi, bj));
        RS_TRY(upload_tiles(h, tiles, &h->tile_buf, &h->tile_buf_bytes));
        memcpy(h->tile_key, key, sizeof(key));
        h->tile_count = (int32_t)tiles.size();
    }
    if (h->tile_count == 0) return RS_OK;

    TcArgs a{};
    a.tiles = reinterpret_cast<const int2 *>(h->tile_buf);
    a.num_tiles = h->tile_count;
    a.n_left = h->n_left;
    a.row_begin = rb;
    a.row_end = re;
    a.mirror = mirror ? 1 : 0;
    a.sims = h->sims;
    a.ld_s = h->ld_s;
    a.row_cnt = h->row_cnt;
    a.row_sum = h->row_sum;
    a.cosums = d_cosums;
    a.cos_row0 = cos_row0;
    a.cos_nrows = cos_nrows;
    int32_t rc;
    switch (mode) {
    case TC_COSINE: rc = use_pair ? launch_pair<TC_COSINE>(h, a) : launch_single<TC_COSINE>(h, a); break;
    case TC_MSD: rc = use_pair ? launch_pair<TC_MSD>(h, a) : launch_single<TC_MSD>(h, a); break;
    case TC_SLOPE: rc = use_pair ? launch_pair<TC_SLOPE>(h, a) : launch_single<TC_SLOPE>(h, a); break;
    case TC_PEARSON: rc = pearson_i128(h) ? launch_single<TC_PEARSON128>(h, a) : launch_single<TC_PEARSON>(h, a); break;
    default: rc = launch_single<TC_COSUMS>(h, a); break;   // TC_COSUMS
    }
    RS_TRY(rc);
    if (!cosums) h->prof.sim_launches++;
    h->prof.total_launches++;
    return RS_OK;
}
