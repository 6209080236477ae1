// gemm_topk_sm100.cu -- K2: the query x database contraction on 5th-gen tensor cores with a fused
// |x|^2 - 2 q.x epilogue and on-chip top-k'.  The distance matrix is never written anywhere.
//
// Replaces faiss's exhaustive_L2sqr_blas / exhaustive_inner_product_blas (sgemm over 4096 x 1024
// blocks + heap update; the nq >= 20 path behind index.search, faiss_store.py:64,
// rag_datastore_manager.py:218) with one persistent, warp-specialised sm_100a kernel:
//
//   warp 0   TMA producer: cp.async.bulk.tensor.2d (SWIZZLE_128B) of bf16 database blocks into an mbarrier ring; the
//            [128 x d] query tile is loaded once per segment and stays resident in shared memory when dpad <= 384
//            (QRES), otherwise it is streamed per k-block with the database block
//   warp 1   MMA issuer: one elected lane issues tcgen05.mma.kind::f16, M = queries x N = 256 database rows x K = 16,
//            fp32 accumulators in TMEM (512 columns = two 128 x 256 accumulators, double buffered); tcgen05.commit
//            frees the smem stage / publishes the accumulator.  Two forms:
//              single CTA   cta_group::1, M = 128
//              CTA pair     cta_group::2, M = 256 over the two SMs of a TPC (batches of >= 2 query tiles): each CTA owns
//                           128 of the pair's queries and stages its 128-row half of every database block; the leader
//                           issues the MMAs for both, commits are multicast to both CTAs
//   warp 2   TMEM allocator
//   warp 3   bias loader: |x~|^2 (L2) / -mu.x (IP) of the tile's 256 rows (+inf past the end) -> smem
//   warps 4-11 (LIST) / 4-7 (HEAP)  epilogue: tcgen05.ld 32 columns at a time (double buffered); queries are the M
//            dimension, so TMEM lane = query and a thread's state is private to (query, column half).  Per value one
//            FFMA (bias - 2 acc), one compare against a register threshold; the rare survivor is kept.  Two modes:
//            LIST: survivors are appended to the thread's candidate list in global memory (fire-and-forget stores).
//              The threshold is SHARED across the units that stream different parts of the database for the same
//              query: voucher lists publish their j-th best key so far; T* = max over g vouchers (g * j >= k') is
//              an upper bound of the global k'-th best, far tighter than any single stream's own k'-th best.
//            HEAP (more than one wave of query tiles, or a database of one tile): thread-private max-heap of k' in
//              shared memory ([slot][thread] layout => conflict free), threshold = heap root.
//
// Work split (LIST): the pass's work -- query tile units x database -- is cut into one EQUAL share per unit (CTA or CTA
// pair, one wave), whatever the two counts are; a unit runs the tail of one query tile and, if its share spills over,
// the head of the next (struct Seg below).  Every segment sweeps the database front to back in rounds, all segments
// together, so a block that several query tiles need is fetched from HBM once and re-read from L2.
//
// Roofline: nq <= 128 -> HBM-bound, algorithmic bytes n * dpad * 2; large nq -> tensor-bound, 2 * nq * n * d flop.
#include <cuda.h>
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "rerank.cuh"

namespace b2f {

namespace k2 {

constexpr int BM = 128;        // queries per tile  (UMMA M)
constexpr int BN = 256;        // database rows per tile (UMMA N)
constexpr int BK = 64;         // bf16 elements per stage along d: 128 bytes = one swizzle atom
constexpr int UMMA_K = 16;
constexpr int STAGES_HEAP = 3;
constexpr int STAGES_LIST = 4;
constexpr int STAGES_QRES = 3;    // Q-resident variant: stages hold database blocks only (32 KB each)
constexpr int QRES_MAX_KB = 6;    // query tile kept resident in smem when dpad <= 384 (6 x 16 KB)
constexpr int LIST_CAP_MIN = 128;  // entries per (query, split) candidate list: 128 / 256 / 512 by stream length
constexpr int JSLOTS = 16;        // register slots for the split-local j-th best (j <= 16: LIST mode from 2 splits up)
constexpr int A_BYTES = BM * BK * 2;  // 16 KB
constexpr int B_BYTES = BN * BK * 2;  // 32 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int EPI_THREADS = 128;          // TMEM lanes = queries per CTA tile
constexpr int EPI_WARPS_HEAP = 4;
constexpr int EPI_WARPS_LIST = 8;         // two warps per TMEM lane quarter, each owning half of the tile's columns
__host__ __device__ constexpr int k2_threads(bool list) { return 128 + 32 * (list ? EPI_WARPS_LIST : EPI_WARPS_HEAP); }
constexpr int TMEM_COLS = 512;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(x), "r"(y)
        : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (rows of 128 bytes, 8-row atoms 1024 B apart)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);  // start address
    d |= (uint64_t)1 << 16;                  // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;        // stride byte offset: next 8-row group
    d |= (uint64_t)1 << 46;                  // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                  // SWIZZLE_128B
    return d;
}

// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, M=128, N=256
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(kIdesc), "r"(accumulate)
        : "memory");
}
// ---- cta_group::2 (CTA pair) primitives --------------------------------------------------------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;  // clears the CTA-rank bit of a shared::cluster address -> the even CTA
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load issued by either CTA of the pair; the bytes are credited to the LEADER CTA's mbarrier
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & kPeerBitMask), "r"(x), "r"(y)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// commit of the pair's MMAs: arrives on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
// arrive on the barrier at the same offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
    asm volatile(
        "{\n\t"
        ".reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(rank)
        : "memory");
}
// kind::f16 instruction descriptor for the pair: M = 256 (128 per CTA), N = 256
constexpr uint32_t kIdescPair = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
constexpr int STAGES_PAIR = 6;        // pair variant: each CTA stages its 128-row half of the database block (16 KB)

__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ uint32_t tmem_ld1(uint32_t taddr) {
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr) : "memory");
    return v;
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Database tiles of every (unit, segment), computed on the host with SegIter and passed by value: the epilogue -- the
// kernel's critical path, at the register cap -- then runs a counted loop and takes each tile's first row from shared
// memory (the bias loader publishes it with the biases) instead of stepping an iterator of its own.
struct SegCounts {
    int32_t n[2 * kNumSMs];
};

template <int KP, int NST, int QKB = 0, bool PAIRED = false>
struct Smem {
    static constexpr size_t q_off = 0;                                   // resident query tile: QKB x 16 KB
    static constexpr size_t stage_bytes = PAIRED ? (size_t)B_BYTES / 2 : (QKB ? (size_t)B_BYTES : (size_t)STAGE_BYTES);
    static constexpr size_t stages_off = (size_t)QKB * A_BYTES;
    static constexpr size_t heapk_off = stages_off + (size_t)NST * stage_bytes;
    static constexpr size_t heapi_off = heapk_off + (size_t)EPI_THREADS * KP * 4;
    static constexpr size_t bias_off = heapi_off + (size_t)EPI_THREADS * KP * 4;
    // LIST mode (KP == 0): per-warp staging of one chunk's 32 accumulators per lane, [warp][column][lane]
    static constexpr size_t xpose_off = bias_off + 2 * BN * 4;
    static constexpr size_t bar_off = xpose_off + (KP == 0 ? (size_t)EPI_WARPS_LIST * 32 * 32 * 4 : 0);
    static constexpr int nbars = 2 * NST + 10;
    static constexpr size_t tmem_off = bar_off + nbars * 8;
    static constexpr size_t total = tmem_off + 32;   // TMEM base holder, die-ticket scratch, row0 of the tile in each bias buffer
    static constexpr size_t alloc = total;  // the dynamic smem base is declared __align__(1024)
};

// LIST-mode arguments (all device pointers)
struct ListArgs {
    float* shared_thr;   // [nq_pad][nsplits]  each split's published j-th best key (init: huge)
    uint2* cand;         // [nq_pad * nsplits][cap]  (key bits, row id)
    int32_t* counts;     // [nq_pad * nsplits]  entries appended (may exceed cap => overflow)
    int kp;              // k': every query's lists together must cover the k' best
    int nl_stride;       // lists per query allocated (the largest per-tile list count)
    int cap;             // entries per list
    float* final_thr;    // [nq_pad * nsplits]  threshold the list was pruned against at the end of the stream
    bool die_aware;      // die-aware unit assignment (takes tickets from die_ctr)
    int32_t* die_ctr;    // [4] ticket counters (zero between launches)
    int bal_T;           // balanced work split: query tile units (pair tiles when PAIR) ...
    int bal_U;           // ... shared evenly by this many units (CTAs / CTA pairs); T <= U
    int bal_R;           // database tiles per round of the interleaved sweep
    const float* range_thr;  // range pass: fixed threshold per query -- every row at or below it is listed; no sharing, no refresh
};

// ---- balanced work split (LIST mode) -----------------------------------------------------------------------------
// The work of a pass is a line of T query tile units x the whole database.  It is cut into U EQUAL intervals, one per
// unit (CTA or CTA pair), whatever T and U are: unit u owns [u T, (u + 1) T) in units of 1/U of a query tile.  With
// T <= U an interval touches at most two query tiles, so a unit runs one or two SEGMENTS (query tile, fraction of the
// database) back to back -- the tail of one tile, then the head of the next.  (Before: units were dealt round-robin
// over the tiles and a pass lasted as long as the tiles with the fewest units -- 32 pair tiles over 74 pairs ran at
// the pace of the 2-unit tiles, 2.31 being the fair share: 15% lost; balancing by query chunking cost extra passes.)
//
// Which database tiles a segment [p0, p1) of a query tile takes: the database is swept in ROUNDS of R tiles; in round
// r the segments of a query tile partition the round's R tiles at cut(p) = (p / U * R + phi_r) >> 32 in 32.32 fixed
// point, phi_r a golden-ratio dither so that every segment's total is proportional to its length (+-2 tiles).  All
// segments therefore move through the database front to back TOGETHER, a round at a time: a block that several
// query tiles need is fetched from HBM once and found in L2 by the others (the point of the former strided walk).
//
// Order of a unit's two segments: the LONGER piece first.  A piece that runs first starts at kernel start ("first
// wave"); the shorter piece follows when the first is done.
//
// Lists / shared thresholds: a query tile's pieces are its list SLOTS -- first-wave pieces in position order (whole
// units, plus the head / tail piece when it is the longer part of its unit: at least half a share), then the second-
// wave pieces.  The first-wave pieces VOUCH: every one of their lists publishes its j-th best key, j proportional to
// the piece's length (a j-th best of few rows is loose, so a shorter piece vouches for fewer rows), scaled so that the
// tile's voucher lists together vouch for >= k' rows.  Every list of the tile, voucher or not, prunes against the
// maximum of the consulted values: with pieces of unequal length all voucher lists are consulted, with whole units
// only (equal j) any g = ceil(k' / j) of them.  The vouchers cover all but the shorter halves of the boundary units
// (~90 % of the rows at 2.3 units per tile), so the shared bound sits close to the k'-th best of everything seen.
struct Seg {
    int qtile;         // query tile unit
    int slot;          // list slot within the tile
    int nv;            // voucher slots of the tile: [0, nv)
    uint32_t p0, p1;   // in-tile range in units of 1/U tile
    int j;             // rows each of this piece's lists vouches for (vouchers; 1 otherwise)
    int g;             // voucher lists a thread of this tile consults
};
struct TileInfo {
    int u_lo, u_hi;               // units that start inside the tile
    int head_len, tail_len;       // head piece (unit u_lo - 1 spilling in) / what a crossing unit u_hi covers; 0 = none
    bool head_first, tail_first;  // the piece is the longer part of its unit, i.e. first wave
    int nfull, nfw, nsw;          // whole units; first-wave pieces = voucher slots [0, nfw); second-wave pieces behind them
    int lv;                       // total voucher length in units of 1/U tile
    int jfull;                    // rows a list of a whole unit vouches for
    int g;                        // voucher lists a thread consults
};
__host__ __device__ __forceinline__ TileInfo tile_info(int t, int T, int U, int kp, int halves) {
    TileInfo ti;
    ti.u_lo = (int)(((int64_t)t * U + T - 1) / T);
    ti.u_hi = (int)((((int64_t)t + 1) * U + T - 1) / T) - 1;
    ti.head_len = (int)((int64_t)ti.u_lo * T - (int64_t)t * U);                    // [0, T)
    const int last_len = (int)(((int64_t)t + 1) * U - (int64_t)ti.u_hi * T);       // (0, T]
    ti.tail_len = last_len < T ? last_len : 0;
    ti.head_first = ti.head_len > 0 && 2 * ti.head_len > T;
    ti.tail_first = ti.tail_len > 0 && 2 * ti.tail_len >= T;
    ti.nfull = ti.u_hi - ti.u_lo + 1 - (ti.tail_len > 0 ? 1 : 0);
    ti.nfw = ti.nfull + (ti.head_first ? 1 : 0) + (ti.tail_first ? 1 : 0);
    ti.nsw = ((ti.head_len > 0 && !ti.head_first) ? 1 : 0) + ((ti.tail_len > 0 && !ti.tail_first) ? 1 : 0);
    ti.lv = ti.nfull * T + (ti.head_first ? ti.head_len : 0) + (ti.tail_first ? ti.tail_len : 0);
    if (kp > 0) {
        ti.jfull = (int)(((int64_t)kp * T + (int64_t)halves * ti.lv - 1) / ((int64_t)halves * ti.lv));
        const bool uniform = !ti.head_first && !ti.tail_first;   // whole units only: every voucher list vouches jfull rows
        const int nvs = ti.nfw * halves;
        ti.g = uniform ? (kp + ti.jfull - 1) / ti.jfull : nvs;
        if (ti.g > nvs) ti.g = nvs;
    } else {
        ti.jfull = 1;
        ti.g = 1;
    }
    return ti;
}
// rows a list of a voucher piece of length len (in 1/U tile) vouches for
__host__ __device__ __forceinline__ int piece_j(const TileInfo& ti, int len, int T) {
    return (int)(((int64_t)ti.jfull * len + T - 1) / T);
}
// The one or two segments of unit u, in the order it runs them; returns their number.
__host__ __device__ __forceinline__ int unit_segments(int u, int T, int U, int kp, int halves, Seg (&seg)[2]) {
    const int64_t S0 = (int64_t)u * T, S1 = S0 + T;
    const int a = (int)(S0 / U), b = (int)(S1 / U);
    const int fa = (int)(S0 - (int64_t)a * U), fb = (int)(S1 - (int64_t)b * U);
    const TileInfo ta = tile_info(a, T, U, kp, halves);
    if (b == a || fb == 0) {   // a whole unit inside tile a
        seg[0].qtile = a; seg[0].slot = (ta.head_first ? 1 : 0) + (u - ta.u_lo); seg[0].nv = ta.nfw;
        seg[0].p0 = (uint32_t)fa; seg[0].p1 = (uint32_t)(b > a ? U : fb);
        seg[0].j = ta.jfull; seg[0].g = ta.g;
        return 1;
    }
    // the unit crosses into tile b = a + 1: a tail piece of tile a, a head piece of tile b
    const TileInfo tb = tile_info(b, T, U, kp, halves);
    Seg tail, head;
    tail.qtile = a; tail.nv = ta.nfw; tail.p0 = (uint32_t)fa; tail.p1 = (uint32_t)U; tail.g = ta.g;
    tail.slot = ta.tail_first ? ta.nfw - 1 : ta.nfw + ((ta.head_len > 0 && !ta.head_first) ? 1 : 0);
    tail.j = ta.tail_first ? piece_j(ta, U - fa, T) : 1;
    head.qtile = b; head.nv = tb.nfw; head.p0 = 0u; head.p1 = (uint32_t)fb; head.g = tb.g;
    head.slot = tb.head_first ? 0 : tb.nfw;
    head.j = tb.head_first ? piece_j(tb, fb, T) : 1;
    const bool tail_runs_first = 2 * (U - fa) >= T;
    seg[0] = tail_runs_first ? tail : head;
    seg[1] = tail_runs_first ? head : tail;
    return 2;
}
// The database tiles of one segment, in sweep order.  Contiguous form (HEAP mode): tiles [t0, t1).
// Every role of the kernel steps one of these per tile and the epilogue is the kernel's critical path, so the state
// is 32-bit and a step is a compare + add; a round change is two mul.hi / mul.lo pairs (the first version carried
// 64-bit fixed point through every step: +9% executed instructions, -8% kernel throughput, ncu r02e).
// (Cost-aware cuts were tried and dropped: a unit that runs two segments pays ~22 us for the switch -- per-unit
// %globaltimer stamps, tools/k2_trace.py: 8192 queries on a 125 k-row shard, units with one segment issue their last MMA
// at 614 us on average, units with two at 641 us.  Warping the cuts so that those units get ~6 tiles less and the whole
// units the same small extra equalised the two groups (630 / 635 us) but not the kernel (0.646 -> 0.648 ms; nq = 4096
// -1.4 %, C2 +0.7 %): the units' speeds are coupled through the chip-wide sustained tensor rate, of which K2 has 97 %.)
struct SegIter {
    uint32_t F0, F1;      // in-tile bounds as Q0.32 fractions of the tile; full1: the segment ends at the tile's end (1.0)
    int R, NR, r, j, jend, base, ntiles;
    bool full1;
    __host__ __device__ __forceinline__ void init(uint32_t p0, uint32_t p1, int U, int R_, int64_t ntiles_) {
        F0 = (uint32_t)(((uint64_t)p0 << 32) / (uint32_t)U);
        full1 = p1 >= (uint32_t)U;
        F1 = full1 ? 0u : (uint32_t)(((uint64_t)p1 << 32) / (uint32_t)U);
        R = R_;
        ntiles = (int)ntiles_;
        NR = (int)((ntiles_ + R_ - 1) / R_);
        r = -1;
        j = jend = 0;
        base = -R_;
    }
    __host__ __device__ __forceinline__ void init_contig(int64_t t0, int64_t t1) {
        F0 = F1 = 0u; full1 = false; R = 0; NR = 0; r = 0; base = 0;
        ntiles = (int)t1;
        j = (int)t0; jend = (int)t1;
    }
    // (F * Rr + phi) >> 32 for a Q0.32 fraction F
    static __host__ __device__ __forceinline__ int cut(uint32_t F, uint32_t Rr, uint32_t phi) {
#ifdef __CUDA_ARCH__
        const uint32_t hi = __umulhi(F, Rr);
#else
        const uint32_t hi = (uint32_t)(((uint64_t)F * Rr) >> 32);
#endif
        const uint32_t lo = F * Rr;
        return (int)(hi + ((lo + phi) < lo ? 1u : 0u));
    }
    __host__ __device__ __forceinline__ int count() {   // tiles of the whole segment (consumes the iterator)
        int c = jend - j;
        while (++r < NR) {
            base += R;
            const uint32_t Rr = (r == NR - 1) ? (uint32_t)(ntiles - base) : (uint32_t)R;
            const uint32_t phi = (uint32_t)r * 2654435769u;
            c += (full1 ? (int)Rr : cut(F1, Rr, phi)) - cut(F0, Rr, phi);
        }
        return c;
    }
    __host__ __device__ __forceinline__ int64_t next() {   // -1 when exhausted
        while (true) {
            if (j < jend) return (int64_t)(base + j++);
            if (++r >= NR) return -1;
            base += R;
            // the last round holds what is left of the database and is shared out the same way
            const uint32_t Rr = (r == NR - 1) ? (uint32_t)(ntiles - base) : (uint32_t)R;
            const uint32_t phi = (uint32_t)r * 2654435769u;
            j = cut(F0, Rr, phi);
            jend = full1 ? (int)Rr : cut(F1, Rr, phi);
        }
    }
};

// thread-private max-heap in shared memory, element j of thread t at [j * 128 + t].
// sift (key,id) down from the root of the first n heap slots.
template <int KP>
__device__ __forceinline__ void heap_sift_down_n(float* hk, int32_t* hi, int tid, int n, float key, int32_t id) {
    int i = 0;
    while (true) {
        const int l = 2 * i + 1;
        if (l >= n) break;
        int m = l;
        float mk = hk[l * EPI_THREADS + tid];
        int32_t mi = hi[l * EPI_THREADS + tid];
        if (l + 1 < n) {
            const float rk = hk[(l + 1) * EPI_THREADS + tid];
            const int32_t ri = hi[(l + 1) * EPI_THREADS + tid];
            if (cand_less(mk, mi, rk, ri)) {
                m = l + 1;
                mk = rk;
                mi = ri;
            }
        }
        if (!cand_less(key, id, mk, mi)) break;
        hk[i * EPI_THREADS + tid] = mk;
        hi[i * EPI_THREADS + tid] = mi;
        i = m;
    }
    hk[i * EPI_THREADS + tid] = key;
    hi[i * EPI_THREADS + tid] = id;
}

// Rare path of the epilogue, kept out of line so the 32x-unrolled compare loop stays small:
// replace the heap root (the current worst of the thread's k' best) and return the new threshold.
template <int KP>
__device__ __noinline__ float heap_push(float* hk, int32_t* hi, int tid, float key, int32_t id) {
    heap_sift_down_n<KP>(hk, hi, tid, KP, key, id);
    return hk[tid];
}


// Diagnostics build only (-DB2F_K2_TRACE, tools/k2_trace.sh): per-CTA %globaltimer stamps of the kernel's phases.
#ifdef B2F_K2_TRACE
__device__ unsigned long long g_k2_trace[2 * kNumSMs * 12];
#define K2_STAMP(slot)                                                   \
    do {                                                                 \
        unsigned long long t_;                                           \
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));           \
        g_k2_trace[blockIdx.x * 12 + (slot)] = t_;                       \
    } while (0)
#define K2_NOTE(slot, v) g_k2_trace[blockIdx.x * 12 + (slot)] = (unsigned long long)(v)
#else
#define K2_STAMP(slot) do { } while (0)
#define K2_NOTE(slot, v) do { } while (0)
#endif

template <int KP, bool L2, bool LIST, bool QRES, bool PAIR>
__global__ void __launch_bounds__(k2_threads(LIST), 1)
tensor_scan_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x,
                   const float* __restrict__ norms, int64_t n, int nq, int kblocks, int nq_tiles, int nsplits,
                   float* __restrict__ pk, int32_t* __restrict__ pi, ListArgs la, const __grid_constant__ SegCounts seg_counts) {
    static_assert(!QRES || LIST, "the Q-resident variant exists for LIST mode only");
    static_assert(!PAIR || QRES, "the CTA-pair variant builds on the Q-resident one");
    constexpr int STAGES = PAIR ? STAGES_PAIR : (QRES ? STAGES_QRES : (LIST ? STAGES_LIST : STAGES_HEAP));
    using L = Smem<LIST ? 0 : KP, STAGES, QRES ? QRES_MAX_KB : 0, PAIR>;
    constexpr uint32_t kStageBytes = (uint32_t)L::stage_bytes;
    constexpr int EPI_WARPS = LIST ? EPI_WARPS_LIST : EPI_WARPS_HEAP;
    constexpr int HALVES = EPI_WARPS / 4;        // column halves of a tile, one per epilogue warp of a lane quarter
    constexpr int COLS = BN / HALVES;            // columns of each tile that one thread examines
    extern __shared__ __align__(1024) uint8_t smem[];  // SWIZZLE_128B tiles need 1024-byte alignment
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    float* heap_k = reinterpret_cast<float*>(smem + L::heapk_off);
    int32_t* heap_i = reinterpret_cast<int32_t*>(smem + L::heapi_off);
    float* bias = reinterpret_cast<float*>(smem + L::bias_off);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::bar_off);
    uint64_t* full_bar = bars;                     // [STAGES]  TMA -> MMA
    uint64_t* empty_bar = bars + STAGES;           // [STAGES]  MMA -> TMA
    uint64_t* tmem_full = bars + 2 * STAGES;       // [2]       MMA -> epilogue
    uint64_t* tmem_empty = bars + 2 * STAGES + 2;  // [2]       epilogue -> MMA, bias loader
    uint64_t* bias_full = bars + 2 * STAGES + 4;   // [2]       bias loader -> epilogue
    uint64_t* q_full = bars + 2 * STAGES + 6;      // [1]       resident query tile landed (QRES)
    uint64_t* bias_empty = bars + 2 * STAGES + 7;  // [2]       epilogue -> bias loader (PAIR: local to each CTA)
    uint64_t* q_empty = bars + 2 * STAGES + 9;     // [1]       MMA -> TMA: the resident query tile may be replaced (next segment)
    uint32_t* tmem_base_holder = reinterpret_cast<uint32_t*>(smem + L::tmem_off);
    volatile int32_t* tile_row0 = reinterpret_cast<volatile int32_t*>(smem + L::tmem_off + 16);   // [2], written with bias[acc]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) K2_STAMP(0);
    // PAIR: a cluster of two CTAs (one TPC) works on 256 queries x one database stream; CTA rank r owns
    // queries [128 r, 128 r + 128) of the pair tile and stages rows [128 r, 128 r + 128) of every
    // 256-row database block; the leader (rank 0) issues tcgen05.mma.cta_group::2 for both.
    const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;
    int unit = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;       // cluster (PAIR) or CTA index
    const int64_t ntiles = (n + BN - 1) / BN;
    if constexpr (LIST) {
        // Die-aware work assignment.  Units whose segments sit at the same place inside their query tiles read the
        // same database tiles of every round at about the same time; when they sit on both dies the second reader
        // pulls every block across the die-to-die L2 fabric.  Logical units are therefore handed out in the order of
        // their position inside the tile (frac(u T / U)): the hardware units of die 0 take tickets from the front of
        // that order, those of die 1 from the back, so each die serves (about) one half of every round's tiles.
        if (la.die_aware) {
            // (in the spare bytes behind the TMEM base holder: the pair variant has no room for static shared memory)
            int& s_unit = *reinterpret_cast<int*>(smem + L::tmem_off + 8);
            int& s_idx = *reinterpret_cast<int*>(smem + L::tmem_off + 12);
            const int U = la.bal_U, T = la.bal_T;
            if (threadIdx.x == 0 && cta_rank == 0) {
                uint32_t smid;
                asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
                const int die = smid >= (uint32_t)(kNumSMs / 2) ? 1 : 0;
                const int t = atomicAdd(la.die_ctr + die, 1);
                s_idx = die == 0 ? t : U - 1 - t;   // front / back of the position order; U tickets in total, no collision
                if (atomicAdd(la.die_ctr + 3, 1) == U - 1) {   // every unit has its ticket: re-arm the counters
                    la.die_ctr[0] = 0; la.die_ctr[1] = 0; la.die_ctr[2] = 0; la.die_ctr[3] = 0;
                }
            }
            if constexpr (PAIR) {
                if (threadIdx.x == 0 && cta_rank == 0) {
                    uint32_t remote;
                    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(&s_idx)), "r"(1));
                    asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(remote), "r"(s_idx) : "memory");
                }
                cluster_sync_all();
            } else {
                __syncthreads();
            }
            // the unit whose (position, index) key has rank s_idx: thread v < U counts the keys below its own
            const int want = s_idx;
            for (int v = threadIdx.x; v < U; v += blockDim.x) {
                const int kv = (v * T) % U;   // U, T <= 148
                int rank = 0, kw = 0;
                for (int w = 0; w < U; w++) {
                    rank += (kw < kv || (kw == kv && w < v)) ? 1 : 0;
                    kw += T;                  // (w T) mod U, incrementally (T <= U)
                    if (kw >= U) kw -= U;
                }
                if (rank == want) s_unit = v;
            }
            __syncthreads();
            unit = s_unit;
        }
    }
    // ---- this unit's work ---------------------------------------------------------------------------------------
    // LIST: one or two segments of the balanced split (see Seg above).  HEAP: one contiguous database range of the
    // (query tile, split) the unit index names.
    Seg seg[2];
    int nseg = 1;
    int64_t heap_t0 = 0, heap_t1 = 0;
    const int units_per_split = nq_tiles;   // HEAP mode only (never PAIR)
    const int split = LIST ? 0 : unit / units_per_split;
    if constexpr (LIST) {
        nseg = unit_segments(unit, la.bal_T, la.bal_U, la.kp, HALVES, seg);
        if (nseg == 1) seg[1] = seg[0];
    } else {
        seg[0].qtile = unit % units_per_split; seg[0].slot = split; seg[0].nv = 0; seg[0].p0 = 0u; seg[0].p1 = 0u;
        seg[0].j = 1; seg[0].g = 1;
        heap_t0 = ntiles * split / nsplits;
        heap_t1 = ntiles * (split + 1) / nsplits;
    }
    // (fields are selected with ?: instead of indexing seg[] with the loop variable: a dynamically indexed local array
    // lives in local memory, and values loaded from there are not warp-uniform for the compiler)
    auto seg_of = [&](int s_) {
        Seg r;
        r.qtile = s_ == 0 ? seg[0].qtile : seg[1].qtile;
        r.slot = s_ == 0 ? seg[0].slot : seg[1].slot;
        r.nv = s_ == 0 ? seg[0].nv : seg[1].nv;
        r.p0 = s_ == 0 ? seg[0].p0 : seg[1].p0;
        r.p1 = s_ == 0 ? seg[0].p1 : seg[1].p1;
        r.j = s_ == 0 ? seg[0].j : seg[1].j;
        r.g = s_ == 0 ? seg[0].g : seg[1].g;
        return r;
    };
    auto seg_iter = [&](int s_) {
        SegIter it;
        if constexpr (LIST) {
            const Seg g = seg_of(s_);
            it.init(g.p0, g.p1, la.bal_U, la.bal_R, ntiles);
        } else {
            it.init_contig(heap_t0, heap_t1);
        }
        return it;
    };
    auto seg_qt = [&](int s_) {
        const int qtile = s_ == 0 ? seg[0].qtile : seg[1].qtile;
        return PAIR ? qtile * 2 + (int)cta_rank : qtile;
    };
    // tiles of segment s_ (host-computed with SegIter, passed by value): the loop count of the roles that need no tile index
    auto seg_tiles_of = [&](int s_) { return LIST ? seg_counts.n[2 * unit + s_] : (int)(heap_t1 - heap_t0); };

#ifdef B2F_K2_TRACE
    if (threadIdx.x == 0) {
        uint32_t smid_;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid_));
        K2_NOTE(8, unit + 1);
        K2_NOTE(9, smid_);
    }
#endif
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_q)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_x)) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; s++) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; a++) {
            mbar_init(&tmem_full[a], 1);
            mbar_init(&tmem_empty[a], (PAIR ? 2 : 1) * EPI_WARPS);  // one arrive per epilogue warp (of both CTAs for a pair)
            mbar_init(&bias_full[a], 1);
            mbar_init(&bias_empty[a], EPI_WARPS);
        }
        mbar_init(q_full, 1);
        mbar_init(q_empty, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        if constexpr (PAIR) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_holder)),
                         "r"((uint32_t)TMEM_COLS)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_holder)),
                         "r"((uint32_t)TMEM_COLS)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();  // the peer's barriers must be initialised before any remote arrive / TMA credit
    tc_fence_after();
    const uint32_t tmem_base = *tmem_base_holder;
    if (threadIdx.x == 0) K2_STAMP(1);

    if (warp == 0) {
        // ===================== TMA producer =====================
        // The WHOLE warp runs the loops (warp-uniform control flow and values, so descriptors and addresses live in the
        // uniform datapath); lane 0 alone issues.  With the loops inside `if (lane == 0)` the compiler loses uniformity
        // as soon as the trip counts come from an iterator: every tcgen05.mma then cost 17 instructions (five
        // R2UR.BROADCAST among them) instead of 10 and the single issuing thread became the kernel's bottleneck
        // (ncu r02e: the epilogue's wait for tmem_full went from 6.6% to 11% of the stall samples, -6% throughput).
        {
            int stage = 0;
            uint32_t phase = 0;
#pragma unroll 1
#pragma unroll 1
        for (int sgi = 0; sgi < nseg; sgi++) {   // (never unrolled: two copies of the loops below thrash the instruction cache)
                const int qt = seg_qt(sgi);
                if constexpr (QRES) {
                    // the whole query tile (all k-blocks) is loaded once per segment and stays in shared memory; a second
                    // segment replaces it once the MMAs of the first have read it for the last time
                    if (sgi > 0) mbar_wait(q_empty, (uint32_t)((sgi - 1) & 1));
                    if (lane == 0) {
                        if constexpr (PAIR) {
                            // both CTAs load their own 128-query tile; the bytes of both are credited to the leader's barrier
                            if (cta_rank == 0) mbar_expect_tx(q_full, (uint32_t)(2 * kblocks * A_BYTES));
                            for (int kb = 0; kb < kblocks; kb++)
                                tma_load_2d_pair(smem + L::q_off + (size_t)kb * A_BYTES, &map_q, kb * BK, qt * BM, q_full);
                        } else {
                            mbar_expect_tx(q_full, (uint32_t)(kblocks * A_BYTES));
                            for (int kb = 0; kb < kblocks; kb++) tma_load_2d(smem + L::q_off + (size_t)kb * A_BYTES, &map_q, kb * BK, qt * BM, q_full);
                        }
                    }
                    __syncwarp();
                }
                SegIter it = seg_iter(sgi);
                for (int64_t dbt; (dbt = it.next()) >= 0;) {
                    const int row0 = __shfl_sync(kFull, (int)(dbt * BN), 0);   // (warp-uniform for the compiler, as in the MMA issuer)
                    for (int kb = 0; kb < kblocks; kb++) {
                        mbar_wait(&empty_bar[stage], phase ^ 1);
                        const int ustage = __shfl_sync(kFull, stage, 0);
                        uint8_t* sa = smem + L::stages_off + (size_t)ustage * kStageBytes;
                        if (lane == 0) {
                            if constexpr (PAIR) {
                                // this CTA's half of the 256-row block; the leader's full barrier collects both halves
                                if (cta_rank == 0) mbar_expect_tx(&full_bar[ustage], 2 * kStageBytes);
                                tma_load_2d_pair(sa, &map_x, kb * BK, row0 + (int)cta_rank * (BN / 2), &full_bar[ustage]);
                            } else {
                                mbar_expect_tx(&full_bar[ustage], kStageBytes);
                                if constexpr (!QRES) tma_load_2d(sa, &map_q, kb * BK, qt * BM, &full_bar[ustage]);
                                tma_load_2d(sa + (QRES ? 0 : A_BYTES), &map_x, kb * BK, row0, &full_bar[ustage]);
                            }
                        }
                        __syncwarp();
                        if (++stage == STAGES) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        // (whole warp, uniform control flow; lane 0 issues -- see the producer)
        if (cta_rank == 0) {  // PAIR: only the leader CTA issues MMAs
            int stage = 0;
            uint32_t phase = 0;
            int gt = 0;   // tiles so far: accumulator buffer and barrier phases run on across segments
#pragma unroll 1
#pragma unroll 1
        for (int sgi = 0; sgi < nseg; sgi++) {   // (never unrolled: two copies of the loops below thrash the instruction cache)
                if constexpr (QRES) mbar_wait(q_full, (uint32_t)(sgi & 1));
                const int seg_tiles = seg_tiles_of(sgi);
#pragma unroll 1
                for (int t = 0; t < seg_tiles; t++, gt++) {
                    const int acc = gt & 1;
                    const uint32_t acc_phase = (gt >> 1) & 1;
                    mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                    tc_fence_after();
                    // (broadcast from lane 0: tells the compiler the operands are warp-uniform, so the descriptor arithmetic
                    // runs in the uniform datapath instead of per-MMA R2UR.BROADCAST sequences)
                    const uint32_t d_tmem = __shfl_sync(kFull, tmem_base + (uint32_t)(acc * BN), 0);
                    for (int kb = 0; kb < kblocks; kb++) {
                        mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        if (gt == 0 && kb == 0 && lane == 0) K2_STAMP(2);
                        const uint32_t sa = __shfl_sync(kFull, smem_u32(smem + L::stages_off + (size_t)stage * kStageBytes), 0);
                        const uint32_t qa = __shfl_sync(kFull, smem_u32(smem + L::q_off + (size_t)kb * A_BYTES), 0);
                        const uint64_t adesc = make_smem_desc(QRES ? qa : sa);
                        const uint64_t bdesc = make_smem_desc(sa + (QRES ? 0 : A_BYTES));
                        if (lane == 0) {
#pragma unroll
                            for (int k = 0; k < BK / UMMA_K; k++) {
                                // advance both descriptors by 32 bytes (16 bf16) inside the 128-byte swizzle atom
                                if constexpr (PAIR)
                                    umma_bf16_pair(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), kIdescPair, (kb | k) != 0 ? 1u : 0u);
                                else
                                    umma_bf16(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), (kb | k) != 0 ? 1u : 0u);
                            }
                            if constexpr (PAIR) umma_commit_pair(&empty_bar[stage]);
                            else umma_commit(&empty_bar[stage]);
                        }
                        __syncwarp();
                        if (++stage == STAGES) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                    if (lane == 0) {
                        if constexpr (PAIR) umma_commit_pair(&tmem_full[acc]);
                        else umma_commit(&tmem_full[acc]);
                    }
                    __syncwarp();
                }
                if constexpr (QRES) {
                    if (sgi + 1 < nseg && lane == 0) K2_STAMP(10);
                    if (sgi + 1 < nseg && lane == 0) {   // every MMA that reads this segment's query tile has been issued: free it
                        if constexpr (PAIR) umma_commit_pair(q_empty);
                        else umma_commit(q_empty);
                    }
                    __syncwarp();
                }
            }
            if (lane == 0) K2_STAMP(3);
        }
        __syncwarp();
    } else if (warp == 3) {
        // ===================== bias loader =====================
        int gt = 0;
#pragma unroll 1
        for (int sgi = 0; sgi < nseg; sgi++) {   // (never unrolled: two copies of the loops below thrash the instruction cache)
            SegIter it = seg_iter(sgi);
            for (int64_t dbt; (dbt = it.next()) >= 0; gt++) {
                const int acc = gt & 1;
                const uint32_t acc_phase = (gt >> 1) & 1;
                mbar_wait(PAIR ? &bias_empty[acc] : &tmem_empty[acc], acc_phase ^ 1);
                const int64_t row0 = dbt * BN;
#pragma unroll
                for (int j = 0; j < BN / 32; j++) {
                    const int64_t row = row0 + j * 32 + lane;
                    float b = __int_as_float(0x7f800000);  // +inf: rows past the end never pass the threshold
                    if (row < n) b = __ldg(norms + row);  // L2: |x~'|^2; IP: -mu.x (0 without centring)
                    bias[acc * BN + j * 32 + lane] = b;
                }
                if (lane == 0) tile_row0[acc] = (int32_t)row0;   // the epilogue takes the tile's first row from here
                __syncwarp();
                if (lane == 0) mbar_arrive(&bias_full[acc]);
            }
        }
    } else if (warp >= 4) {
        // ===================== epilogue: fused distance + top-k' =====================
        const int ew = warp - 4;                      // epilogue warp index
        const int wq = ew & 3;                        // TMEM lane quarter this warp may access (= warp % 4)
        const int half = ew >> 2;                     // which COLS-wide slice of every tile this warp examines
        const int tid = wq * 32 + lane;               // 0..127 == TMEM lane == query row in the tile
        const uint32_t lane_taddr = tmem_base + ((uint32_t)(wq * 32) << 16);

        // Hot loop (both modes): 32 accumulator columns per tcgen05.ld; per value one FFMA + one compare +
        // one predicated OR into one of four partial bit masks (four short dependency chains instead of
        // one 32-long one).  Survivors are rare, so the cold path is a warp-uniform loop over the union of
        // the lanes' masks; the needed accumulator is picked out of the registers by a 32-way switch --
        // nothing is unrolled 32x, which keeps the epilogue inside the instruction cache (ncu: the unrolled
        // version stalled 46% of issue slots on no_instruction).
        auto chunk_mask = [&](const uint32_t (&r)[32], const float* tbc, float thr) -> uint32_t {
            uint32_t m0 = 0, m1 = 0, m2 = 0, m3 = 0;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const float sdot = __uint_as_float(r[j + u]);
                    const float key = L2 ? fmaf(-2.f, sdot, tbc[j + u]) : tbc[j + u] - sdot;
                    const bool pass = LIST ? (key <= thr) : (key < thr);
                    if (u == 0) { if (pass) m0 |= 1u << (j + u); }
                    else if (u == 1) { if (pass) m1 |= 1u << (j + u); }
                    else if (u == 2) { if (pass) m2 |= 1u << (j + u); }
                    else { if (pass) m3 |= 1u << (j + u); }
                }
            }
            return (m0 | m1) | (m2 | m3);
        };
        auto pick = [](const uint32_t (&r)[32], int j) -> uint32_t {  // j is warp-uniform: a branch table, no memory
            uint32_t v = 0;
            switch (j) {
#define B2F_PICK(i) case i: v = r[i]; break;
                B2F_PICK(0) B2F_PICK(1) B2F_PICK(2) B2F_PICK(3) B2F_PICK(4) B2F_PICK(5) B2F_PICK(6) B2F_PICK(7)
                B2F_PICK(8) B2F_PICK(9) B2F_PICK(10) B2F_PICK(11) B2F_PICK(12) B2F_PICK(13) B2F_PICK(14) B2F_PICK(15)
                B2F_PICK(16) B2F_PICK(17) B2F_PICK(18) B2F_PICK(19) B2F_PICK(20) B2F_PICK(21) B2F_PICK(22) B2F_PICK(23)
                B2F_PICK(24) B2F_PICK(25) B2F_PICK(26) B2F_PICK(27) B2F_PICK(28) B2F_PICK(29) B2F_PICK(30) B2F_PICK(31)
#undef B2F_PICK
            }
            return v;
        };

        if constexpr (LIST) {
            // ---- LIST mode: shared cross-segment threshold + append-only candidate lists ----------------
            // Every (segment, column half) pair of a query tile is a "virtual split" with its own list; the
            // virtual splits of the tile's voucher segments also publish their j-th best so far.
            const float kInf = __int_as_float(0x7f800000);
            uint32_t* xpose = reinterpret_cast<uint32_t*>(smem + L::xpose_off) + ew * 1024;  // this warp's staging area
            const int64_t gstride = (int64_t)nq_tiles * BM;
            int gt = 0;   // tiles so far (accumulator / barrier phases run on across segments)
#pragma unroll 1
#pragma unroll 1
        for (int sgi = 0; sgi < nseg; sgi++) {   // (never unrolled: two copies of the loops below thrash the instruction cache)
            const Seg sg = seg_of(sgi);
            const int qrow = seg_qt(sgi) * BM + tid;
            const bool active = qrow < nq;
            const int vsplit = sg.slot * HALVES + half;
            const int nvs = sg.nv * HALVES;          // voucher virtual splits of this query tile
            const bool voucher = sg.slot < sg.nv;
            const int jv = sg.j;   // rows this list vouches for (vouchers)
            const int gv = sg.g;   // voucher lists consulted: together they vouch for >= k' rows
            const int vstart = voucher ? vsplit : vsplit % nvs;   // own value first; the others spread over the vouchers
            float best[JSLOTS];  // ascending; the first JSLOTS - j slots are pinned at -inf, so best[JSLOTS-1] = j-th best
#pragma unroll
            for (int i = 0; i < JSLOTS; i++) best[i] = (i < JSLOTS - jv) ? -kInf : kInf;
            float thr = 3.0e38f, pub = kInf;  // refreshed before the first compare; never +inf (padding rows have key +inf)
            // range pass (second tensor pass over queries the first could not certify): the threshold is FIXED per query --
            // every true top-k row has a coarse key at or below it (launch_range_thresholds) -- so the lists end up holding
            // every such row; nothing is published, consulted or pruned
            const bool ranged = la.range_thr != nullptr;
            if (ranged) thr = active ? la.range_thr[qrow] : -kInf;
            int cnt = 0;
            uint2* mylist = la.cand + ((int64_t)(active ? qrow : 0) * la.nl_stride + vsplit) * la.cap;
            // shared thresholds are laid out [virtual split][query] so that a warp's loads for one split coalesce
            float* gq = la.shared_thr + (active ? qrow : 0);
            // The refresh sits on the epilogue's critical path (~24 times per stream; the epilogue is what the tile period
            // waits for), and its cost is L2 round trips: `wide` keeps 32 loads in flight -- one round trip for g <= 32 --
            // where no accumulators are live (top of the tile loop, end of the segment); inside a tile 16.
            auto refresh = [&](bool wide) {
                if (ranged) return;
                if (voucher && best[JSLOTS - 1] < pub) {
                    pub = best[JSLOTS - 1];
                    __stcg(gq + (int64_t)vsplit * gstride, pub);
                }
                float t0 = -kInf;
                if (wide) {
#pragma unroll 1
                    for (int i0 = 0; i0 < gv; i0 += 32) {
                        float v[32];
#pragma unroll
                        for (int u = 0; u < 32; u++) {
                            int s2 = vstart + i0 + u;
                            if (s2 >= nvs) s2 -= nvs;
                            v[u] = (i0 + u < gv) ? __ldcg(gq + (int64_t)s2 * gstride) : -kInf;
                        }
#pragma unroll
                        for (int u = 0; u < 32; u++) t0 = fmaxf(t0, v[u]);
                    }
                } else {
#pragma unroll 1
                    for (int i0 = 0; i0 < gv; i0 += 16) {  // 16 independent L2 loads in flight
                        float v[16];
#pragma unroll
                        for (int u = 0; u < 16; u++) {
                            int s2 = vstart + i0 + u;
                            if (s2 >= nvs) s2 -= nvs;
                            v[u] = (i0 + u < gv) ? __ldcg(gq + (int64_t)s2 * gstride) : -kInf;
                        }
#pragma unroll
                        for (int u = 0; u < 16; u++) t0 = fmaxf(t0, v[u]);
                    }
                }
                thr = t0;
            };
            auto process = [&](const uint32_t (&r)[32], bool do_refresh, bool first_wait, const float* tbc, int32_t rowc) {
                // refresh schedule (the caller's rmask): thresholds move like 1/rows_seen, so consult the other splits
                // often at the start and rarely later (from the third tile on the refresh happens at the top of the tile
                // loop, while the thread would otherwise wait for the MMAs of the tile -- see below)
                if (active && do_refresh) {
                    refresh(false);
                    if (first_wait) {   // second chunk of the segment's first tile
                        // Every first-wave virtual split has now seen 32 rows and published.  CTAs start a few
                        // microseconds apart; wait (bounded -- never a hard dependency) for the slowest of
                        // the vouchers we consult instead of appending blindly into the list meanwhile.
                        for (int spin = 0; spin < 64 && thr > 1.0e38f; spin++) {
                            __nanosleep(256);
                            refresh(false);
                        }
                    }
                }
                const uint32_t mask = active ? chunk_mask(r, tbc, thr) : 0u;
                // Survivors are rare.  When some lane of the warp has one, every lane parks its 32 accumulators
                // in the warp's shared-memory staging area ([column][lane]: conflict free) and then walks ITS OWN
                // survivors, all lanes in parallel.  (The previous version walked the union of the lanes'
                // survivors in a warp-uniform loop that picked the accumulator out of the registers with a
                // branch table: ~440 cycles per survivor on a lone warp -- clock64 instrumentation showed it
                // was half of the kernel time at nq = 32 and a quarter at nq = 1024.)
                if (__any_sync(kFull, mask != 0u)) {
                    // park: lane-major rows of 32 words, written as eight 16-byte stores whose chunk index is
                    // XOR-swizzled with the lane so that every quarter-warp covers all 32 banks (8 store
                    // instructions instead of 32; the tile period is set by the slowest of the pair's 16 epilogue
                    // warps, i.e. by these events)
                    uint32_t* st = xpose + lane * 32;
#pragma unroll
                    for (int c4 = 0; c4 < 8; c4++)
                        *reinterpret_cast<uint4*>(st + ((c4 ^ (lane & 7)) << 2)) = make_uint4(r[4 * c4], r[4 * c4 + 1], r[4 * c4 + 2], r[4 * c4 + 3]);
                    uint32_t m = mask;
                    while (m) {
                        const int j = __ffs(m) - 1;
                        m &= m - 1;
                        const float sdot = __uint_as_float(st[((((j >> 2) ^ (lane & 7)) << 2)) + (j & 3)]);
                        const float key = L2 ? fmaf(-2.f, sdot, tbc[j]) : tbc[j] - sdot;
                        if (cnt < la.cap) mylist[cnt] = make_uint2(__float_as_uint(key), (uint32_t)(rowc + j));
                        cnt++;
                        if (jv == 1) {
                            best[JSLOTS - 1] = fminf(best[JSLOTS - 1], key);  // one row per virtual split: a running minimum
                        } else if (key < best[JSLOTS - 1]) {
                            // sorted insert without a dependency chain: new[i] = max(old[i-1], min(old[i], key))
                            float nb[JSLOTS];
#pragma unroll
                            for (int i = 0; i < JSLOTS; i++) nb[i] = fmaxf(i > 0 ? best[i - 1] : -kInf, fminf(best[i], key));
#pragma unroll
                            for (int i = 0; i < JSLOTS; i++) best[i] = nb[i];
                        }
                    }
                }
            };
            const int seg_tiles = seg_tiles_of(sgi);   // (host-computed with SegIter: no iterator in this role)
#pragma unroll 1
            for (int t = 0; t < seg_tiles; t++, gt++) {   // t: tile index within the segment (refresh schedule)
                const int acc = gt & 1;
                const uint32_t acc_phase = (gt >> 1) & 1;
                // Scheduled refresh of the shared threshold BEFORE waiting for the tile's accumulator: the ~1.4 us
                // of L2 round trips overlap the MMAs the thread would wait for anyway, and no accumulator registers
                // are live yet (same-box A/B: the refreshes inside the tile cost 3-4% of the kernel).  After the first 32
                // tiles, every 32nd (same-box A/B over periods 4..128: 32 is the flat optimum, profiles/r01_j_ab_refresh.txt).
                if (active && t >= 2 && (t < 8 || (t < 32 && (t & 3) == 0) || (t & 31) == 0)) refresh(true);
                // which chunks of this tile start with a refresh: all of tile 0, every other one of tile 1
                const uint32_t rmask = t == 0 ? 0xffffffffu : (t == 1 ? 0x55555555u : 0u);
                mbar_wait(&bias_full[acc], acc_phase);
                mbar_wait(&tmem_full[acc], acc_phase);
                tc_fence_after();
                const int32_t row0 = tile_row0[acc] + half * COLS;
                const float* tb = bias + acc * BN + half * COLS;
                const uint32_t tile_taddr = lane_taddr + (uint32_t)(acc * BN + half * COLS);
                uint32_t ra[32], rb[32];
                tmem_ld32(tile_taddr, ra);
#pragma unroll 1
                for (int c = 0; c < COLS / 32; c += 2) {
                    tmem_ld_wait();
                    tmem_ld32(tile_taddr + (uint32_t)((c + 1) * 32), rb);
                    process(ra, ((rmask >> c) & 1u) != 0u, false, tb + c * 32, row0 + c * 32);
                    tmem_ld_wait();
                    if (c + 2 < COLS / 32) tmem_ld32(tile_taddr + (uint32_t)((c + 2) * 32), ra);
                    process(rb, ((rmask >> (c + 1)) & 1u) != 0u, t == 0 && c == 0, tb + (c + 1) * 32, row0 + (c + 1) * 32);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if constexpr (PAIR) {
                        mbar_arrive(&bias_empty[acc]);             // this CTA's bias buffer is free again
                        mbar_arrive_cluster(&tmem_empty[acc], 0);  // the leader may overwrite both CTAs' accumulators
                    } else {
                        mbar_arrive(&tmem_empty[acc]);
                    }
                }
            }
            if (warp == 4 && lane == 0) K2_STAMP(4);
            if (active) {
                // End-of-segment pruning: the final shared threshold is far tighter than the ones most
                // entries were admitted under (the first chunk is admitted blindly), so re-filter the
                // thread's own list in place.  Shrinks the merge input ~10x (C2: 1460 -> ~100 per query).
                // (tools/k2_trace.py: ~13 us per segment -- a refresh and three or four DEPENDENT round trips through a memory
                // system the other CTAs keep saturated.  Tried and dropped, same-box A/B: requesting the first 32 entries
                // before the refresh in the registers the accumulators no longer need -- the main loop's register allocation
                // paid 2 % of the kernel for it; prefetch.global.L2 of the list lines -- no effect, they are L2 hits already.)
                const int have = cnt <= la.cap ? cnt : 0;  // an overflowed list is left as is (the query falls back)
                refresh(true);
                int w = 0;
#pragma unroll 1
                for (int i0 = 0; i0 < have; i0 += 16) {
                    uint2 e[16];
#pragma unroll
                    for (int u = 0; u < 16; u++) e[u] = (i0 + u < have) ? mylist[i0 + u] : make_uint2(0x7f800000u, 0u);
#pragma unroll
                    for (int u = 0; u < 16; u++)
                        if (i0 + u < have && __uint_as_float(e[u].x) <= thr) mylist[w++] = e[u];
                }
                la.counts[(int64_t)qrow * la.nl_stride + vsplit] = cnt > la.cap ? cnt : w;  // > cap marks an overflow
                // every row of this virtual split with key <= thr is in the list: the merge certifies against the
                // smallest of these over the query's lists
                la.final_thr[(int64_t)qrow * la.nl_stride + vsplit] = thr;
            }
            if (warp == 4 && lane == 0) K2_STAMP(5);
            }  // segments
        } else {
            // ---- HEAP mode: thread-private max-heap of k' in shared memory ------------------------------
            const int qrow = seg[0].qtile * BM + tid;
            const bool active = qrow < nq;
            for (int j = 0; j < KP; j++) {
                heap_k[j * EPI_THREADS + tid] = FLT_MAX;
                heap_i[j * EPI_THREADS + tid] = -1;
            }
            float thr = FLT_MAX;
            const int heap_tiles = seg_tiles_of(0);
            for (int t = 0; t < heap_tiles; t++) {
                const int acc = t & 1;
                const uint32_t acc_phase = (t >> 1) & 1;
                mbar_wait(&bias_full[acc], acc_phase);
                mbar_wait(&tmem_full[acc], acc_phase);
                tc_fence_after();
                const int32_t row0 = tile_row0[acc];
                const float* tb = bias + acc * BN;
                const uint32_t tile_taddr = lane_taddr + (uint32_t)(acc * BN);
#pragma unroll 1
                for (int c = 0; c < BN / 32; c++) {
                    uint32_t r[32];
                    tmem_ld32(tile_taddr + (uint32_t)(c * 32), r);
                    tmem_ld_wait();
                    const float* tbc = tb + c * 32;
                    const uint32_t mask = active ? chunk_mask(r, tbc, thr) : 0u;
                    uint32_t um = __reduce_or_sync(kFull, mask);
                    while (um) {
                        const int j = __ffs(um) - 1;
                        um &= um - 1;
                        const uint32_t v = pick(r, j);
                        if (mask & (1u << j)) {
                            const float sdot = __uint_as_float(v);
                            const float key = L2 ? fmaf(-2.f, sdot, tbc[j]) : tbc[j] - sdot;
                            // the mask was computed with the threshold of the chunk start: re-test
                            if (key < thr) thr = heap_push<KP>(heap_k, heap_i, tid, key, row0 + c * 32 + j);
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            }
            // heap sort (ascending) and write the partial list of (query, split)
            if (active) {
                for (int m = KP - 1; m > 0; m--) {
                    const float lk_ = heap_k[m * EPI_THREADS + tid];
                    const int32_t li_ = heap_i[m * EPI_THREADS + tid];
                    heap_k[m * EPI_THREADS + tid] = heap_k[tid];
                    heap_i[m * EPI_THREADS + tid] = heap_i[tid];
                    heap_sift_down_n<KP>(heap_k, heap_i, tid, m, lk_, li_);
                }
                float* ok = pk + ((int64_t)qrow * nsplits + split) * KP;
                int32_t* oi = pi + ((int64_t)qrow * nsplits + split) * KP;
                for (int j = 0; j < KP; j++) {
                    ok[j] = heap_k[j * EPI_THREADS + tid];
                    oi[j] = heap_i[j * EPI_THREADS + tid];
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();  // neither CTA may free TMEM / exit while the other still uses the pair
    if (threadIdx.x == 0) K2_STAMP(6);
    if (warp == 2) {
        tc_fence_after();
        if constexpr (PAIR)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
        if (lane == 0) K2_STAMP(7);
    }
}

// ---- K3b + K4: per query, merge the candidate lists, re-rank exactly, certify, write (D, I) ---------------
// One CTA per query.  Candidates become 64-bit composites (order-preserving key bits << 32 | row id) in
// shared memory.  Up to RANK_MAX entries (the usual case after end-of-stream pruning) they are ranked
// directly -- each element counts the composites below it and lands on its sorted slot; beyond that the
// k'-th smallest is found by bisection (first over the 32 key bits, then, only when equal keys straddle the
// cut, over the 32 id bits).  The k' best are re-ranked in exact fp32 arithmetic and certified against the
// k'-th coarse key (rerank.cuh).
//
// Extended certification.  Thresholds only ever fall, so the lists hold EVERY row whose coarse key is <= T_c,
// the smallest threshold any of the query's lists was finally pruned against -- typically 2-4x more rows than
// k'.  When the k' best do not certify, all list entries are re-ranked and the bound becomes T_c: the query is
// answered exactly from rows the tensor pass already found, without another pass over the database.
constexpr int MERGE_THREADS = kRerankThreads;  // 256
constexpr int MERGE_MAX = 4096;   // composites held in shared memory (32 KB) at most; more -> the query falls back
constexpr int RANK_MAX = 1024;    // direct ranking and extended certification up to this many list entries
constexpr int KP_MAX = 256;
static_assert(MERGE_MAX == kRangeHitsMax, "range search stages as many entries per query as the merge holds");

__device__ __forceinline__ int block_count_le(const unsigned long long* comp, int M, unsigned long long bound, int* s_cnt,
                                              int it, int tid, int lane) {
    if (tid == 0) s_cnt[(it + 1) % 3] = 0;  // for the next step
    int c = 0;
    for (int i = tid; i < M; i += MERGE_THREADS) c += comp[i] <= bound ? 1 : 0;
    c = __reduce_add_sync(kFull, c);
    if (lane == 0 && c) atomicAdd(&s_cnt[it % 3], c);
    __syncthreads();
    return s_cnt[it % 3];
}

// One step of the 8-bit radix select after the 256-bin histogram is filled: block-wide inclusive scan (warp scans +
// the 8 warp totals), the bin holding the `need`-th element extends `lo`, `need` becomes the rank inside that bin.
__device__ __forceinline__ void radix_pick(int* s_hist, int* s_wsum, int* s_sel, int shift, unsigned int& lo, int& need,
                                           int tid, int lane, int warp) {
    __syncthreads();
    const int h = s_hist[tid];
    int incl = h;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int up = __shfl_up_sync(kFull, incl, d);
        if (lane >= d) incl += up;
    }
    if (lane == 31) s_wsum[warp] = incl;
    __syncthreads();
    int base = 0;
    for (int w = 0; w < warp; w++) base += s_wsum[w];
    incl += base;
    if (incl >= need && incl - h < need) {  // exactly one bin
        s_sel[0] = tid;
        s_sel[1] = need - (incl - h);
    }
    __syncthreads();
    lo |= (unsigned int)s_sel[0] << shift;
    need = s_sel[1];
    __syncthreads();
}

// (register-limited to four CTAs per SM; forcing five or six with launch bounds was measured: no gain, the spills cost what
// the extra CTAs bring)
__global__ void __launch_bounds__(MERGE_THREADS)
merge_lists_kernel(const uint2* __restrict__ cand, const int32_t* __restrict__ counts, const float* __restrict__ final_thr,
                   int nl_stride, int tile_queries, int ntile_units, int total_units, int halves, int kp, int list_cap,
                   int cap_entries, unsigned long long* __restrict__ total_entries, const uint8_t* __restrict__ only_flagged,
                   const RerankArgs ra) {
    extern __shared__ __align__(16) unsigned long long comp[];  // [max(cap_entries, RANK_MAX)], later the re-rank scratch
    if (only_flagged && !only_flagged[blockIdx.x]) return;   // big batches: the warp-per-query kernel answered this query
    __shared__ int s_off[2 * kNumSMs + 2];
    __shared__ int s_cnt[3];
    __shared__ int s_nsurv, s_nrest;
    __shared__ int s_hist[MERGE_THREADS], s_wsum[MERGE_THREADS / 32], s_sel[2];
    __shared__ int s_ovf;
    __shared__ unsigned int s_tc_enc;
    const int cap_c = cap_entries > RANK_MAX ? cap_entries : RANK_MAX;
    unsigned long long* surv = comp + cap_c;                       // [KP_MAX]
    float* sk = reinterpret_cast<float*>(surv + KP_MAX);           // [RANK_MAX] coarse keys, ascending
    int32_t* si = reinterpret_cast<int32_t*>(sk + RANK_MAX);       // [RANK_MAX]
    unsigned short* owner = reinterpret_cast<unsigned short*>(si + RANK_MAX);  // [cap_entries] list of every gathered entry
    float* ek = reinterpret_cast<float*>(comp);                    // [RANK_MAX] exact keys   (comp is dead by then)
    int32_t* ei = reinterpret_cast<int32_t*>(ek + RANK_MAX);       // [RANK_MAX]
    const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tile = q / tile_queries;
    int nsplits;   // lists of this query = (pieces of its tile: first wave + second wave, see Seg) x column halves
    {
        const TileInfo ti = tile_info(tile, ntile_units, total_units, 0, halves);
        nsplits = (ti.nfw + ti.nsw) * halves;
    }
    // list lengths and final thresholds: one parallel sweep (up to 296 lists), then a warp-level prefix sum
    if (tid == 0) {
        s_tc_enc = 0xffffffffu;
        s_ovf = 0;
        s_nsurv = 0;
        s_nrest = 0;
        s_cnt[0] = 0;
    }
    __syncthreads();
    {
        float tc = 3.0e38f;
        int o = 0;
        for (int s2 = tid; s2 < nsplits; s2 += MERGE_THREADS) {
            int c = counts[(int64_t)q * nl_stride + s2];
            tc = fminf(tc, final_thr[(int64_t)q * nl_stride + s2]);
            if (c > list_cap) {
                c = list_cap;
                o = 1;
            }
            s_off[s2 + 1] = c;
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) tc = fminf(tc, __shfl_xor_sync(kFull, tc, d));
        o = __reduce_or_sync(kFull, o);
        if (lane == 0) {
            atomicMin(&s_tc_enc, enc_key(tc));
            if (o) s_ovf = 1;
        }
    }
    __syncthreads();
    if (warp == 0) {
        int run = 0;
        for (int s0 = 0; s0 < nsplits; s0 += 32) {
            const int s2 = s0 + lane;
            const int c = s2 < nsplits ? s_off[s2 + 1] : 0;
            int incl = c;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int up = __shfl_up_sync(kFull, incl, d);
                if (lane >= d) incl += up;
            }
            __syncwarp();
            if (s2 < nsplits) s_off[s2 + 1] = run + incl;  // s_off[s] = entries before list s; s_off[nsplits] = total
            run += __shfl_sync(kFull, incl, 31);
        }
        if (lane == 0) {
            s_off[0] = 0;
            if (total_entries) atomicAdd(total_entries, (unsigned long long)run);
            if (run > cap_entries && (ra.range || !ra.certify)) s_ovf = 1;
        }
    }
    __syncthreads();
    if (ra.out_map && ra.out_map[q] < 0) return;   // range pass: an unused slot of the compacted batch
    if (s_ovf) {
        // some candidates were dropped: only the exact scan can answer (it rewrites this query's D / I rows)
        if (tid == 0) rerank_record_failure(ra, q, true);
        return;
    }
    int M = s_off[nsplits];
    // More entries than the merge holds in shared memory, none dropped (thresholds that never tightened: e.g. a
    // query whose best rows all sit in one or two lists because near-duplicates are stored next to each other).
    // The k' best are still in the lists: find the k'-th coarse key K by the same radix select run over the lists in
    // global memory, keep the entries with keys <= K and go on with those.  Such a query seldom certifies -- but
    // it fails WITH its exact k-th distance, which is what the range pass needs to answer it without the exact scan.
    const bool big = M > cap_entries;
    if (big) {
        unsigned int lo = 0;
        int need = kp;
#pragma unroll 1
        for (int pass = 0; pass < 4; pass++) {
            const int shift = 24 - 8 * pass;
            s_hist[tid] = 0;
            __syncthreads();
#pragma unroll 1
            for (int l = 0; l < nsplits; l++) {
                const int c = s_off[l + 1] - s_off[l];
                const uint2* p = cand + ((int64_t)q * nl_stride + l) * list_cap;
                for (int j0 = 0; j0 < c; j0 += MERGE_THREADS) {
                    const int j = j0 + tid;
                    const unsigned int key = j < c ? enc_key(__uint_as_float(p[j].x)) : 0u;
                    const bool in = j < c && (pass == 0 || (key >> (shift + 8)) == (lo >> (shift + 8)));
                    const unsigned int bin = (key >> shift) & 255u;
                    const unsigned int peers = __match_any_sync(kFull, in ? bin : 256u + (unsigned)lane);
                    if (in && lane == __ffs(peers) - 1) atomicAdd(&s_hist[bin], __popc(peers));
                }
            }
            radix_pick(s_hist, s_wsum, s_sel, shift, lo, need, tid, lane, warp);
        }
#pragma unroll 1
        for (int l = 0; l < nsplits; l++) {
            const int c = s_off[l + 1] - s_off[l];
            const uint2* p = cand + ((int64_t)q * nl_stride + l) * list_cap;
            for (int j = tid; j < c; j += MERGE_THREADS) {
                const uint2 e = p[j];
                const unsigned int key = enc_key(__uint_as_float(e.x));
                if (key <= lo) {
                    const int slot = atomicAdd(&s_nrest, 1);
                    if (slot < cap_entries) comp[slot] = ((unsigned long long)key << 32) | (unsigned long long)e.y;
                }
            }
        }
        __syncthreads();
        M = s_nrest;   // >= k'
        __syncthreads();
        if (tid == 0) s_nrest = 0;
        if (M > cap_entries) {   // that many equal keys: give up
            if (tid == 0) rerank_record_failure(ra, q, true);
            return;
        }
        __syncthreads();
    } else {
    // gather the lists into one array of composites: flattened over all candidates so every thread has independent
    // loads in flight; the owning list of element i comes from a map filled by one thread per list
    for (int l = tid; l < nsplits; l += MERGE_THREADS) {
        const int o = s_off[l], e = s_off[l + 1];
        for (int i = o; i < e; i++) owner[i] = (unsigned short)l;
    }
    __syncthreads();
    for (int i0 = tid; i0 < M; i0 += 4 * MERGE_THREADS) {
        uint2 e[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = i0 + u * MERGE_THREADS;
            e[u] = make_uint2(0u, 0u);
            if (i < M) {
                const int l = owner[i];
                e[u] = cand[((int64_t)q * nl_stride + l) * list_cap + (i - s_off[l])];
            }
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int i = i0 + u * MERGE_THREADS;
            if (i < M) comp[i] = ((unsigned long long)enc_key(__uint_as_float(e[u].x)) << 32) | (unsigned long long)e[u].y;
        }
    }
    }
    __syncthreads();
    // Selection.  sk / si [0, min(k', M)): the k' best, ascending; [k', M) (when M <= RANK_MAX): the other list
    // entries in no particular order -- only the extended certification looks at them.
    if (M <= MERGE_THREADS) {
        // one element per thread: count the composites below it (distinct: row ids) and land on the sorted slot
        if (tid < M) {
            const unsigned long long mine = comp[tid];
            int rank = 0;
            for (int j = 0; j < M; j++) rank += comp[j] < mine ? 1 : 0;
            sk[rank] = dec_key((uint32_t)(mine >> 32));
            si[rank] = (int32_t)(uint32_t)(mine & 0xffffffffu);
        }
    } else {
        unsigned long long T = ~0ull;
        int it = 0;
        // K = key of the k'-th smallest composite: radix select over the 32 key bits, 8 bits per pass (256-bin
        // histogram in shared memory, warp-aggregated increments, block-wide scan) -- 4 passes instead of 32
        // bisection steps
        unsigned int lo = 0;
        int need = kp;
#pragma unroll 1
        for (int pass = 0; pass < 4; pass++) {
            const int shift = 24 - 8 * pass;
            s_hist[tid] = 0;  // MERGE_THREADS == 256 bins
            __syncthreads();
            for (int i0 = 0; i0 < M; i0 += MERGE_THREADS) {
                const int i = i0 + tid;
                const unsigned int key = i < M ? (unsigned int)(comp[i] >> 32) : 0u;
                const bool in = i < M && (pass == 0 || (key >> (shift + 8)) == (lo >> (shift + 8)));
                const unsigned int bin = (key >> shift) & 255u;
                const unsigned int peers = __match_any_sync(kFull, in ? bin : 256u + (unsigned)lane);
                if (in && lane == __ffs(peers) - 1) atomicAdd(&s_hist[bin], __popc(peers));
            }
            radix_pick(s_hist, s_wsum, s_sel, shift, lo, need, tid, lane, warp);
        }
        const unsigned long long kbits = (unsigned long long)lo << 32;
        T = kbits | 0xffffffffull;
        if (block_count_le(comp, M, T, s_cnt, it++, tid, lane) > kp) {
            // equal keys straddle the cut: take the lowest ids among them
            unsigned int ilo = 0, ihi = 0xffffffffu;
            while (ilo < ihi) {
                const unsigned int mid = ilo + ((ihi - ilo) >> 1);
                const int total = block_count_le(comp, M, kbits | mid, s_cnt, it++, tid, lane);
                if (total >= kp) ihi = mid;
                else ilo = mid + 1;
            }
            T = kbits | ilo;
        }
        for (int i = tid; i < M; i += MERGE_THREADS) {
            const unsigned long long v = comp[i];
            if (v <= T) {
                const int slot = atomicAdd(&s_nsurv, 1);
                if (slot < kp) surv[slot] = v;
            } else if (M <= RANK_MAX) {
                const int slot = kp + atomicAdd(&s_nrest, 1);
                if (slot < RANK_MAX) {
                    sk[slot] = dec_key((uint32_t)(v >> 32));
                    si[slot] = (int32_t)(uint32_t)(v & 0xffffffffu);
                }
            }
        }
        __syncthreads();
        const int ns = s_nsurv < kp ? s_nsurv : kp;   // == kp (composites are distinct and M > kp)
        for (int t = tid; t < ns; t += MERGE_THREADS) {
            const unsigned long long mine = surv[t];
            int rank = 0;
            for (int j = 0; j < ns; j++) rank += surv[j] < mine ? 1 : 0;
            sk[rank] = dec_key((uint32_t)(mine >> 32));
            si[rank] = (int32_t)(uint32_t)(mine & 0xffffffffu);
        }
    }
    __syncthreads();
    // K4: exact fp32 re-rank of the k' best + certification + faiss-formatted output
    const float tc = dec_key(s_tc_enc);
    const int nc1 = M < kp ? M : kp;
    const float bound1 = (M > kp || big) ? fminf(sk[kp - 1], tc) : tc;   // big: rows beyond the kept entries have keys >= sk[k' - 1]
    __shared__ float s_tau_last;   // exact k-th key of the last re-rank (what a failed query hands to the range pass)
    bool cert = false;
    if (ra.range) {
        // range pass: the lists hold every row whose coarse key is <= the query's fixed threshold (= tc), among them
        // every true top-k row: re-rank them all; certification against tc holds by construction of the threshold
        if (M <= RANK_MAX) cert = rerank_block(ra, q, sk, si, M, tc, false, ek, ei, &s_tau_last);
        else if (tid == 0) s_tau_last = FLT_MAX;
    } else {
        cert = rerank_block(ra, q, sk, si, nc1, bound1, M < kp, ek, ei, &s_tau_last);
        if (!cert && ra.certify && !big && M > kp && M <= RANK_MAX) {
            // every list entry: rows outside the lists have coarse keys above T_c
            cert = rerank_block(ra, q, sk, si, M, tc, false, ek, ei, &s_tau_last);
            if (tid == 0 && cert) atomicAdd(ra.fail_count + 4, 1);  // diagnostics: queries rescued by the extended pass
        }
    }
    if (tid == 0 && ra.certify && !cert) rerank_record_failure(ra, q, false, s_tau_last);
}

// ---- K3b + K4 for big batches: one WARP per query ---------------------------------------------------------
// The block kernel above is a chain of dependent steps per query (~10 us) with five CTAs resident per SM: fine for a
// thousand queries (one wave), but 8192 queries (the N = 8 weak-scaling shape) are eleven waves of it.  After the
// end-of-stream pruning a query of a big batch has ~80 list entries, so one warp can do everything a CTA does: 64
// queries in flight per SM instead of five.  Queries it cannot hold (more than WM_MAX entries, an overflowed list)
// are flagged and answered by the block kernel launched right behind (it skips unflagged queries).  Measured gain:
// 8 % of the merge at 8192 queries, a loss below that -- it is used from 8192 queries up (same-box A/B, r02n: 8192
// queries 125 -> 114 us, 4096 queries 78 -> 82 us, 1024 queries 47 -> 73 us).
constexpr int WM_WARPS = 8;      // queries per CTA
constexpr int WM_MIN_NQ = 8192;  // batch size from which the warp kernel runs first
constexpr int WM_MAX = 128;      // list entries per query
constexpr int WM_LISTS = 64;     // lists per query

// Exact re-rank of the first nc candidates (sk / si: coarse keys ascending) by one warp; writes the best k in faiss
// conventions, returns whether the result is certified (warp-uniform).  ek / ei: nc floats / ints of scratch.
__device__ __forceinline__ bool warp_rerank(const RerankArgs& a, int q, const float* sk, const int32_t* si, int nc, float bound,
                                            bool all_rows, float* ek, int32_t* ei, int lane, float& tau_out) {
    const float* qv = a.q + (int64_t)q * a.d;
    const bool l2 = a.metric == B2F_METRIC_L2;
    const int sl = lane & 7;
    for (int c0 = 0; c0 < nc; c0 += 4) {   // 8 lanes per candidate, 4 candidates per pass
        const int c = c0 + (lane >> 3);
        int32_t id = c < nc ? si[c] : -1;
        if ((int64_t)id >= a.ntotal) id = -1;
        const float key = exact_key_8lanes(a, qv, id, sl, l2);
        if (sl == 0 && c < nc) {
            const bool ok = id >= 0 && !(key != key);
            ek[c] = ok ? key : FLT_MAX;
            ei[c] = ok ? id : -1;
        }
    }
    __syncwarp();
    float tau = FLT_MAX;
    for (int t = lane; t < nc; t += 32) {
        const float mk = ek[t];
        const int32_t mi = ei[t];
        int rank = 0;
        for (int j = 0; j < nc; j++) {
            const float ok_ = ek[j];
            const int32_t oi_ = ei[j];
            rank += (cand_less(ok_, oi_, mk, mi) || (ok_ == mk && oi_ == mi && j < t)) ? 1 : 0;
        }
        if (rank < a.k) {
            const int64_t o = (int64_t)q * a.k + rank;
            a.D[o] = mi < 0 ? (l2 ? FLT_MAX : -FLT_MAX) : (l2 ? mk : -mk);
            a.I[o] = mi < 0 ? -1 : (int64_t)mi + a.id_offset;
        }
        if (rank == a.k - 1) tau = mk;
    }
    for (int t = nc + lane; t < a.k; t += 32) {   // fewer candidates than k: pad
        a.D[(int64_t)q * a.k + t] = l2 ? FLT_MAX : -FLT_MAX;
        a.I[(int64_t)q * a.k + t] = -1;
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) tau = fminf(tau, __shfl_xor_sync(kFull, tau, d));   // exactly one lane holds the k-th key
    __syncwarp();
    tau_out = tau;
    return all_rows || rerank_certified(a, q, tau, bound);
}

__global__ void __launch_bounds__(WM_WARPS * 32)
merge_lists_warp_kernel(const uint2* __restrict__ cand, const int32_t* __restrict__ counts, const float* __restrict__ final_thr,
                        int nl_stride, int tile_queries, int ntile_units, int total_units, int halves, int kp, int list_cap,
                        unsigned long long* __restrict__ total_entries, uint8_t* __restrict__ big_flag, int nq, const RerankArgs ra) {
    __shared__ __align__(16) unsigned long long s_comp[WM_WARPS][WM_MAX];
    __shared__ float s_sk[WM_WARPS][WM_MAX], s_ek[WM_WARPS][WM_MAX];
    __shared__ int32_t s_si[WM_WARPS][WM_MAX], s_ei[WM_WARPS][WM_MAX];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * WM_WARPS + warp;
    if (q >= nq) return;
    unsigned long long* comp = s_comp[warp];
    float* sk = s_sk[warp];
    int32_t* si = s_si[warp];
    int nlists;
    {
        const TileInfo ti = tile_info(q / tile_queries, ntile_units, total_units, 0, halves);
        nlists = (ti.nfw + ti.nsw) * halves;   // <= WM_LISTS (host-checked)
    }
    // list lengths, final thresholds, offsets: lane l owns lists l and l + 32
    int c0 = 0, c1 = 0;
    float tc = 3.0e38f;
    bool ovf = false;
    if (lane < nlists) {
        c0 = counts[(int64_t)q * nl_stride + lane];
        tc = fminf(tc, final_thr[(int64_t)q * nl_stride + lane]);
    }
    if (lane + 32 < nlists) {
        c1 = counts[(int64_t)q * nl_stride + lane + 32];
        tc = fminf(tc, final_thr[(int64_t)q * nl_stride + lane + 32]);
    }
    ovf = c0 > list_cap || c1 > list_cap;
    int i0 = c0, i1 = c1;   // inclusive scans
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int u0 = __shfl_up_sync(kFull, i0, d), u1 = __shfl_up_sync(kFull, i1, d);
        if (lane >= d) { i0 += u0; i1 += u1; }
    }
    const int tot0 = __shfl_sync(kFull, i0, 31), M = tot0 + __shfl_sync(kFull, i1, 31);
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) tc = fminf(tc, __shfl_xor_sync(kFull, tc, d));
    ovf = __any_sync(kFull, ovf);
    if (lane == 0 && total_entries) atomicAdd(total_entries, (unsigned long long)(ovf ? 0 : M));
    if (ovf || M > WM_MAX) {   // the block kernel answers this one
        if (lane == 0) big_flag[q] = 1;
        return;
    }
    if (lane == 0) big_flag[q] = 0;
    // gather: every lane copies its own (short) lists
    {
        const uint2* l0 = cand + ((int64_t)q * nl_stride + lane) * list_cap;
        const int o0 = i0 - c0;
        for (int i = 0; i < c0; i++) {
            const uint2 e = l0[i];
            comp[o0 + i] = ((unsigned long long)enc_key(__uint_as_float(e.x)) << 32) | (unsigned long long)e.y;
        }
        const uint2* l1 = cand + ((int64_t)q * nl_stride + lane + 32) * list_cap;
        const int o1 = tot0 + i1 - c1;
        for (int i = 0; i < c1; i++) {
            const uint2 e = l1[i];
            comp[o1 + i] = ((unsigned long long)enc_key(__uint_as_float(e.x)) << 32) | (unsigned long long)e.y;
        }
    }
    __syncwarp();
    // full sort by rank counting (composites are distinct: row ids)
    for (int t = lane; t < M; t += 32) {
        const unsigned long long mine = comp[t];
        int rank = 0;
        for (int j = 0; j < M; j++) rank += comp[j] < mine ? 1 : 0;
        sk[rank] = dec_key((uint32_t)(mine >> 32));
        si[rank] = (int32_t)(uint32_t)(mine & 0xffffffffu);
    }
    __syncwarp();
    // exact re-rank + certification: the k' best, then every list entry (see merge_lists_kernel)
    const int nc1 = M < kp ? M : kp;
    const float bound1 = (M > kp) ? fminf(sk[kp - 1], tc) : tc;
    float tau = FLT_MAX;
    bool cert = warp_rerank(ra, q, sk, si, nc1, bound1, M < kp, s_ek[warp], s_ei[warp], lane, tau);
    if (!cert && ra.certify && M > kp) {
        cert = warp_rerank(ra, q, sk, si, M, tc, false, s_ek[warp], s_ei[warp], lane, tau);
        if (lane == 0 && cert) atomicAdd(ra.fail_count + 4, 1);
    }
    if (lane == 0 && ra.certify && !cert) rerank_record_failure(ra, q, false, tau);
}

// ---- host side --------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

static int make_map(CUtensorMap* map, const void* base, uint64_t inner, uint64_t rows, uint64_t pitch_elems, uint32_t box_rows) {
    EncodeTiledFn enc = get_encode();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return B2F_ECUDA;
    }
    cuuint64_t dims[2] = {inner, rows};
    cuuint64_t strides[1] = {pitch_elems * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
        return B2F_ECUDA;
    }
    return B2F_OK;
}

// Database tiles of every (unit, segment) of a LIST plan -- the epilogue's loop counts.  Cached per thread: a serving
// loop repeats the same (tile units, units, round, database) shape, and one evaluation walks units x rounds steps.
static const SegCounts& segment_counts(const TensorScanPlan& plan, int64_t ntiles) {
    struct Key {
        int T, U, R;
        int64_t ntiles;
    };
    static thread_local Key key{-1, -1, -1, -1};
    static thread_local SegCounts sc;
    if (key.T != plan.tile_units || key.U != plan.units || key.R != plan.round_tiles || key.ntiles != ntiles) {
        for (int i = 0; i < 2 * kNumSMs; i++) sc.n[i] = 0;
        for (int u = 0; u < plan.units && u < kNumSMs; u++) {
            Seg seg[2];
            const int nseg = unit_segments(u, plan.tile_units, plan.units, plan.kp, EPI_WARPS_LIST / 4, seg);
            for (int sg = 0; sg < nseg; sg++) {
                SegIter it;
                it.init(seg[sg].p0, seg[sg].p1, plan.units, plan.round_tiles, ntiles);
                sc.n[2 * u + sg] = it.count();
            }
        }
        key = Key{plan.tile_units, plan.units, plan.round_tiles, ntiles};
    }
    return sc;
}

template <int KP, bool L2, bool LIST, bool QRES, bool PAIR = false>
static int launch_k2(const CUtensorMap& mq, const CUtensorMap& mx, const float* norms, int64_t n, int nq, int kblocks,
                     const TensorScanPlan& plan, float* pk, int32_t* pi, const ListArgs& la, cudaStream_t st) {
    auto kern = tensor_scan_kernel<KP, L2, LIST, QRES, PAIR>;
    static const SegCounts no_counts{};
    const SegCounts& sc = LIST ? segment_counts(plan, (n + BN - 1) / BN) : no_counts;
    constexpr size_t smem = Smem < LIST ? 0 : KP, PAIR ? STAGES_PAIR : (QRES ? STAGES_QRES : (LIST ? STAGES_LIST : STAGES_HEAP)),
                     QRES ? QRES_MAX_KB : 0, PAIR > ::alloc;
    static_assert(smem <= 232448, "shared memory budget exceeded");
    {
        static bool configured[kMaxDevices] = {};
        const int dev = current_device_slot();
        std::lock_guard<std::mutex> lk(launch_cache_mutex());
        if (!configured[dev]) {
            B2F_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            configured[dev] = true;
        }
    }
    if constexpr (PAIR) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)(2 * plan.units));  // one cluster of 2 CTAs per unit
        cfg.blockDim = dim3(k2_threads(LIST));
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        B2F_CUDA(cudaLaunchKernelEx(&cfg, kern, mq, mx, norms, n, nq, kblocks, plan.nq_tiles, plan.nsplits, pk, pi, la, sc));
    } else {
        kern<<<plan.units, k2_threads(LIST), smem, st>>>(mq, mx, norms, n, nq, kblocks, plan.nq_tiles, plan.nsplits,
                                                                  pk, pi, la, sc);
    }
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

// ---- range search: filter the lists of a range-threshold pass down to the exact hits -----------------------------------
// One CTA per query.  The pass listed every row whose coarse key is <= thr(tau), a proven superset of the rows whose exact
// key is <= tau.  Each entry's exact key (exact_key_8lanes, as everywhere else) decides; the strict hits are sorted by row
// id (bitonic over (id, key) composites; non-hits are all-ones and sort last) and staged in skey / sid [q][MERGE_MAX].
// A query whose lists overflowed, that has more than MERGE_MAX entries or a NaN threshold goes to scan_list instead.
__global__ void __launch_bounds__(MERGE_THREADS)
range_collect_kernel(const uint2* __restrict__ cand, const int32_t* __restrict__ counts, const float* __restrict__ thr,
                     int nl_stride, int tile_queries, int ntile_units, int total_units, int halves, int list_cap, float tau,
                     const RerankArgs ra, float* __restrict__ skey, int32_t* __restrict__ sid, int32_t* __restrict__ staged,
                     int32_t* __restrict__ count, int32_t* __restrict__ scan_list, int32_t* __restrict__ scan_n) {
    __shared__ unsigned long long comp[MERGE_MAX];
    __shared__ int s_off[2 * kNumSMs + 2];
    __shared__ int s_ovf, s_hits;
    const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const TileInfo ti = tile_info(q / tile_queries, ntile_units, total_units, 0, halves);
    const int nsplits = (ti.nfw + ti.nsw) * halves;
    if (tid == 0) {
        s_ovf = !(thr[q] == thr[q]);
        s_hits = 0;
    }
    __syncthreads();
    for (int s2 = tid; s2 < nsplits; s2 += MERGE_THREADS) {
        const int c = counts[(int64_t)q * nl_stride + s2];
        if (c > list_cap) s_ovf = 1;
        s_off[s2 + 1] = c;
    }
    __syncthreads();
    if (tid < 32) {
        int run = 0;
        for (int s0 = 0; s0 < nsplits; s0 += 32) {
            const int s2 = s0 + lane;
            int incl = s2 < nsplits ? s_off[s2 + 1] : 0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int up = __shfl_up_sync(kFull, incl, d);
                if (lane >= d) incl += up;
            }
            __syncwarp();
            if (s2 < nsplits) s_off[s2 + 1] = run + incl;
            run += __shfl_sync(kFull, incl, 31);
        }
        if (lane == 0) {
            s_off[0] = 0;
            if (run > MERGE_MAX) s_ovf = 1;
        }
    }
    __syncthreads();
    if (s_ovf) {
        if (tid == 0) {
            scan_list[atomicAdd(scan_n, 1)] = q;
            staged[q] = 0;
            count[q] = 0;   // the exact range scan adds this query's hits
        }
        return;
    }
    const int M = s_off[nsplits];
    for (int l = 0; l < nsplits; l++) {
        const uint2* p = cand + ((int64_t)q * nl_stride + l) * list_cap;
        for (int j = tid; j < s_off[l + 1] - s_off[l]; j += MERGE_THREADS) comp[s_off[l] + j] = (unsigned long long)p[j].y << 32;
    }
    __syncthreads();
    const float* qv = ra.q + (int64_t)q * ra.d;
    const bool l2 = ra.metric == B2F_METRIC_L2;
    const int sl = lane & 7;
    for (int c0 = 0; c0 < M; c0 += MERGE_THREADS / 8) {
        const int c = c0 + (tid >> 3);
        int32_t id = c < M ? (int32_t)(comp[c] >> 32) : -1;
        if ((int64_t)id >= ra.ntotal) id = -1;
        const float key = exact_key_8lanes(ra, qv, id, sl, l2);
        if (sl == 0 && c < M) {
            const bool hit = id >= 0 && key < tau;   // NaN is never a hit
            comp[c] = hit ? (comp[c] | __float_as_uint(key)) : ~0ull;
            if (hit) atomicAdd(&s_hits, 1);
        }
    }
    int N = 1;
    while (N < M) N <<= 1;
    for (int i = M + tid; i < N; i += MERGE_THREADS) comp[i] = ~0ull;
    __syncthreads();
    for (int k = 2; k <= N; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < N; i += MERGE_THREADS) {
                const int p = i ^ j;
                if (p > i) {
                    const unsigned long long a = comp[i], b = comp[p];
                    if ((a > b) == ((i & k) == 0)) {
                        comp[i] = b;
                        comp[p] = a;
                    }
                }
            }
            __syncthreads();
        }
    const int H = s_hits;
    for (int i = tid; i < H; i += MERGE_THREADS) {
        const unsigned long long v = comp[i];
        skey[(int64_t)q * MERGE_MAX + i] = __uint_as_float((uint32_t)v);
        sid[(int64_t)q * MERGE_MAX + i] = (int32_t)(v >> 32);
    }
    if (tid == 0) {
        staged[q] = H;
        count[q] = H;
    }
}

}  // namespace k2

// force_heap: skip LIST mode.  An index whose data defeats the shared thresholds -- rows stored in an order that puts a
// query's best rows into one or two lists, so that the thresholds never tighten and the lists overflow -- is searched
// with per-thread heaps instead (exact top-k' of every split whatever the order, ~6x the epilogue cost), for k' = 32 / 64.
int plan_tensor_scan(int nq, int64_t n, int d, int kp, bool force_heap, TensorScanPlan* plan) {
    if (kp < 8 || kp > 256 || n <= 0 || nq <= 0) return B2F_EINVAL;
    plan->kp = kp;
    plan->nq_tiles = (nq + k2::BM - 1) / k2::BM;
    plan->pair_mode = 0;
    plan->list_mode = 0;
    plan->round_tiles = 0;
    const int halves = k2::EPI_WARPS_LIST / 4;
    const int64_t ntiles = (n + k2::BN - 1) / k2::BN;
    const int kblocks = (d + k2::BK - 1) / k2::BK;
    // A "unit" is one CTA, or one CTA pair (cta_group::2).  LIST mode: the pass's work (query tile units x database)
    // is cut into one EQUAL share per unit (k2::Seg); it needs every unit resident at once (one wave), at least as
    // many units as query tile units, a few database tiles per unit, and j = ceil(k' / voucher lists of a tile) <=
    // JSLOTS for every tile.
    auto try_list = [&](int tiles, int max_units, int* units_out, int* nv_min_out, int* nseg_max_out) -> bool {
        if (tiles > max_units || ntiles < 2) return false;   // more than one wave; a single database tile
        int units = max_units;
        // >= 4 database tiles per unit: a voucher segment (at least half a share) then always has rows to vouch for;
        // a database of a few tiles gets one unit per query tile unit
        const int64_t by_db = (int64_t)tiles * ntiles / 4;
        if (by_db < units) units = (int)(by_db > tiles ? by_db : tiles);
        // A unit count that is a multiple of the tile count gives every tile the same number of whole units: no unit
        // runs two segments (no query tile reload), every list vouches, thresholds are tighter.  Same-box A/B: C3
        // (16 tiles) 144 units 25.7 ms vs 148 balanced 28.8 ms; C2 (4 pair tiles) 72 vs 74: equal.  So up to 6% of the
        // units are left idle for it; beyond that (16 or 32 pair tiles over 74 pairs: 64 of 74) the balanced split wins.
        {
            const int even = units / tiles * tiles;
            if (even >= tiles && (int64_t)units * 100 <= (int64_t)even * 106) units = even;
        }
        int j_max = 0, nseg_max = 0;
        for (int t = 0; t < tiles; t++) {
            const k2::TileInfo ti = k2::tile_info(t, tiles, units, kp, halves);
            if (ti.jfull > j_max) j_max = ti.jfull;
            if (ti.nfw + ti.nsw > nseg_max) nseg_max = ti.nfw + ti.nsw;
        }
        if (j_max > k2::JSLOTS) return false;   // rows a whole unit's list vouches for
        *units_out = units;
        *nv_min_out = j_max;
        *nseg_max_out = nseg_max;
        return true;
    };
    // (1) CTA pairs halve the L2->SM traffic of the database blocks; worth it once the batch spans several
    //     128-query tiles (an odd tile count wastes half a pair on padding).
    const bool heap_only = force_heap && (kp == 32 || kp == 64);
    int units = 0, nv_min = 1, nseg_max = 1;
    if (!heap_only && kblocks <= k2::QRES_MAX_KB && plan->nq_tiles >= 2 &&
        (plan->nq_tiles % 2 == 0 || plan->nq_tiles >= 7) && try_list((plan->nq_tiles + 1) / 2, kNumSMs / 2, &units, &nv_min, &nseg_max)) {
        plan->pair_mode = 1;
        plan->list_mode = 1;
        plan->nq_tiles = 2 * ((plan->nq_tiles + 1) / 2);
        plan->tile_units = plan->nq_tiles / 2;
    } else if (!heap_only && try_list(plan->nq_tiles, kNumSMs, &units, &nv_min, &nseg_max)) {
        plan->list_mode = 1;
        plan->tile_units = plan->nq_tiles;
    } else {
        // (2) HEAP mode: uniform splits, any number of waves; the heaps exist for k' = 32 and 64 only
        if (kp != 32 && kp != 64) return B2F_EINVAL;
        int ns = kNumSMs / plan->nq_tiles;
        if (ns < 1) ns = 1;
        if (ns > ntiles) ns = (int)ntiles;
        plan->tile_units = plan->nq_tiles;
        units = plan->nq_tiles * ns;
    }
    plan->units = units;
    plan->nsplits = units / plan->tile_units;   // HEAP mode: exact; LIST mode: whole units per query tile (diagnostics)
    if (!plan->list_mode) {
        plan->nlists = plan->nsplits;
        plan->list_j = kp;
        plan->list_g = 1;
        plan->list_cap = 0;
        return B2F_OK;
    }
    plan->nlists = nseg_max * halves;           // lists allocated per query (stride)
    const int j = nv_min;   // (try_list returns the largest j of any tile here)
    plan->list_j = j;
    plan->list_g = (kp + j - 1) / j;
    // database tiles per round of the interleaved sweep: about two per full-length segment
    {
        int r = 2 * ((units + plan->tile_units - 1) / plan->tile_units);
        if (r < 2) r = 2;
        if (r > 512) r = 512;
        plan->round_tiles = r;
    }
    // expected list length ~ 32 (blind first chunk) + (j + spread) * ln(rows per list / 32); 2.5x headroom
    {
        const double rows_per_list = (double)n * plan->tile_units / units / halves;
        const double expected = 32.0 + (j + 2.5) * log(rows_per_list > 64.0 ? rows_per_list / 32.0 : 2.0);
        int cap = (int)(2.5 * expected);
        cap = (cap + 63) / 64 * 64;
        if (cap < k2::LIST_CAP_MIN) cap = k2::LIST_CAP_MIN;
        if (cap > 1024) cap = 1024;
        plan->list_cap = cap;
    }
    return B2F_OK;
}

// diagnostics / CPU tests: the work of one unit under the balanced split, computed by the very functions the kernel runs
int plan_unit_work(int T, int U, int R, int64_t ntiles, int kp, int unit, int32_t* seg_info, int64_t* tiles, int64_t cap, int32_t* counts) {
    if (T < 1 || U < T || R < 1 || ntiles < 0 || kp < 1 || unit < 0 || unit >= U || !seg_info || !counts) return -1;
    k2::Seg seg[2];
    const int nseg = k2::unit_segments(unit, T, U, kp, k2::EPI_WARPS_LIST / 4, seg);
    for (int s = 0; s < nseg; s++) {
        seg_info[7 * s + 0] = seg[s].qtile;
        seg_info[7 * s + 1] = seg[s].slot;
        seg_info[7 * s + 2] = seg[s].nv;
        seg_info[7 * s + 3] = (int32_t)seg[s].p0;
        seg_info[7 * s + 4] = (int32_t)seg[s].p1;
        seg_info[7 * s + 5] = seg[s].j;
        seg_info[7 * s + 6] = seg[s].g;
        k2::SegIter it;
        it.init(seg[s].p0, seg[s].p1, U, R, ntiles);
        int32_t c = 0;
        for (int64_t t; (t = it.next()) >= 0; c++)
            if (tiles && c < cap) tiles[(int64_t)s * cap + c] = t;
        counts[s] = c;
    }
    return nseg;
}

int launch_tensor_scan(const __nv_bfloat16* scan, int64_t dpad, const float* norms, int64_t n, int metric,
                       const __nv_bfloat16* qb, int nq, int nq_pad, const TensorScanPlan& plan, float* pk, int32_t* pi,
                       const TensorScanLists& lists, cudaStream_t st) {
    // cuTensorMapEncodeTiled costs microseconds of host time per call and sits between two launches, so the
    // two descriptors are cached per thread and re-encoded only when a pointer or shape changes
    struct MapKey {
        const void* base;
        uint64_t inner, rows;
        uint32_t box;
        bool operator==(const MapKey& o) const { return base == o.base && inner == o.inner && rows == o.rows && box == o.box; }
    };
    static thread_local MapKey kq{}, kx{};
    static thread_local CUtensorMap mq, mx;
    const MapKey nkq{qb, (uint64_t)dpad, (uint64_t)nq_pad, (uint32_t)k2::BM};
    const MapKey nkx{scan, (uint64_t)dpad, (uint64_t)n, (uint32_t)(plan.pair_mode ? k2::BN / 2 : k2::BN)};
    if (!(nkq == kq)) {
        B2F_TRY(k2::make_map(&mq, qb, (uint64_t)dpad, (uint64_t)nq_pad, (uint64_t)dpad, k2::BM));
        kq = nkq;
    }
    if (!(nkx == kx)) {
        B2F_TRY(k2::make_map(&mx, scan, (uint64_t)dpad, (uint64_t)n, (uint64_t)dpad, nkx.box));
        kx = nkx;
    }
    const int kblocks = (int)(dpad / k2::BK);
    const bool l2 = metric == B2F_METRIC_L2;
    k2::ListArgs la{};
    if (plan.list_mode) {
        la.shared_thr = lists.shared_thr;
        la.cand = reinterpret_cast<uint2*>(lists.cand);
        la.counts = lists.counts;
        la.kp = plan.kp;
        la.nl_stride = plan.nlists;
        la.cap = plan.list_cap;
        la.final_thr = lists.final_thr;
        la.die_aware = lists.die_ctr && plan.tile_units > 1;   // one query tile: every block has one reader
        la.die_ctr = lists.die_ctr;
        la.bal_T = plan.tile_units;
        la.bal_U = plan.units;
        la.bal_R = plan.round_tiles;
        la.range_thr = lists.range_thr;
        // lists.shared_thr was filled with 0x7f7f7f7f (3.39e38, "no information yet") by the query-prep kernel
        if (plan.pair_mode)
            return l2 ? k2::launch_k2<0, true, true, true, true>(mq, mx, norms, n, nq, kblocks, plan, pk, pi, la, st)
                      : k2::launch_k2<0, false, true, true, true>(mq, mx, norms, n, nq, kblocks, plan, pk, pi, la, st);
        if (kblocks <= k2::QRES_MAX_KB)
            return l2 ? k2::launch_k2<0, true, true, true>(mq, mx, norms, n, nq, kblocks, plan, pk, pi, la, st)
                      : k2::launch_k2<0, false, true, true>(mq, mx, norms, n, nq, kblocks, plan, pk, pi, la, st);
        return l2 ? k2::launch_k2<0, true, true, false>(mq, mx, norms, n, nq, kblocks, plan, pk, pi, la, st)
                  : k2::launch_k2<0, false, true, false>(mq, mx, norms, n, nq, kblocks, plan, pk, pi, la, st);
    }
    if (plan.kp == 32)
        return l2 ? k2::launch_k2<32, true, false, false>(mq, mx, norms, n, nq, kblocks, plan, pk, pi, la, st)
                  : k2::launch_k2<32, false, false, false>(mq, mx, norms, n, nq, kblocks, plan, pk, pi, la, st);
    if (plan.kp == 64)
        return l2 ? k2::launch_k2<64, true, false, false>(mq, mx, norms, n, nq, kblocks, plan, pk, pi, la, st)
                  : k2::launch_k2<64, false, false, false>(mq, mx, norms, n, nq, kblocks, plan, pk, pi, la, st);
    set_error("tensor scan: k' = %d not supported", plan.kp);
    return B2F_EINVAL;
}

int launch_merge_lists(const TensorScanLists& lists, int nq, const TensorScanPlan& plan, unsigned long long* total_entries,
                       const RerankArgs& ra, cudaStream_t st) {
    if (nq <= 0) return B2F_OK;
    if (plan.kp > k2::KP_MAX || plan.nlists > 2 * kNumSMs) {
        set_error("merge: k' = %d / %d lists per query not supported", plan.kp, plan.nlists);
        return B2F_EINVAL;
    }
    // composites staged in shared memory: the lists arrive pruned against the final threshold, which leaves
    // about k' + (2..3) x lists entries per query; 4x that (at least RANK_MAX) keeps the CTA small enough for
    // a whole batch to be resident at once.  A query with more entries is counted as an overflow (exact scan).
    int cap_entries = plan.nlists * plan.list_cap;
    const int expect = 4 * (plan.kp + 3 * plan.nlists);
    if (cap_entries > expect) cap_entries = expect;
    if (cap_entries < k2::RANK_MAX) cap_entries = k2::RANK_MAX;
    if (cap_entries > k2::MERGE_MAX) cap_entries = k2::MERGE_MAX;
    const int cap_c = cap_entries > k2::RANK_MAX ? cap_entries : k2::RANK_MAX;
    const size_t smem = (size_t)cap_c * 8 + (size_t)k2::KP_MAX * 8 + (size_t)k2::RANK_MAX * 8 + (size_t)cap_entries * 2;
    {
        static bool configured[kMaxDevices] = {};
        const int dev = current_device_slot();
        std::lock_guard<std::mutex> lk(launch_cache_mutex());
        if (!configured[dev]) {
            B2F_CUDA(cudaFuncSetAttribute(k2::merge_lists_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)((size_t)k2::MERGE_MAX * 10 + (size_t)k2::KP_MAX * 8 + (size_t)k2::RANK_MAX * 8)));
            configured[dev] = true;
        }
    }
    // big batches: one warp per query first; what it cannot hold is flagged for the block kernel behind it
    const uint8_t* only_flagged = nullptr;
    if (nq >= k2::WM_MIN_NQ && lists.big_flag && plan.nlists <= k2::WM_LISTS && plan.kp <= k2::WM_MAX / 2 && ra.D &&
        !ra.range && !ra.out_map) {
        k2::merge_lists_warp_kernel<<<(nq + k2::WM_WARPS - 1) / k2::WM_WARPS, k2::WM_WARPS * 32, 0, st>>>(
            reinterpret_cast<const uint2*>(lists.cand), lists.counts, lists.final_thr, plan.nlists, plan.pair_mode ? 2 * k2::BM : k2::BM,
            plan.tile_units, plan.units, k2::EPI_WARPS_LIST / 4, plan.kp, plan.list_cap, total_entries, lists.big_flag, nq, ra);
        B2F_CUDA(cudaGetLastError());
        only_flagged = lists.big_flag;
        total_entries = nullptr;   // counted by the warp kernel (queries it passes on are counted by neither: diagnostics only)
    }
    k2::merge_lists_kernel<<<nq, k2::MERGE_THREADS, smem, st>>>(reinterpret_cast<const uint2*>(lists.cand), lists.counts, lists.final_thr,
                                                               plan.nlists, plan.pair_mode ? 2 * k2::BM : k2::BM, plan.tile_units, plan.units,
                                                               k2::EPI_WARPS_LIST / 4, plan.kp, plan.list_cap, cap_entries, total_entries,
                                                               only_flagged, ra);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

int launch_range_collect(const TensorScanLists& lists, int nq, const TensorScanPlan& plan, float tau, const RerankArgs& ra,
                         float* skey, int32_t* sid, int32_t* staged, int32_t* count, int32_t* scan_list, int32_t* scan_n,
                         cudaStream_t st) {
    if (nq <= 0) return B2F_OK;
    if (!plan.list_mode || plan.nlists > 2 * kNumSMs) {
        set_error("range collect: a LIST-mode plan of at most %d lists per query is required", 2 * kNumSMs);
        return B2F_EINVAL;
    }
    k2::range_collect_kernel<<<nq, k2::MERGE_THREADS, 0, st>>>(reinterpret_cast<const uint2*>(lists.cand), lists.counts, lists.range_thr,
                                                               plan.nlists, plan.pair_mode ? 2 * k2::BM : k2::BM, plan.tile_units,
                                                               plan.units, k2::EPI_WARPS_LIST / 4, plan.list_cap, tau, ra, skey, sid,
                                                               staged, count, scan_list, scan_n);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

}  // namespace b2f

#ifdef B2F_K2_TRACE
// diagnostics build only: the %globaltimer stamps of the last K2 launch, 12 per CTA (0 entry, 1 set-up done, 2 first
// tile landed, 3 last MMA issued, 4 last tile examined, 5 lists pruned, 6 all warps done, 7 TMEM freed, 8 logical unit + 1, 9 SM id, 10 first segment's MMAs issued)
extern "C" __attribute__((visibility("default"))) int b2f_debug_k2_trace(unsigned long long* out, int n) {
    if (n > 2 * b2f::kNumSMs * 12) n = 2 * b2f::kNumSMs * 12;
    if (cudaMemcpyFromSymbol(out, b2f::k2::g_k2_trace, (size_t)n * 8) != cudaSuccess) return -1;
    static unsigned long long zeros[2 * b2f::kNumSMs * 12] = {};
    return cudaMemcpyToSymbol(b2f::k2::g_k2_trace, zeros, sizeof(zeros)) == cudaSuccess ? 0 : -1;   // re-armed for the next launch
}
#endif
