// common.cuh -- shared device/host helpers for the flat-search kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <float.h>
#include <stdint.h>
#include <stdio.h>

#include <mutex>

#include "../../include/b200flat.h"

namespace b2f {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kNumSMs = 148;  // B200: 2 dies x 74

// Selection keys are "smaller is better": L2 -> squared distance, IP -> -inner product.
// Candidates are totally ordered by (key, id); id -1 (empty slot) compares as the largest id,
// so an empty slot (FLT_MAX, -1) loses against everything that faiss would admit.
struct Cand {
    float key;
    int32_t id;
};

__host__ __device__ __forceinline__ bool cand_less(float ka, int32_t ia, float kb, int32_t ib) {
    return ka < kb || (ka == kb && (uint32_t)ia < (uint32_t)ib);
}

// Order-preserving float <-> uint32 map (64-bit (key,id) composites, atomicMin on keys)
__device__ __forceinline__ uint32_t enc_key(float f) {
    const uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float dec_key(uint32_t e) {
    return __uint_as_float((e & 0x80000000u) ? (e & 0x7fffffffu) : ~e);
}

// ---- warp-level helpers ------------------------------------------------------------------------

// Sum V values across the warp with V-1 + (5 - log2 V) * V shuffles instead of 5 * V: after the
// call lane l holds the warp-wide total of v[l & (V-1)] in v[0].  V must be a power of two <= 32.
template <int V>
__device__ __forceinline__ void warp_multi_reduce(float (&v)[V], int lane) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        if (s >= V) {
#pragma unroll
            for (int i = 0; i < V; i++) v[i] += __shfl_xor_sync(kFull, v[i], s);
        } else {
            const bool upper = (lane & s) != 0;
#pragma unroll
            for (int i = 0; i < s; i++) {
                float send = upper ? v[i] : v[i + s];
                float keep = upper ? v[i + s] : v[i];
                v[i] = keep + __shfl_xor_sync(kFull, send, s);
            }
        }
    }
}

// Insert (key,id) into an ascending (key,id)-sorted list of length k held in shared/global memory,
// dropping the last element.  Called by all 32 lanes with the same arguments.  The caller has
// already established (key,id) < list[k-1].
__device__ __forceinline__ void warp_sorted_insert(float* lk, int32_t* li, int k, float key, int32_t id,
                                                   int lane) {
    for (int base = ((k - 1) / kWarp) * kWarp; base >= 0; base -= kWarp) {
        const int j = base + lane;
        float nk = 0.f;
        int32_t ni = 0;
        bool wr = false;
        if (j < k) {
            const float ck = lk[j];
            const int32_t ci = li[j];
            if (cand_less(key, id, ck, ci)) {  // new element lands at or before j
                wr = true;
                if (j > 0 && cand_less(key, id, lk[j - 1], li[j - 1])) {
                    nk = lk[j - 1];
                    ni = li[j - 1];
                } else {
                    nk = key;
                    ni = id;
                }
            }
        }
        __syncwarp();
        if (wr) {
            lk[j] = nk;
            li[j] = ni;
        }
        __syncwarp();
    }
}

// Merge up to 32 ascending lists (list l starts at keys + l*stride, length len) into the k best,
// written by lane 0 to (ok, oi).  One warp.  Lists may contain (FLT_MAX,-1) padding.
// CG: read the lists with ld.global.cg (they were written by other SMs during this kernel: bypass L1).
template <bool CG = false>
__device__ __forceinline__ void warp_merge_lists(const float* keys, const int32_t* ids, int nlists, int len,
                                                 int64_t stride, int k, float* ok, int32_t* oi, int lane) {
    int pos = 0;
    float hk = FLT_MAX;
    int32_t hi = -1;
    const bool have = lane < nlists;
    if (have && len > 0) {
        hk = CG ? __ldcg(keys + (int64_t)lane * stride) : keys[(int64_t)lane * stride];
        hi = CG ? __ldcg(ids + (int64_t)lane * stride) : ids[(int64_t)lane * stride];
    }
    for (int o = 0; o < k; o++) {
        float bk = hk;
        int32_t bi = hi;
        int bl = lane;
#pragma unroll
        for (int s = 16; s >= 1; s >>= 1) {
            float tk = __shfl_xor_sync(kFull, bk, s);
            int32_t ti = __shfl_xor_sync(kFull, bi, s);
            int tl = __shfl_xor_sync(kFull, bl, s);
            if (cand_less(tk, ti, bk, bi) || (tk == bk && ti == bi && tl < bl)) {
                bk = tk;
                bi = ti;
                bl = tl;
            }
        }
        if (lane == 0) {
            ok[o] = bk;
            oi[o] = bi;
        }
        if (lane == bl && have) {
            pos++;
            if (pos < len) {
                hk = CG ? __ldcg(keys + (int64_t)lane * stride + pos) : keys[(int64_t)lane * stride + pos];
                hi = CG ? __ldcg(ids + (int64_t)lane * stride + pos) : ids[(int64_t)lane * stride + pos];
            } else {
                hk = FLT_MAX;
                hi = -1;
            }
        }
    }
}

__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}

// cudaFuncSetAttribute / occupancy are per device: launchers cache what they configured per device, so one
// process may drive indexes on several GPUs.
constexpr int kMaxDevices = 64;
// Launchers keep small per-device caches (configured shared-memory sizes, occupancy).  The index mutex is per
// index, so two indexes searched from two threads reach the same launcher concurrently: the caches are guarded by
// one process-wide mutex (taken only around the cache look-up, never around a launch).
std::mutex& launch_cache_mutex();
inline int current_device_slot() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= kMaxDevices) d = 0;
    return d;
}

// ---- host-side error plumbing ------------------------------------------------------------------
void set_error(const char* fmt, ...);

#define B2F_CUDA(expr)                                                                              \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            b2f::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return B2F_ECUDA;                                                                       \
        }                                                                                           \
    } while (0)

#define B2F_TRY(expr)            \
    do {                         \
        int _rc = (expr);        \
        if (_rc != B2F_OK) return _rc; \
    } while (0)

// ---- kernel launchers (one per .cu file) -------------------------------------------------------

// K1: fp32 exact-difference streaming scan + fused merge + faiss formatting, ONE cooperative launch for any
// number of queries (walked in groups of <= 8 inside the kernel).
struct ScanFuse {                  // device-side view (kernel argument)
    float* D;                      // [*, k] faiss-formatted distances
    int64_t* I;                    // [*, k] labels (+ id_offset)
    int64_t id_offset;
    const int32_t* qsel;           // optional: query slot i reads row qsel[i] of q and writes row qsel[i] of D / I
    const int32_t* nsel_dev;       // optional: number of queries, read on the device (overrides nsel)
    int nsel;
    float* pk;                     // [2][NQ][parts][k] per-CTA partial lists (double buffered over query groups)
    int32_t* pi;
    float* mk;                     // [NQ][33][k] merge scratch
    int32_t* mi;
    int32_t* counters;             // optional [8]: the search's counters, published by this (final) kernel
    unsigned long long* totals;    // optional [2]: running totals of the index (fallbacks, overflows)
    int32_t* host_flag;            // optional mapped host memory [16]
    int32_t seq;
    int32_t nq_batch, certify;     // echoed to the host flag (adaptive slack)
    uint32_t* tub;                 // persistent [2][3][8]: per-query upper bound of the k-th best key (min over CTAs), all-ones when idle
    int32_t parity;                // launch parity: this launch uses tub[parity] and re-arms tub[parity ^ 1]
    const float* mu;               // bf16 rows: centre added back to every stored row (null: none)
};
struct ScanArgs {                  // host-side launch description
    const float* rows_f32;         // fp32 rows, or
    const __nv_bfloat16* rows_bf16;
    int64_t pitch_bf16;
    const float* mu;               // bf16 rows: the centre added back to every stored row (null: none)
    int64_t n;
    int d, metric, k;
    const float* q;                // [*, d] device fp32
    const int32_t* qsel;           // optional (device)
    const int32_t* nsel_dev;       // optional (device)
    int nsel;
    float* D;
    int64_t* I;
    int64_t id_offset;
    void* scratch;                 // scan_scratch_bytes(k) bytes
    int32_t* counters;
    unsigned long long* totals;
    int32_t* host_flag;
    int32_t seq;
    int32_t nq_batch, certify;
    uint32_t* tub;
    int32_t parity;
};
constexpr int kScanTubWords = 2 * 3 * 8;
int scan_max_parts();
size_t scan_scratch_bytes(int k);
int launch_scan(const ScanArgs& a, cudaStream_t st);

// K3: merge nparts sorted lists per query into the best kout: pk/pi [nq][nparts][klist] -> ok/oi [nq][kout]
int launch_merge_parts(const float* pk, const int32_t* pi, int nq, int nparts, int klist, int kout, float* ok,
                       int32_t* oi, cudaStream_t st);
// final formatting: keys -> faiss distances, int32 local ids -> int64 labels (+offset), padding.
// qsel (optional) scatters row r of the input to output row qsel[r].
int launch_finalize(const float* keys, const int32_t* ids, int nq, int kin, int k, int metric, int64_t id_offset,
                    const int32_t* qsel, float* D, int64_t* I, cudaStream_t st);
// multi-GPU merge of nparts faiss-formatted [nq][k] lists; part p of the distances / labels sits p * stride bytes
// after part 0 (dense [nparts][nq][k] arrays, or one packed message per rank)
int launch_merge_faiss(int metric, int64_t nq, int64_t k, int nparts, const float* Dp, const int64_t* Ip,
                       int64_t stride_d_bytes, int64_t stride_i_bytes, float* D, int64_t* I, cudaStream_t st);
// multi-GPU merge of nparts range-search results (lims [nparts][nq + 1], any base; hits of part p stride * p bytes after
// part 0) into one result in ascending label order per query
int launch_merge_range(int64_t nq, int nparts, const int64_t* lims, const float* Dp, const int64_t* Ip, int64_t stride,
                       float* D, int64_t* I, cudaStream_t st);

// K5: ingest. src fp32 [n,d] (device) -> rows fp32 (optional), bf16 scan copy (pitch dpad), norms.
// stats (device, 2 floats): running max |bf16(x)|^2 and max |x - bf16(x)|^2 (certification bound).
// mu (optional, device [d]): the scan copy / norms / stats are taken of the centred rows x - mu; ip_bias: store
// -mu.x instead of |x~'|^2 in norms (inner-product indexes: the row's bias in the tensor pass).
// bf16_auth: bf16 storage -- the authoritative row is fl32(mu + scan row); the IP bias and stats[1] refer to it.
int launch_ingest(const float* src, int64_t n, int d, float* rows_f32, __nv_bfloat16* scan, int64_t dpad,
                  float* norms, float* stats, const float* mu, int ip_bias, int bf16_auth, cudaStream_t st);
// mu[c] = mean of column c over m rows, which may arrive in pieces: begin; pass 0 over every piece; pass 1 over every
// piece; finish.  src of a piece holds its `rows` rows from row row0 (a multiple of 64) on.  acc: d 64-bit words + d floats.
int launch_mean_begin(int d, unsigned long long* acc, cudaStream_t st);
int launch_mean_pass(const float* src, int64_t row0, int64_t rows, int64_t m, int d, unsigned long long* acc, int pass,
                     cudaStream_t st);
int launch_mean_finish(int64_t m, int d, float* mu, unsigned long long* acc, cudaStream_t st);
// K7: pooling (+normalise) of encoder output, optionally fused with the ingest writes.
int launch_pool(const float* hidden, const int64_t* mask, int64_t B, int64_t T, int d, int pool, int normalize,
                float* out_f32, __nv_bfloat16* scan, int64_t dpad, float* norms, float* stats, cudaStream_t st);
int launch_synth(uint64_t seed, int64_t row0, int64_t nrows, int d, int normalize, float* out, cudaStream_t st);
// query preparation for the tensor path: bf16 copy (pitch dpad, rows padded to nq_pad with zeros),
// |q|^2 in fp32 and the norm of the bf16 rounding error of each query.
// also clears `zero_words` 32-bit words at `zero` and fills `fill_words` words at `fill` with 0x7f7f7f7f
// (the "no information yet" value of the shared thresholds), saving two memset launches per search
int launch_prep_queries(const float* q, int nq, int nq_pad, int d, __nv_bfloat16* qb, int64_t dpad, float* qnorm,
                        float* qerr, float* qconst, const float* mu, uint32_t* zero, int zero_words, uint32_t* fill,
                        int64_t fill_words, cudaStream_t st);
// range pass helpers (ingest.cu)
int launch_gather_failed(const float* q, int d, const int32_t* fail_list, const float* fail_tau, const int32_t* nfail, int nfail_host,
                         int cap, float* qf, float* tau2, int32_t* out_map, int32_t* range_count, int32_t* fail_list2,
                         int32_t* fail_count2, cudaStream_t st);
// thr[i] for tau = tau2[i] (tau2 null: tau_all for every i); out_map (optional): slots with out_map[i] < 0 list nothing
int launch_range_thresholds(const float* tau2, float tau_all, const int32_t* out_map, int n, int d, int metric, const float* qnorm,
                            const float* qerr, const float* qconst, float max_row_norm, float max_row_err, float mu_norm, float* thr,
                            cudaStream_t st);
int launch_bf16_to_f32(const __nv_bfloat16* src, int64_t pitch, int64_t n, int d, const float* mu, float* dst, cudaStream_t st);

// K4: exact fp32 re-rank of coarse candidates + certification.
struct RerankArgs {
    const float* rows_f32;          // authoritative fp32 rows (or null)
    const __nv_bfloat16* rows_bf16; // bf16 storage: the stored rows x~'; the authoritative row is fl32(centre + x~')
    int64_t pitch_bf16;
    const float* centre;            // bf16 storage: the index's centre mu [d] (null: mu = 0)
    const float* q;                 // [nq, d] fp32
    const float* qnorm;             // |q|^2
    const float* qerr;              // |q' - bf16(q')|   (q' = q - mu)
    const float* qconst;            // q.mu - mu.mu (0 without centring): true inner product = centred one + mu.x + qconst
    float mu_norm;                  // |mu|
    const float* cand_key;          // [nq, kp] coarse keys (sorted ascending)
    const int32_t* cand_id;         // [nq, kp]
    int nq, kp, k, d, metric;
    int64_t ntotal;
    float max_row_norm;             // max |x~| over the index (bf16 copy)
    float max_row_err;              // max |x - bf16(x)| over the index (0 for bf16 storage)
    int certify;
    float* out_key;                 // [nq, k] exact keys   (used when D == nullptr)
    int32_t* out_id;                // [nq, k]
    float* D;                       // optional fused finalize: faiss-formatted distances [nq, k]
    int64_t* I;                     //                          labels [nq, k] (+ id_offset)
    int64_t id_offset;
    int32_t* fail_list;             // queries that could not be certified (q + q_base), re-run by the closing exact scan
    int32_t* fail_count;            // [0] uncertified queries, [1] of which list overflows, [2..3] u64 list entries
    int32_t q_base;                 // first query of this pass within the whole batch (query chunks)
    float* fail_tau;                // optional [nq]: exact k-th key found for fail_list[i] (FLT_MAX: none) -- the range pass's input
    const int32_t* out_map;         // optional: query q of this launch writes row out_map[q] of D / I (< 0: skip) and is
                                    // recorded under that index when it fails (range pass over compacted failed queries)
    int32_t range;                  // 1: range pass -- the lists hold EVERY row with coarse key <= the fixed threshold: re-rank all
};
int launch_rerank(const RerankArgs& a, cudaStream_t st);

// K2: tcgen05 / TMEM / TMA contraction with fused top-k (gemm_topk_sm100.cu)
struct TensorScanPlan {
    int nq_tiles;      // ceil(nq / 128)
    int nsplits;       // database streams per query tile (LIST mode: whole units per tile; the balanced split gives every unit units/tile_units of a tile)
    int units;         // CTAs (or CTA pairs) launched
    int tile_units;    // query tile units (pair tiles when pair_mode) whose work the units share equally
    int nlists;        // LIST mode: candidate lists allocated per query = (most segments of any tile) x column halves
    int kp;            // candidates kept per query
    int list_mode;     // 1: shared-threshold candidate lists (K3b merge), 0: per-thread heaps (K3 merge)
    int pair_mode;     // 1: CTA pairs (tcgen05 cta_group::2, M = 256 queries per pair); nq_tiles is then even
    int list_j;        // rows each split vouches for
    int list_g;        // splits consulted for the shared threshold (g * j >= kp)
    int list_cap;      // entries per (query, split) list
    int round_tiles;   // LIST mode: database tiles per round of the interleaved sweep (k2::SegIter)
};
struct TensorScanLists {  // LIST-mode scratch (device)
    float* shared_thr;    // [nlists][nq_pad]
    void* cand;           // [nq_pad * nlists][list_cap] x 8 bytes
    int32_t* counts;      // [nq_pad * nlists]
    float* final_thr;     // [nq_pad * nlists]  the threshold each list was pruned against at the end of the stream
    int32_t* die_ctr;     // [4] ticket counters of the die-aware unit assignment (zero between launches), or null
    uint8_t* big_flag;    // [nq_pad] big batches: queries the warp-per-query merge passes on to the block kernel
    const float* range_thr;  // optional [nq_pad]: range pass -- fixed per-query thresholds (no shared thresholds, no refresh)
};
// force_heap: per-thread heaps instead of LIST mode (k' = 32 / 64)
int plan_tensor_scan(int nq, int64_t n, int d, int kp, bool force_heap, TensorScanPlan* plan);
int plan_unit_work(int T, int U, int R, int64_t ntiles, int kp, int unit, int32_t* seg_info, int64_t* tiles, int64_t cap, int32_t* counts);
int launch_tensor_scan(const __nv_bfloat16* scan, int64_t dpad, const float* norms, int64_t n, int metric,
                       const __nv_bfloat16* qb, int nq, int nq_pad, const TensorScanPlan& plan, float* pk,
                       int32_t* pi, const TensorScanLists& lists, cudaStream_t st);
// K3b + K4 fused: per query, merge the variable-length lists, re-rank the kp best exactly, certify (retrying
// with every list entry when the first attempt fails), write (D, I); uncertified queries go to ra.fail_list
int launch_merge_lists(const TensorScanLists& lists, int nq, const TensorScanPlan& plan, unsigned long long* total_entries,
                       const RerankArgs& ra, cudaStream_t st);

// ---- range search (index.range_search(x, radius)): hit <=> exact key (ra: rows and queries, as K4) < tau ----------------
constexpr int kRangeHitsMax = 4096;   // list entries one query of the tensor path filters (= the merge's MERGE_MAX)
// The lists of a range-threshold tensor pass (lists.range_thr) -> each query's hits, sorted by row id, staged in
// skey / sid [nq][kRangeHitsMax] with their number in staged[q] and count[q]; queries the lists cannot answer (overflow, more
// than kRangeHitsMax entries, NaN threshold) get staged[q] = count[q] = 0 and are appended to scan_list / *scan_n.
int launch_range_collect(const TensorScanLists& lists, int nq, const TensorScanPlan& plan, float tau, const RerankArgs& ra,
                         float* skey, int32_t* sid, int32_t* staged, int32_t* count, int32_t* scan_list, int32_t* scan_n,
                         cudaStream_t st);
// The exact range scan's row tiles: the rows split into at most 2 x kNumSMs contiguous tiles
struct RangeScanGeometry {
    int64_t tile_rows;
    int ntiles;
};
RangeScanGeometry range_scan_geometry(int64_t n);
// Exact range scan of the listed queries (list null: 0..nlist_max-1; nlist_dev null: nlist_max of them) over all rows.
// emit = false: hits per (list slot, tile) to tile_counts [nlist_max][ntiles], added to count[query].  emit = true: the same
// hits, in row order, to D / I at base + lims[query] (+ the query's hits in earlier tiles).
int launch_range_scan(const RerankArgs& a, float tau, const int32_t* list, const int32_t* nlist_dev, int nlist_max,
                      int32_t* tile_counts, int32_t* count, const int64_t* lims, int64_t base, float* D, int64_t* I,
                      int64_t id_offset, bool emit, cudaStream_t st);
// lims[0..n]: exclusive prefix sums of count[0..n) (n <= 1024)
int launch_range_offsets(const int32_t* count, int n, int64_t* lims, cudaStream_t st);
// staged hits of queries 0..nq-1 to D / I at base + lims[q] in faiss format (L2: key, IP: -key; label = id + id_offset)
int launch_range_emit(const float* skey, const int32_t* sid, const int32_t* staged, const int64_t* lims, int nq, int64_t base, int metric,
                      float* D, int64_t* I, int64_t id_offset, cudaStream_t st);

}  // namespace b2f
