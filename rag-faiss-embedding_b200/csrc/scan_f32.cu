// scan_f32.cu -- K1: coalesced, 128-bit vectorised streaming scan for small query batches.
//
// Replaces faiss's exhaustive_L2sqr_seq / exhaustive_inner_product_seq (the nq < 20 path behind
// index.search at faiss_store.py:64 and rag_datastore_manager.py:218).  Arithmetic is the reference's:
// fp32 exact-difference sum((x - q)^2) for L2, fp32 dot product for IP -- no expanded form, no
// reduced precision, so its distances are final (no re-rank).
//
// HBM-bound by design: every database row is read exactly once per call with 16-byte loads
// (ld.global.nc.L1::no_allocate), R=4 rows x NQ<=8 queries are register-tiled so each query chunk
// read from shared memory is reused 4x, warps keep 8 x 16 B loads in flight, and the per-(query,row)
// totals come out of a transposing butterfly (31 shuffles per 32 results).  Top-k is a per-warp
// sorted list in shared memory guarded by a register threshold; after the first few hundred rows
// almost nothing passes the threshold, so selection costs ~nothing and the distance matrix never
// exists anywhere.  Algorithmic bytes per launch: n * d * sizeof(row element).
//
// One cooperative launch serves any number of queries: the kernel walks them in groups of NQ, and after
// each group a grid-wide barrier lets one CTA per query merge the per-CTA partial lists and write the
// faiss-formatted (D, I) rows -- no separate merge / finalize launches.  The query list can live on the
// device (qsel + a count the kernel reads itself): that is how the tensor path's uncertified queries are
// re-run without the host ever learning how many there were (no synchronisation inside a search).
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace b2f {

constexpr int kScanWarps = 8;
constexpr int kScanThreads = kScanWarps * kWarp;
constexpr int kRowsPerGroup = 4;
constexpr int kGatherCap = 1024;   // survivors of the cross-CTA threshold ranked directly in shared memory

template <typename RowT>
struct RowVec;

template <>
struct RowVec<float> {  // 4 fp32 per 16-byte load
    static constexpr int N = 4;
    using Raw = float4;
    float v[4];
    static __device__ __forceinline__ Raw load_raw(const float* p) { return ldg_stream(reinterpret_cast<const float4*>(p)); }
    static __device__ __forceinline__ Raw zero_raw() { return make_float4(0.f, 0.f, 0.f, 0.f); }
    __device__ __forceinline__ void unpack(const Raw& t) { v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
};

template <>
struct RowVec<__nv_bfloat16> {  // 8 bf16 per 16-byte load, widened to fp32 exactly when consumed
    static constexpr int N = 8;
    using Raw = float4;   // the prefetched chunk stays packed (4 registers, not 8)
    float v[8];
    static __device__ __forceinline__ Raw load_raw(const __nv_bfloat16* p) { return ldg_stream(reinterpret_cast<const float4*>(p)); }
    static __device__ __forceinline__ Raw zero_raw() { return make_float4(0.f, 0.f, 0.f, 0.f); }
    __device__ __forceinline__ void unpack(const Raw& t) {
        const uint32_t w[4] = {__float_as_uint(t.x), __float_as_uint(t.y), __float_as_uint(t.z), __float_as_uint(t.w)};
#pragma unroll
        for (int i = 0; i < 4; i++) {
            v[2 * i] = __uint_as_float(w[i] << 16);
            v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
    }
};

struct ScalarRow {  // d % 4 != 0: rows are not 16-byte aligned, one element per lane per step
    static constexpr int N = 1;
    using Raw = float;
    float v[1];
    static __device__ __forceinline__ Raw load_raw(const float* p) { return __ldg(p); }
    static __device__ __forceinline__ Raw zero_raw() { return 0.f; }
    __device__ __forceinline__ void unpack(const Raw& t) { v[0] = t; }
};

template <int NQ, bool L2, typename RowT, typename Vec>
__global__ void __launch_bounds__(kScanThreads)
scan_kernel(const RowT* __restrict__ rows, int64_t pitch, int64_t n, int d, int dq, const float* __restrict__ q, int k,
            const ScanFuse f) {
    constexpr int R = kRowsPerGroup;
    constexpr int V = R * NQ;
    constexpr int VN = Vec::N;
    extern __shared__ __align__(16) float smem[];
    float* sq = smem;                                                   // [NQ][dq]
    float* lk = sq + NQ * dq;                                           // [warps][NQ][k]
    int32_t* li = reinterpret_cast<int32_t*>(lk + kScanWarps * NQ * k);  // [warps][NQ][k]
    // [kGatherCap] (key, id) composites of the final selection, 8-byte aligned behind the lists
    unsigned long long* gath = reinterpret_cast<unsigned long long*>(smem + (((size_t)NQ * dq + 2 * (size_t)kScanWarps * NQ * k + 1) & ~(size_t)1));
    // bf16 storage: the authoritative row is fl32(mu + stored value) -- the centre [dq] sits behind the gather area
    // (zeros when the index is not centred: x + 0 is exact)
    constexpr bool kBf16Rows = sizeof(RowT) == 2;
    float* smu = reinterpret_cast<float*>(gath + kGatherCap);
    __shared__ int s_m;
    if constexpr (kBf16Rows) {
        for (int i = threadIdx.x; i < dq; i += kScanThreads) smu[i] = (f.mu && i < d) ? f.mu[i] : 0.f;
    }

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    cg::grid_group grid = cg::this_grid();
    const int32_t* __restrict__ qsel = f.qsel;
    // the number of queries is grid-uniform: either a launch argument or a counter earlier kernels left behind
    const int nsel = f.nsel_dev ? *reinterpret_cast<const volatile int32_t*>(f.nsel_dev) : f.nsel;
    if (f.counters && blockIdx.x == 0 && threadIdx.x == 0) {
        // last kernel of a tensor-path search: fold its counters into the index totals and publish them to
        // mapped host memory (diagnostics only -- nothing waits for this)
        const int32_t c0 = f.counters[0], c1 = f.counters[1], c4 = f.counters[4];
        if (f.totals) {
            if (c0) atomicAdd(f.totals, (unsigned long long)c0);
            if (c1) atomicAdd(f.totals + 1, (unsigned long long)c1);
            if (c4) atomicAdd(f.totals + 2, (unsigned long long)c4);
        }
        if (f.host_flag) {
            volatile int32_t* hf = f.host_flag;
            hf[0] = c0;
            hf[1] = c1;
            hf[2] = f.counters[2];
            hf[3] = f.counters[3];
            hf[5] = c4;
            hf[6] = f.nq_batch;
            hf[7] = f.certify;
            __threadfence_system();
            hf[4] = f.seq;
        }
    }
    // re-arm the other launch parity's bounds (last used by the previous launch, next used by the next one)
    if (blockIdx.x == 0 && threadIdx.x < 24) f.tub[(f.parity ^ 1) * 24 + threadIdx.x] = 0xffffffffu;
    const int nparts = (int)gridDim.x;
    const int nchunk = dq / VN;
    const int64_t ngroups = (n + R - 1) / R;
    const int64_t W = (int64_t)gridDim.x * kScanWarps;
    float* wlk = lk + warp * NQ * k;
    int32_t* wli = li + warp * NQ * k;
    const int myq = lane & (NQ - 1);

    for (int g0 = 0, gi = 0; g0 < nsel; g0 += NQ, gi++) {
    const int nq_valid = nsel - g0 < NQ ? nsel - g0 : NQ;
    __syncthreads();  // the previous group's in-CTA merge has finished with the shared lists
    for (int i = threadIdx.x; i < NQ * dq; i += kScanThreads) {
        const int qi = i / dq, c = i - qi * dq;
        sq[i] = (qi < nq_valid && c < d) ? q[(int64_t)(qsel ? qsel[g0 + qi] : g0 + qi) * d + c] : 0.f;
    }
    for (int i = threadIdx.x; i < kScanWarps * NQ * k; i += kScanThreads) {
        lk[i] = FLT_MAX;
        li[i] = -1;
    }
    __syncthreads();
    float thr_k = FLT_MAX;
    int32_t thr_i = -1;

    // Software pipeline over the row groups: while a lane consumes its last chunk of a group it already has the
    // first chunk of the warp's NEXT group in flight, so the butterfly reduction, the threshold test and the rare
    // insertion never leave the memory system idle (before, every group started with an exposed load).
    // (fp32 rows with one or two queries are already bandwidth-bound at four CTAs per SM; there the extra live
    // registers of the cross-group prefetch cost a CTA of occupancy and 1-4% of bandwidth, so it is compiled in
    // for the issue-bound variants only: bf16 rows 48% -> 84% of HBM, fp32 with 8 queries +12%)
    constexpr bool kPipe = !(sizeof(RowT) == 4 && NQ <= 2);
    typename Vec::Raw xn[R];
    if constexpr (kPipe) {
        const int64_t g_first = (int64_t)blockIdx.x * kScanWarps + warp;
        if (g_first < ngroups && lane < nchunk) {
#pragma unroll
            for (int r = 0; r < R; r++)
                xn[r] = (g_first * R + r < n) ? Vec::load_raw(rows + (g_first * R + r) * pitch + (int64_t)lane * VN) : Vec::zero_raw();
        }
    }
    for (int64_t g = (int64_t)blockIdx.x * kScanWarps + warp; g < ngroups; g += W) {
        const int64_t row0 = g * R;
        const int64_t nrow0 = (g + W) * R;   // first row of this warp's next group
        float acc[V];
#pragma unroll
        for (int i = 0; i < V; i++) acc[i] = 0.f;

        if constexpr (!kPipe) {
            if (lane < nchunk) {
#pragma unroll
                for (int r = 0; r < R; r++)
                    xn[r] = (row0 + r < n) ? Vec::load_raw(rows + (row0 + r) * pitch + (int64_t)lane * VN) : Vec::zero_raw();
            }
        }
        for (int c = lane; c < nchunk; c += kWarp) {
            Vec x[R];
#pragma unroll
            for (int r = 0; r < R; r++) x[r].unpack(xn[r]);
            if constexpr (kBf16Rows) {
                float mv[VN];
#pragma unroll
                for (int h = 0; h < VN / 4; h++) {
                    const float4 t = *reinterpret_cast<const float4*>(smu + c * VN + 4 * h);
                    mv[4 * h] = t.x; mv[4 * h + 1] = t.y; mv[4 * h + 2] = t.z; mv[4 * h + 3] = t.w;
                }
#pragma unroll
                for (int r = 0; r < R; r++) {
#pragma unroll
                    for (int e = 0; e < VN; e++) x[r].v[e] = mv[e] + x[r].v[e];
                }
            }
            if (c + kWarp < nchunk) {
#pragma unroll
                for (int r = 0; r < R; r++)
                    xn[r] = (row0 + r < n) ? Vec::load_raw(rows + (row0 + r) * pitch + (int64_t)(c + kWarp) * VN) : Vec::zero_raw();
            } else if (kPipe && g + W < ngroups) {
#pragma unroll
                for (int r = 0; r < R; r++)
                    xn[r] = (nrow0 + r < n) ? Vec::load_raw(rows + (nrow0 + r) * pitch + (int64_t)lane * VN) : Vec::zero_raw();
            }
#pragma unroll
            for (int qi = 0; qi < NQ; qi++) {
                float qv[VN];
                if constexpr (VN == 1) {
                    qv[0] = sq[qi * dq + c];
                } else {
#pragma unroll
                    for (int h = 0; h < VN / 4; h++) {
                        const float4 t = *reinterpret_cast<const float4*>(sq + qi * dq + c * VN + 4 * h);
                        qv[4 * h] = t.x; qv[4 * h + 1] = t.y; qv[4 * h + 2] = t.z; qv[4 * h + 3] = t.w;
                    }
                }
#pragma unroll
                for (int r = 0; r < R; r++) {
#pragma unroll
                    for (int e = 0; e < VN; e++) {
                        if constexpr (L2) {
                            const float t = x[r].v[e] - qv[e];
                            acc[r * NQ + qi] = fmaf(t, t, acc[r * NQ + qi]);
                        } else {
                            acc[r * NQ + qi] = fmaf(x[r].v[e], qv[e], acc[r * NQ + qi]);
                        }
                    }
                }
            }
        }
        warp_multi_reduce<V>(acc, lane);
        const float key = L2 ? acc[0] : -acc[0];
        const int v = lane & (V - 1);
        const int64_t row = row0 + v / NQ;
        // filtered search: a row is looked up in the allow bitmap only when it would otherwise enter a list
        const bool pass = lane < V && row < n && (v % NQ) < nq_valid && cand_less(key, (int32_t)row, thr_k, thr_i) &&
                          (!f.allow || ((__ldg(f.allow + (row >> 5)) >> (row & 31)) & 1u));
        unsigned m = __ballot_sync(kFull, pass);
        if (m) {
            while (m) {
                const int src = __ffs(m) - 1;
                m &= m - 1;
                const float ck = __shfl_sync(kFull, key, src);
                const int32_t ci = __shfl_sync(kFull, (int32_t)row, src);
                const int cq = src % NQ;
                float* qk = wlk + cq * k;
                int32_t* qi_ = wli + cq * k;
                if (cand_less(ck, ci, qk[k - 1], qi_[k - 1])) warp_sorted_insert(qk, qi_, k, ck, ci, lane);
            }
            __syncwarp();
            thr_k = wlk[myq * k + k - 1];
            thr_i = wli[myq * k + k - 1];
        }
    }
    __syncthreads();
    // in-CTA merge: warp w < NQ merges the 8 per-warp lists of query w into this CTA's partial list
    // (double buffered over groups: the selection of group g may still be reading while group g+1 is written)
    float* pk = f.pk + (size_t)(gi & 1) * NQ * nparts * k;
    int32_t* pi = f.pi + (size_t)(gi & 1) * NQ * nparts * k;
    // Each CTA's k-th best is an upper bound of the query's global k-th best; the smallest of them (atomicMin
    // on the order-preserving encoding) leaves only ~k + a few rows alive across all CTAs.  Three slots
    // rotate over the groups: slot (gi+1)%3 was last read two groups ago and is re-armed here.
    uint32_t* tub = f.tub + f.parity * 24 + (gi % 3) * 8;
    if (gi >= 2 && blockIdx.x == 0 && threadIdx.x < 8) f.tub[f.parity * 24 + ((gi + 1) % 3) * 8 + threadIdx.x] = 0xffffffffu;
    if (warp < NQ && warp < nq_valid) {
        const int64_t o = ((int64_t)warp * nparts + blockIdx.x) * k;
        warp_merge_lists(lk + warp * k, li + warp * k, kScanWarps, k, (int64_t)NQ * k, k, pk + o, pi + o, lane);
        __syncwarp();
        if (lane == 0) atomicMin(tub + warp, enc_key(pk[o + k - 1]));  // FLT_MAX when this CTA saw fewer than k rows
    }
    grid.sync();
    // one CTA per query: gather the rows at or below the bound from all partial lists (sorted: stop at the
    // first one above it), rank them directly, write the best k in faiss conventions
    for (int qi = blockIdx.x; qi < nq_valid; qi += nparts) {
        const float* qk = pk + (int64_t)qi * nparts * k;
        const int32_t* qid = pi + (int64_t)qi * nparts * k;
        const int64_t orow = qsel ? qsel[g0 + qi] : g0 + qi;
        const float T = dec_key(__ldcg(tub + qi));
        if (threadIdx.x == 0) s_m = 0;
        __syncthreads();
        for (int l = threadIdx.x; l < nparts; l += kScanThreads) {
            for (int j = 0; j < k; j++) {
                const float key = __ldcg(qk + (int64_t)l * k + j);
                const int32_t id = __ldcg(qid + (int64_t)l * k + j);
                if (id < 0 || !(key <= T)) break;
                const int slot = atomicAdd(&s_m, 1);
                if (slot < kGatherCap) gath[slot] = ((unsigned long long)enc_key(key) << 32) | (uint32_t)id;
            }
        }
        __syncthreads();
        const int M = s_m;
        if (M <= kGatherCap) {
            unsigned long long mine[kGatherCap / kScanThreads];
            int rank[kGatherCap / kScanThreads];
#pragma unroll
            for (int u = 0; u < kGatherCap / kScanThreads; u++) {
                const int i = threadIdx.x + u * kScanThreads;
                mine[u] = i < M ? gath[i] : ~0ull;
                rank[u] = 0;
            }
            for (int j = 0; j < M; j++) {
                const unsigned long long o = gath[j];
#pragma unroll
                for (int u = 0; u < kGatherCap / kScanThreads; u++) rank[u] += o < mine[u] ? 1 : 0;  // composites are distinct (row ids)
            }
#pragma unroll
            for (int u = 0; u < kGatherCap / kScanThreads; u++) {
                if (threadIdx.x + u * kScanThreads < M && rank[u] < k) {
                    const float key = dec_key((uint32_t)(mine[u] >> 32));
                    const int64_t o = orow * k + rank[u];
                    f.D[o] = L2 ? key : -key;
                    f.I[o] = (int64_t)(uint32_t)(mine[u] & 0xffffffffu) + f.id_offset;
                }
            }
            for (int j = M + threadIdx.x; j < k; j += kScanThreads) {  // fewer than k rows in the index
                f.D[orow * k + j] = L2 ? FLT_MAX : -FLT_MAX;
                f.I[orow * k + j] = -1;
            }
        } else {
            // (ties / tiny shards with k close to the shard size) two-level merge of the sorted partial lists
            const int nl1 = (nparts + kWarp - 1) / kWarp;
            float* mk = f.mk + (int64_t)qi * (kWarp + 1) * k;
            int32_t* mi = f.mi + (int64_t)qi * (kWarp + 1) * k;
            float* fk = mk + (int64_t)kWarp * k;   // final list
            int32_t* fi = mi + (int64_t)kWarp * k;
            if (nl1 == 1) {
                if (warp == 0) warp_merge_lists<true>(qk, qid, nparts, k, k, k, fk, fi, lane);
            } else {
                for (int g = warp; g < nl1; g += kScanWarps) {
                    const int first = g * kWarp;
                    const int cnt = nparts - first < kWarp ? nparts - first : kWarp;
                    warp_merge_lists<true>(qk + (int64_t)first * k, qid + (int64_t)first * k, cnt, k, k, k, mk + (int64_t)g * k, mi + (int64_t)g * k, lane);
                }
                __syncthreads();
                if (warp == 0) warp_merge_lists<true>(mk, mi, nl1, k, k, k, fk, fi, lane);
            }
            __syncthreads();
            for (int j = threadIdx.x; j < k; j += kScanThreads) {
                const float key = __ldcg(fk + j);
                const int32_t id = __ldcg(fi + j);
                const int64_t o = orow * k + j;
                if (id < 0) {
                    f.D[o] = L2 ? FLT_MAX : -FLT_MAX;
                    f.I[o] = -1;
                } else {
                    f.D[o] = L2 ? key : -key;
                    f.I[o] = (int64_t)id + f.id_offset;
                }
            }
        }
        __syncthreads();
    }
    }  // query groups
}

int scan_max_parts() { return kNumSMs * 4; }

// queries per pass the per-warp lists allow (8 warps x NQ x k x 8 bytes of shared memory): NQ * k <= 1024
static int scan_nq_cap(int k) {
    int p = 1;
    const int lim = 1024 / k > 0 ? 1024 / k : 1;
    while (p * 2 <= lim && p < 8) p *= 2;
    return p;
}
static size_t scan_pbytes(int k) { return 2 * (size_t)scan_nq_cap(k) * scan_max_parts() * (size_t)k * 4 + 256; }
static size_t scan_mbytes(int k) { return (size_t)scan_nq_cap(k) * (kWarp + 1) * (size_t)k * 4 + 256; }

size_t scan_scratch_bytes(int k) {
    // pk/pi: [2][NQ][max parts][k] double-buffered partial lists; mk/mi: [NQ][33][k] merge scratch
    return 2 * scan_pbytes(k) + 2 * scan_mbytes(k);
}

template <int NQ, bool L2, typename RowT, typename Vec>
static int launch_one(const RowT* rows, int64_t pitch, const ScanArgs& a, cudaStream_t st) {
    const int dq = ((a.rows.d + Vec::N - 1) / Vec::N) * Vec::N;
    const size_t smem = (((size_t)NQ * dq + 2 * (size_t)kScanWarps * NQ * a.k + 1) & ~(size_t)1) * 4 + (size_t)kGatherCap * 8 +
                        (sizeof(RowT) == 2 ? (size_t)dq * 4 : 0);   // + the centre (bf16 rows)
    auto kern = scan_kernel<NQ, L2, RowT, Vec>;
    int occ = 1;
    {
        // per template instantiation AND per device; guarded, because the index mutex is per index
        static size_t configured_smem[kMaxDevices] = {};
        static size_t occ_smem[kMaxDevices];
        static int occ_cached[kMaxDevices];
        static bool occ_valid[kMaxDevices] = {};
        const int dev = current_device_slot();
        std::lock_guard<std::mutex> lk(launch_cache_mutex());
        if (configured_smem[dev] == 0 || smem > configured_smem[dev]) {
            B2F_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem > 65536 ? smem : 65536)));
            configured_smem[dev] = smem > 65536 ? smem : 65536;
        }
        // occupancy per (kernel, device, smem) is cached: the query costs microseconds and sits on the search path
        if (!occ_valid[dev] || occ_smem[dev] != smem) {
            int o = 1;
            B2F_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, kScanThreads, smem));
            occ_cached[dev] = o;
            occ_smem[dev] = smem;
            occ_valid[dev] = true;
        }
        occ = occ_cached[dev];
    }
    if (occ < 1) {
        set_error("scan kernel does not fit: smem %zu", smem);
        return B2F_EINVAL;
    }
    const int use = occ > 4 ? 4 : occ;
    const int64_t ngroups = (a.rows.n + kRowsPerGroup - 1) / kRowsPerGroup;
    int64_t want = (ngroups + kScanWarps - 1) / kScanWarps;
    int blocks = (int)(want < (int64_t)kNumSMs * use ? want : (int64_t)kNumSMs * use);
    if (blocks < 1) blocks = 1;
    ScanFuse f{};
    f.D = a.D;
    f.I = a.I;
    f.id_offset = a.id_offset;
    f.qsel = a.qsel;
    f.nsel_dev = a.nsel_dev;
    f.nsel = a.nsel;
    char* sc = static_cast<char*>(a.scratch);
    const size_t pbytes = scan_pbytes(a.k), mbytes = scan_mbytes(a.k);
    f.pk = reinterpret_cast<float*>(sc);
    f.pi = reinterpret_cast<int32_t*>(sc + pbytes);
    f.mk = reinterpret_cast<float*>(sc + 2 * pbytes);
    f.mi = reinterpret_cast<int32_t*>(sc + 2 * pbytes + mbytes);
    f.counters = a.counters;
    f.totals = a.totals;
    f.host_flag = a.host_flag;
    f.seq = a.seq;
    f.nq_batch = a.nq_batch;
    f.certify = a.certify;
    f.tub = a.tub;
    f.parity = a.parity;
    f.mu = a.rows.centre;
    f.allow = a.allow;
    const RowT* rows_ = rows;
    int64_t pitch_ = pitch, n_ = a.rows.n;
    int d_ = a.rows.d, dq_ = dq, k_ = a.k;
    const float* q_ = a.q;
    void* args[] = {(void*)&rows_, (void*)&pitch_, (void*)&n_, (void*)&d_, (void*)&dq_, (void*)&q_, (void*)&k_, (void*)&f};
    // cooperative: every CTA is resident (the grid is sized from the occupancy query), so grid.sync() is legal
    B2F_CUDA(cudaLaunchCooperativeKernel((const void*)kern, dim3((unsigned)blocks), dim3(kScanThreads), args, smem, st));
    return B2F_OK;
}

template <typename RowT, typename Vec>
static int dispatch(const RowT* rows, int64_t pitch, const ScanArgs& a, cudaStream_t st) {
    const bool l2 = a.rows.metric == B2F_METRIC_L2;
    // queries per pass: bounded by the per-warp lists (8 warps x NQ x k x 8 bytes) and the query tile in smem
    int g = 8;
    auto pow2_le = [](int x) { int p = 1; while (p * 2 <= x) p *= 2; return p; };
    const int by_k = scan_nq_cap(a.k);
    const int dq = ((a.rows.d + Vec::N - 1) / Vec::N) * Vec::N;
    const int by_smem = 16384 / (dq > 0 ? dq : 1);
    if (by_smem < 1) {
        set_error("d=%d too large for the streaming scan", a.rows.d);
        return B2F_EINVAL;
    }
    if (g > by_k) g = by_k;
    if (g > pow2_le(by_smem)) g = pow2_le(by_smem);
    // device-side query count (the tensor path's fallback): usually 0..2 queries -> a 4-wide register tile
    const int want = a.nsel_dev ? 4 : a.nsel;
#define B2F_SCAN_CASE(NQ)                                                       \
    return l2 ? launch_one<NQ, true, RowT, Vec>(rows, pitch, a, st)         \
              : launch_one<NQ, false, RowT, Vec>(rows, pitch, a, st)
    if (want <= 1 || g == 1) { B2F_SCAN_CASE(1); }
    if (want <= 2 || g == 2) { B2F_SCAN_CASE(2); }
    if (want <= 4 || g == 4) { B2F_SCAN_CASE(4); }
    B2F_SCAN_CASE(8);
#undef B2F_SCAN_CASE
}

int launch_scan(const ScanArgs& a, cudaStream_t st) {
    if (a.k <= 0 || a.k > 1024) {
        set_error("scan: k=%d out of range", a.k);
        return B2F_EINVAL;
    }
    const StoredRows& r = a.rows;
    if (r.f32) {
        if (r.d % 4 == 0) return dispatch<float, RowVec<float>>(r.f32, r.d, a, st);
        return dispatch<float, ScalarRow>(r.f32, r.d, a, st);
    }
    return dispatch<__nv_bfloat16, RowVec<__nv_bfloat16>>(r.bf16, r.pitch, a, st);
}

}  // namespace b2f
