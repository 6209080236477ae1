// merge.cu -- K3: merge of per-CTA partial top-k lists, final formatting to faiss conventions, and
// the post-all-gather merge of per-GPU results (SURVEY 8e).  All latency-bound, one CTA / warp per query.
#include "common.cuh"

namespace b2f {

constexpr int kMergeWarps = 8;

// pk/pi: [nq][nparts][klist] ascending lists -> ok/oi: [nq][kout]
__global__ void __launch_bounds__(kMergeWarps* kWarp)
merge_parts_kernel(const float* __restrict__ pk, const int32_t* __restrict__ pi, int nparts, int klist, int kout,
                   float* __restrict__ ok, int32_t* __restrict__ oi) {
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.x;
    const int ngroups = (nparts + kWarp - 1) / kWarp;
    const float* qk = pk + (int64_t)q * nparts * klist;
    const int32_t* qi = pi + (int64_t)q * nparts * klist;
    if (ngroups == 1) {
        if (warp == 0) warp_merge_lists(qk, qi, nparts, klist, klist, kout, ok + (int64_t)q * kout, oi + (int64_t)q * kout, lane);
        return;
    }
    float* sk = smem;                                               // [ngroups][kout]
    int32_t* si = reinterpret_cast<int32_t*>(smem + ngroups * kout);  // [ngroups][kout]
    for (int g = warp; g < ngroups; g += kMergeWarps) {
        const int first = g * kWarp;
        const int cnt = nparts - first < kWarp ? nparts - first : kWarp;
        warp_merge_lists(qk + (int64_t)first * klist, qi + (int64_t)first * klist, cnt, klist, klist, kout,
                         sk + g * kout, si + g * kout, lane);
    }
    __syncthreads();
    if (warp == 0) warp_merge_lists(sk, si, ngroups, kout, kout, kout, ok + (int64_t)q * kout, oi + (int64_t)q * kout, lane);
}

int launch_merge_parts(const float* pk, const int32_t* pi, int nq, int nparts, int klist, int kout, float* ok,
                       int32_t* oi, cudaStream_t st) {
    if (nq <= 0) return B2F_OK;
    const int ngroups = (nparts + kWarp - 1) / kWarp;
    if (ngroups > kWarp) {
        set_error("merge: %d partial lists exceed 1024", nparts);
        return B2F_EINVAL;
    }
    const size_t smem = ngroups > 1 ? (size_t)ngroups * kout * 8 : 0;
    if (smem > 48 * 1024) {
        static size_t configured[kMaxDevices] = {};
        const int dev = current_device_slot();
        std::lock_guard<std::mutex> lk(launch_cache_mutex());
        if (smem > configured[dev]) {
            B2F_CUDA(cudaFuncSetAttribute(merge_parts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            configured[dev] = 200 * 1024;
        }
    }
    if (smem > 200 * 1024) {
        set_error("merge: %zu bytes of shared memory needed", smem);
        return B2F_EINVAL;
    }
    merge_parts_kernel<<<nq, kMergeWarps * kWarp, smem, st>>>(pk, pi, nparts, klist, kout, ok, oi);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

// keys/ids [nq][kin] (ascending, int32 local ids) -> D/I [.][k] in faiss conventions
__global__ void finalize_kernel(const float* __restrict__ keys, const int32_t* __restrict__ ids, int nq, int kin, int k,
                                int l2, int64_t id_offset, const int32_t* __restrict__ qsel, float* __restrict__ D,
                                int64_t* __restrict__ I) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)nq * k) return;
    const int r = (int)(t / k), j = (int)(t % k);
    const int orow = qsel ? qsel[r] : r;
    float key = FLT_MAX;
    int32_t id = -1;
    if (j < kin) {
        key = keys[(int64_t)r * kin + j];
        id = ids[(int64_t)r * kin + j];
    }
    const int64_t o = (int64_t)orow * k + j;
    if (id < 0) {
        D[o] = l2 ? FLT_MAX : -FLT_MAX;
        I[o] = -1;
    } else {
        D[o] = l2 ? key : -key;
        I[o] = (int64_t)id + id_offset;
    }
}

int launch_finalize(const float* keys, const int32_t* ids, int nq, int kin, int k, int metric, int64_t id_offset,
                    const int32_t* qsel, float* D, int64_t* I, cudaStream_t st) {
    const int64_t total = (int64_t)nq * k;
    if (total <= 0) return B2F_OK;
    finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(keys, ids, nq, kin, k, metric == B2F_METRIC_L2,
                                                                      id_offset, qsel, D, I);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

// Dp/Ip: [nparts][nq][k] faiss-formatted per-shard results -> D/I [nq][k].  One warp per query,
// lane l walks list l.  Ties go to the lower label, -1 padding loses to everything.
__global__ void merge_faiss_kernel(int l2, int64_t nq, int k, int nparts, const float* __restrict__ Dp,
                                   const int64_t* __restrict__ Ip, int64_t stride_d_bytes, int64_t stride_i_bytes,
                                   float* __restrict__ D, int64_t* __restrict__ I) {
    const int lane = threadIdx.x & 31;
    const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= nq) return;
    const bool have = lane < nparts;
    const float* dl = reinterpret_cast<const float*>(reinterpret_cast<const char*>(Dp) + (have ? lane : 0) * stride_d_bytes) + q * k;
    const int64_t* il = reinterpret_cast<const int64_t*>(reinterpret_cast<const char*>(Ip) + (have ? lane : 0) * stride_i_bytes) + q * k;
    int pos = 0;
    float hk = FLT_MAX;
    int64_t hi = -1;
    if (have) {
        hi = il[0];
        hk = hi < 0 ? FLT_MAX : (l2 ? dl[0] : -dl[0]);
    }
    for (int o = 0; o < k; o++) {
        float bk = hk;
        int64_t bi = hi;
        int bl = lane;
#pragma unroll
        for (int s = 16; s >= 1; s >>= 1) {
            const float tk = __shfl_xor_sync(kFull, bk, s);
            const int64_t ti = __shfl_xor_sync(kFull, bi, s);
            const int tl = __shfl_xor_sync(kFull, bl, s);
            const bool less = tk < bk || (tk == bk && ((uint64_t)ti < (uint64_t)bi || (ti == bi && tl < bl)));
            if (less) { bk = tk; bi = ti; bl = tl; }
        }
        if (lane == 0) {
            D[q * k + o] = bi < 0 ? (l2 ? FLT_MAX : -FLT_MAX) : (l2 ? bk : -bk);
            I[q * k + o] = bi;
        }
        if (have && lane == bl) {
            pos++;
            if (pos < k) {
                hi = il[pos];
                hk = hi < 0 ? FLT_MAX : (l2 ? dl[pos] : -dl[pos]);
            } else {
                hi = -1;
                hk = FLT_MAX;
            }
        }
    }
}

int launch_merge_faiss(int metric, int64_t nq, int64_t k, int nparts, const float* Dp, const int64_t* Ip,
                       int64_t stride_d_bytes, int64_t stride_i_bytes, float* D, int64_t* I, cudaStream_t st) {
    if (nq <= 0 || k <= 0) return B2F_OK;
    if (nparts < 1 || nparts > kWarp) {
        set_error("merge_topk: nparts %d not in [1,32]", nparts);
        return B2F_EINVAL;
    }
    const int wpb = 4;
    merge_faiss_kernel<<<(unsigned)((nq + wpb - 1) / wpb), wpb * kWarp, 0, st>>>(metric == B2F_METRIC_L2, nq, (int)k,
                                                                                nparts, Dp, Ip, stride_d_bytes, stride_i_bytes, D, I);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

// Range-search results of nparts shards -> one result, query by query in ascending label order.  Part p: lims
// lims[p * (nq + 1) ..] (any base), hits at Dp / Ip + p * stride bytes.  One thread per input hit: it finds its query
// by binary search over its part's lims, and its output slot as the query's output base + its index in its own list
// + the labels below it in every other part's list of that query (one lower_bound per part).  Labels are disjoint
// across parts, so the slots are a permutation: no thread waits for another, and a query with 10^5 hits is spread
// over as many threads as it has hits.  The hit count is read from the device lims, so the grid strides over it.
constexpr int kRangeMergeThreads = 256;

__global__ void __launch_bounds__(kRangeMergeThreads)
merge_range_kernel(int64_t nq, int nparts, const int64_t* __restrict__ lims, const char* __restrict__ Dp,
                   const char* __restrict__ Ip, int64_t stride, float* __restrict__ D, int64_t* __restrict__ I) {
    __shared__ int64_t base[kWarp];       // lims[p][0]
    __shared__ int64_t first[kWarp + 1];  // hits of parts < p
    if (threadIdx.x < kWarp) {
        const int lane = threadIdx.x;
        int64_t b = 0, inc = 0;
        if (lane < nparts) {
            b = lims[lane * (nq + 1)];
            inc = lims[lane * (nq + 1) + nq] - b;
        }
#pragma unroll
        for (int s = 1; s < kWarp; s <<= 1) {
            const int64_t t = __shfl_up_sync(kFull, inc, s);
            if (lane >= s) inc += t;
        }
        base[lane] = b;
        first[lane + 1] = inc;
        if (lane == 0) first[0] = 0;
    }
    __syncthreads();
    const int64_t total = first[nparts];
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        int p = 0;
        while (first[p + 1] <= t) p++;
        const int64_t e = t - first[p];
        const int64_t* lp = lims + p * (nq + 1);
        const int64_t key = e + base[p];
        int64_t lo = 0, hi = nq;   // the last query q with lp[q] <= key: the one whose list holds e
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (lp[mid] <= key) lo = mid;
            else hi = mid;
        }
        const int64_t q = lo;
        const int64_t label = reinterpret_cast<const int64_t*>(Ip + p * stride)[e];
        const float dist = reinterpret_cast<const float*>(Dp + p * stride)[e];
        int64_t o = key - lp[q];
        for (int r = 0; r < nparts; r++) {
            const int64_t* lr = lims + r * (nq + 1);
            const int64_t s = lr[q] - base[r];
            o += s;
            if (r == p) continue;
            const int64_t* ir = reinterpret_cast<const int64_t*>(Ip + r * stride) + s;
            int64_t a = 0, z = lr[q + 1] - lr[q];   // lower_bound of label in part r's list of query q
            while (a < z) {
                const int64_t mid = (a + z) >> 1;
                if (ir[mid] < label) a = mid + 1;
                else z = mid;
            }
            o += a;
        }
        D[o] = dist;
        I[o] = label;
    }
}

int launch_merge_range(int64_t nq, int nparts, const int64_t* lims, const float* Dp, const int64_t* Ip, int64_t stride,
                       float* D, int64_t* I, cudaStream_t st) {
    if (nq <= 0) return B2F_OK;
    // enough resident threads to hide the dependent loads of the searches; the grid strides over the device's hit count
    merge_range_kernel<<<kNumSMs * 8, kRangeMergeThreads, 0, st>>>(nq, nparts, lims, reinterpret_cast<const char*>(Dp),
                                                                   reinterpret_cast<const char*>(Ip), stride, D, I);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

}  // namespace b2f
