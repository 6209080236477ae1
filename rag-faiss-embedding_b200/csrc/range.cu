// range.cu -- range search kernels besides the list filter (range_collect_kernel, gemm_topk_sm100.cu): the exact range
// scan, the per-chunk offsets and the emit of staged hits.  A row is a hit of a query when its exact key, computed by
// exact_key_8lanes like on every other path, is strictly below tau (L2: the radius; IP: minus the radius).
#include "rerank.cuh"

namespace b2f {

namespace {

constexpr int kScanThreads = 256;
constexpr int kScanGroup = 8;   // queries per work item: one warp each when the hits are written

// The exact range scan, two passes over the same work items (a group of <= 8 listed queries x a tile of tile_rows rows).
// COUNT: hits per (query, tile) to tile_counts[slot][tile], and their total added to count[query].  EMIT: each tile's hits
// in row order at lims[query] + the hits of the query's earlier tiles.  The list and its length live on the device (null
// list: queries 0..n-1, null nlist_dev: nlist_host of them); a persistent grid walks the items tile by tile so that the
// groups working on the same rows share them in L2.
template <bool EMIT>
__global__ void __launch_bounds__(kScanThreads, 4)
range_scan_kernel(const RerankArgs a, float tau, const int32_t* __restrict__ list, const int32_t* __restrict__ nlist_dev, int nlist_host,
                  int64_t tile_rows, int ntiles, int32_t* __restrict__ tile_counts, int32_t* __restrict__ count,
                  const int64_t* __restrict__ lims, int64_t base, float* __restrict__ D, int64_t* __restrict__ I, int64_t id_offset) {
    __shared__ float s_key[kScanGroup][32];
    __shared__ int s_hit[kScanGroup][32];
    __shared__ int s_cnt[kScanGroup];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, sl = lane & 7, rg = tid >> 3;
    const bool l2 = a.rows.metric == B2F_METRIC_L2;
    const int nl = nlist_dev ? *nlist_dev : nlist_host;
    const int ngroups = (nl + kScanGroup - 1) / kScanGroup;
    const int64_t items = (int64_t)ngroups * ntiles;
    for (int64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const int tile = (int)(it / ngroups), g = (int)(it % ngroups);
        const int s0 = g * kScanGroup;
        const int nqg = nl - s0 < kScanGroup ? nl - s0 : kScanGroup;
        const int64_t r_lo = (int64_t)tile * tile_rows;
        const int64_t r_hi = r_lo + tile_rows < a.rows.n ? r_lo + tile_rows : a.rows.n;
        int64_t off = 0;   // EMIT: where warp w's query writes next
        if (EMIT) {
            if (warp < nqg) {
                const int slot = s0 + warp;
                int c = 0;
                for (int t = lane; t < tile; t += 32) c += tile_counts[(int64_t)slot * ntiles + t];
                c = __reduce_add_sync(kFull, c);
                off = base + lims[list ? list[slot] : slot] + c;
            }
        } else if (tid < kScanGroup) {
            s_cnt[tid] = 0;
        }
        __syncthreads();
        for (int64_t r0 = r_lo; r0 < r_hi; r0 += kScanThreads / 8) {
            const int64_t row = r0 + rg;
            // filtered search: an excluded row is neither read nor counted
            const bool valid = row < r_hi && (!a.allow || ((__ldg(a.allow + (row >> 5)) >> (row & 31)) & 1u));
#pragma unroll 1
            for (int i = 0; i < nqg; i++) {
                const int32_t qi = list ? list[s0 + i] : s0 + i;
                const float key = exact_key_8lanes(a.rows, a.q + (int64_t)qi * a.rows.d, valid ? (int32_t)row : -1, sl, l2);
                const bool hit = valid && key < tau;   // NaN is never a hit
                if (EMIT) {
                    if (sl == 0) {
                        s_key[i][rg] = key;
                        s_hit[i][rg] = hit;
                    }
                } else {
                    const int c = __popc(__ballot_sync(kFull, sl == 0 && hit));
                    if (lane == 0 && c) atomicAdd(&s_cnt[i], c);
                }
            }
            if (EMIT) {
                __syncthreads();
                if (warp < nqg) {   // warp w writes query w's hits among these 32 rows, in row order
                    const unsigned m = __ballot_sync(kFull, s_hit[warp][lane] != 0);
                    if (s_hit[warp][lane]) {
                        const int64_t o = off + __popc(m & ((1u << lane) - 1u));
                        D[o] = l2 ? s_key[warp][lane] : -s_key[warp][lane];
                        I[o] = r0 + lane + id_offset;
                    }
                    off += __popc(m);
                }
                __syncthreads();
            }
        }
        if (!EMIT) {
            __syncthreads();
            if (tid < nqg) {
                tile_counts[(int64_t)(s0 + tid) * ntiles + tile] = s_cnt[tid];
                if (s_cnt[tid]) atomicAdd(count + (list ? list[s0 + tid] : s0 + tid), s_cnt[tid]);
            }
            __syncthreads();
        }
    }
}

// lims[i] = hits of queries [0, i) of the chunk, for i <= n (one block; n <= 1024)
__global__ void __launch_bounds__(1024) range_offsets_kernel(const int32_t* __restrict__ count, int n, int64_t* __restrict__ lims) {
    __shared__ int64_t s_w[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int64_t v = tid < n ? count[tid] : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t up = __shfl_up_sync(kFull, v, d);
        if (lane >= d) v += up;
    }
    if (lane == 31) s_w[warp] = v;
    __syncthreads();
    int64_t before = 0;
    for (int w = 0; w < warp; w++) before += s_w[w];
    v += before;
    if (tid < n) lims[tid + 1] = v;
    if (tid == 0) lims[0] = 0;
}

// The staged hits of query q (range_collect_kernel) to D / I at base + lims[q]: L2 distance = key, IP = -key
__global__ void __launch_bounds__(256) range_emit_kernel(const float* __restrict__ skey, const int32_t* __restrict__ sid,
                                                         const int32_t* __restrict__ staged, const int64_t* __restrict__ lims,
                                                         int64_t base, int l2, float* __restrict__ D, int64_t* __restrict__ I,
                                                         int64_t id_offset) {
    const int q = blockIdx.x;
    const int h = staged[q];
    const int64_t o = base + lims[q];
    for (int i = threadIdx.x; i < h; i += blockDim.x) {
        const float k = skey[(int64_t)q * kRangeHitsMax + i];
        D[o + i] = l2 ? k : -k;
        I[o + i] = (int64_t)sid[(int64_t)q * kRangeHitsMax + i] + id_offset;
    }
}

}  // namespace

RangeScanGeometry range_scan_geometry(int64_t n) {
    RangeScanGeometry g;
    g.tile_rows = (n + 2 * kNumSMs - 1) / (2 * kNumSMs);
    g.tile_rows = (g.tile_rows + 31) / 32 * 32;
    if (g.tile_rows < 64) g.tile_rows = 64;
    g.ntiles = n > 0 ? (int)((n + g.tile_rows - 1) / g.tile_rows) : 0;
    return g;
}

int launch_range_scan(const RerankArgs& a, float tau, const int32_t* list, const int32_t* nlist_dev, int nlist_max,
                      int32_t* tile_counts, int32_t* count, const int64_t* lims, int64_t base, float* D, int64_t* I,
                      int64_t id_offset, bool emit, cudaStream_t st) {
    const RangeScanGeometry g = range_scan_geometry(a.rows.n);
    const int64_t items = (int64_t)((nlist_max + kScanGroup - 1) / kScanGroup) * g.ntiles;
    if (items <= 0) return B2F_OK;
    const int blocks = (int)(items < 4 * kNumSMs ? items : 4 * kNumSMs);
    if (emit)
        range_scan_kernel<true><<<blocks, kScanThreads, 0, st>>>(a, tau, list, nlist_dev, nlist_max, g.tile_rows, g.ntiles, tile_counts,
                                                                  count, lims, base, D, I, id_offset);
    else
        range_scan_kernel<false><<<blocks, kScanThreads, 0, st>>>(a, tau, list, nlist_dev, nlist_max, g.tile_rows, g.ntiles, tile_counts,
                                                                   count, lims, base, D, I, id_offset);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

int launch_range_offsets(const int32_t* count, int n, int64_t* lims, cudaStream_t st) {
    if (n > 1024) {
        set_error("range offsets: %d queries in one chunk (at most 1024)", n);
        return B2F_EINVAL;
    }
    range_offsets_kernel<<<1, 1024, 0, st>>>(count, n, lims);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

int launch_range_emit(const float* skey, const int32_t* sid, const int32_t* staged, const int64_t* lims, int nq, int64_t base, int metric,
                      float* D, int64_t* I, int64_t id_offset, cudaStream_t st) {
    if (nq <= 0) return B2F_OK;
    range_emit_kernel<<<nq, 256, 0, st>>>(skey, sid, staged, lims, base, metric == B2F_METRIC_L2 ? 1 : 0, D, I, id_offset);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

}  // namespace b2f
