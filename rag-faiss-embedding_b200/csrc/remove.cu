// remove.cu -- row removal (index.remove_ids): the surviving rows of the three row arrays (fp32 rows, bf16 scan copy,
// norms) compacted in place in one pass.  (The certification stats over the survivors: ingest.cu.)
//
// The rows a call removes are sorted disjoint runs [start_j, end_j) (RemoveRuns).  Rows below the first run stay where
// they are; survivor s above it moves down to s - removed_before(s).  The moved region [first, ntotal) is cut into tiles
// of whole source rows, which CTAs take by ticket, in increasing order.  Per tile: the survivors are loaded into shared
// memory (compacted), "read" is published with a release flag, the CTA waits (acquire) for every tile whose source rows
// its destination overlaps -- all lower-numbered, since no row moves up -- and stores.  Every moved byte is read once and
// written once, and no second copy of the database is ever held.
#include <algorithm>
#include <vector>

#include "remove.cuh"

namespace b2f {

constexpr int kRemoveThreads = 256;
constexpr int kLoadBatch = 4;

int64_t remove_tile_rows(int64_t row_bytes) {
    const int64_t r = kRemoveTileBytes / (row_bytes > 0 ? row_bytes : 1);
    return r > 0 ? r : 1;
}

__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Every tile's span, one thread per tile, ahead of the compaction: its four binary searches over the run list are
// dependent loads that would otherwise sit on each tile's critical path.
__global__ void __launch_bounds__(256)
remove_spans_kernel(RemoveRuns runs, int64_t first, int64_t ntotal, int64_t tile_rows, int64_t ntiles, RemoveSpan* __restrict__ spans) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < ntiles) spans[t] = remove_tile_span(runs, first, ntotal, tile_rows, t);
}

// V: uint4 for rows of a multiple of 16 bytes (16-byte accesses), else uint32_t.  base: the array as 32-bit words, rw
// words per row.  flags[0]: the ticket counter (zero at launch); flags[1 + t]: tile t has been read when it equals epoch.
template <typename V>
__global__ void __launch_bounds__(kRemoveThreads, 4)
remove_compact_kernel(uint32_t* __restrict__ base, int rw, int tile_rows, RemoveRuns runs, const RemoveSpan* __restrict__ spans, int64_t ntiles,
                      uint32_t* __restrict__ flags, uint32_t epoch) {
    extern __shared__ __align__(16) unsigned char smem[];
    int32_t* slot = reinterpret_cast<int32_t*>(smem);                                  // [tile_rows]: compacted row, -1 removed
    V* buf = reinterpret_cast<V*>(smem + (((size_t)tile_rows * 4 + 15) & ~(size_t)15));  // [tile_rows][rw] compacted survivors
    __shared__ int64_t s_t;
    __shared__ RemoveSpan s_sp;
    constexpr int kVw = (int)(sizeof(V) / 4);
    const int rv = rw / kVw;   // vectors per row
    for (;;) {
        if (threadIdx.x == 0) {
            s_t = (int64_t)atomicAdd(flags, 1u);
            if (s_t < ntiles) s_sp = spans[s_t];
        }
        __syncthreads();
        const int64_t t = s_t;
        if (t >= ntiles) break;
        const RemoveSpan sp = s_sp;
        const int rows = (int)(sp.s1 - sp.s0);
        // where each source row of the tile goes in the compacted tile (the runs that touch this tile: [j0, j1))
        for (int i = threadIdx.x; i < rows; i += blockDim.x) {
            const int64_t to = remove_dest(runs, sp.s0 + i, sp.j0, sp.j1);
            slot[i] = to < 0 ? -1 : (int32_t)(to - sp.dlo);
        }
        __syncthreads();
        const V* src = reinterpret_cast<const V*>(base + sp.s0 * rw);
        const int nv = rows * rv;
        for (int v0 = threadIdx.x; v0 < nv; v0 += kLoadBatch * kRemoveThreads) {
            // kLoadBatch loads in flight per thread before any lands in shared memory
            V r[kLoadBatch];
            int to[kLoadBatch];
#pragma unroll
            for (int u = 0; u < kLoadBatch; u++) {
                const int v = v0 + u * kRemoveThreads;
                to[u] = -1;
                if (v < nv) {
                    const int i = v / rv;
                    const int sl = slot[i];
                    if (sl >= 0) {
                        to[u] = sl * rv + (v - i * rv);
                        r[u] = __ldcg(src + v);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < kLoadBatch; u++)
                if (to[u] >= 0) buf[to[u]] = r[u];
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            st_release_gpu(flags + 1 + t, epoch);
            // Forward progress: a CTA waits only after it has read and published its own tile, and only for lower tiles.
            // Tickets go out in increasing order to running CTAs, so every lower tile is held by a running CTA that either
            // has published it or is reading it -- and reading never waits.  The lowest unpublished tile therefore always
            // completes, and no cycle of waits can form.
            for (int64_t u = sp.w0; u < sp.w1; u++)
                while (ld_acquire_gpu(flags + 1 + u) != epoch) __nanosleep(64);
        }
        __syncthreads();
        V* dst = reinterpret_cast<V*>(base + sp.dlo * rw);
        const int nst = (int)(sp.dhi - sp.dlo) * rv;
        for (int v = threadIdx.x; v < nst; v += blockDim.x) __stcg(dst + v, buf[v]);
        __syncthreads();   // slot / buf are reused by the next tile
    }
}

int launch_remove_compact(void* base, int64_t row_bytes, const RemoveRuns& runs, int64_t first, int64_t ntotal, RemoveSpan* spans,
                          uint32_t* flags, uint32_t epoch, cudaStream_t st) {
    if (ntotal <= first) return B2F_OK;
    if (row_bytes % 4 != 0) {
        set_error("remove: rows of %lld bytes are not whole 32-bit words", (long long)row_bytes);
        return B2F_EINVAL;
    }
    const int64_t tile_rows = remove_tile_rows(row_bytes);
    const int64_t ntiles = (ntotal - first + tile_rows - 1) / tile_rows;
    const int rw = (int)(row_bytes / 4);
    const bool vec = rw % 4 == 0;
    const size_t smem = (((size_t)tile_rows * 4 + 15) & ~(size_t)15) + (size_t)tile_rows * row_bytes;
    const void* kern = vec ? (const void*)remove_compact_kernel<uint4> : (const void*)remove_compact_kernel<uint32_t>;
    int occ = 0;
    {
        static size_t configured[2][kMaxDevices] = {};
        const int dev = current_device_slot();
        std::lock_guard<std::mutex> lk(launch_cache_mutex());
        if (smem > 48 * 1024 && smem > configured[vec][dev]) {
            B2F_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            configured[vec][dev] = smem;
        }
    }
    B2F_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kRemoveThreads, smem));
    if (occ < 1) {
        set_error("remove: compaction kernel does not fit (%zu bytes of shared memory)", smem);
        return B2F_EINVAL;
    }
    const int64_t grid = std::min<int64_t>(ntiles, (int64_t)kNumSMs * occ);
    B2F_CUDA(cudaMemsetAsync(flags, 0, 4, st));
    remove_spans_kernel<<<(unsigned)((ntiles + 255) / 256), 256, 0, st>>>(runs, first, ntotal, tile_rows, ntiles, spans);
    B2F_CUDA(cudaGetLastError());
    uint32_t* base_ = static_cast<uint32_t*>(base);
    int rw_ = rw, tr_ = (int)tile_rows;
    RemoveRuns runs_ = runs;
    const RemoveSpan* spans_ = spans;
    int64_t ntiles_ = ntiles;
    uint32_t* flags_ = flags;
    uint32_t epoch_ = epoch;
    void* args[] = {(void*)&base_, (void*)&rw_, (void*)&tr_, (void*)&runs_, (void*)&spans_, (void*)&ntiles_, (void*)&flags_, (void*)&epoch_};
    // cooperative, as K1: the whole grid is resident (the waits need it only for tickets already taken, which running CTAs hold)
    B2F_CUDA(cudaLaunchCooperativeKernel(kern, dim3((unsigned)grid), dim3(kRemoveThreads), args, smem, st));
    return B2F_OK;
}

// ids (any order) -> sorted disjoint runs [a, b) of the rows in [0, ntotal) they name, flattened (a0, b0, a1, b1, ...)
std::vector<int64_t> remove_runs_from_ids(int64_t ntotal, int64_t n, const int64_t* ids) {
    std::vector<int64_t> v;
    v.reserve((size_t)n);
    for (int64_t i = 0; i < n; i++)
        if (ids[i] >= 0 && ids[i] < ntotal) v.push_back(ids[i]);
    std::sort(v.begin(), v.end());
    std::vector<int64_t> runs;
    for (size_t i = 0; i < v.size();) {
        size_t j = i + 1;
        while (j < v.size() && v[j] <= v[j - 1] + 1) j++;   // duplicates and neighbours extend the run
        runs.push_back(v[i]);
        runs.push_back(v[j - 1] + 1);
        i = j;
    }
    return runs;
}

// flattened runs -> the RemoveRuns layout in `words` (start [nruns], end [nruns], cum [nruns + 1])
void remove_runs_layout(const std::vector<int64_t>& runs, std::vector<int64_t>& words) {
    const size_t nr = runs.size() / 2;
    words.assign(3 * nr + 1, 0);
    for (size_t j = 0; j < nr; j++) {
        words[j] = runs[2 * j];
        words[nr + j] = runs[2 * j + 1];
        words[2 * nr + j + 1] = words[2 * nr + j] + runs[2 * j + 1] - runs[2 * j];
    }
}

RemoveRuns remove_runs_view(const int64_t* words, int64_t nruns) {
    RemoveRuns r;
    r.start = words;
    r.end = words + nruns;
    r.cum = words + 2 * nruns;
    r.nruns = nruns;
    return r;
}

}  // namespace b2f
