// filter.cu -- filtered search (faiss ID selectors): the per-call allow bitmap and the masked row bias.
//
// A row r is searched when the selector contains its label r + id_offset.  The bitmap holds one bit per row,
// ceil(ntotal / 32) words.  K1 and the exact range scan test it directly.  The tensor pass (K2) is not changed: it
// reads each row's bias from a copy of the norms in which every excluded row's bias is NaN, and a NaN key fails every
// threshold comparison K2 makes, so an excluded row is never listed (DESIGN §3.7).
#include "common.cuh"

namespace b2f {

namespace {

constexpr int kFilterThreads = 256;

// RANGE and BITMAP: every word from the selector; BATCH: the start value of the scatter (0, or all ones under Not).
// win [hi - lo]: the bitmap's bytes lo .. hi - 1 (label i is bit i & 7 of byte i >> 3).
__global__ void __launch_bounds__(kFilterThreads)
allow_fill_kernel(int kind, int negate, int64_t imin, int64_t imax, const uint8_t* __restrict__ win, int64_t lo, int64_t hi,
                  int64_t id_offset, int64_t ntotal, int64_t nwords, uint32_t* __restrict__ allow) {
    for (int64_t w = (int64_t)blockIdx.x * kFilterThreads + threadIdx.x; w < nwords; w += (int64_t)gridDim.x * kFilterThreads) {
        uint32_t m = 0;
        if (kind == B2F_SEL_BATCH) {
            m = negate ? 0xffffffffu : 0u;
        } else {
            for (int b = 0; b < 32; b++) {
                const int64_t label = w * 32 + b + id_offset;
                bool in;
                if (kind == B2F_SEL_RANGE) {
                    in = imin <= label && label < imax;
                } else {
                    const int64_t byte = label >= 0 ? label >> 3 : -1;
                    in = byte >= lo && byte < hi && ((win[byte - lo] >> (label & 7)) & 1);
                }
                m |= (uint32_t)(in != (negate != 0)) << b;
            }
        }
        const int64_t valid = ntotal - w * 32;   // rows past the end stay clear
        if (valid < 32) m &= (1u << valid) - 1u;
        allow[w] = m;
    }
}

// BATCH: each id names the row id - id_offset; ids with no row are never matched, duplicates set the same bit
__global__ void __launch_bounds__(kFilterThreads)
allow_scatter_kernel(const int64_t* __restrict__ ids, int64_t n, int64_t id_offset, int64_t ntotal, int negate,
                     uint32_t* __restrict__ allow) {
    for (int64_t i = (int64_t)blockIdx.x * kFilterThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kFilterThreads) {
        const int64_t id = ids[i];
        if (id < 0) continue;
        const int64_t r = id - id_offset;
        if (r < 0 || r >= ntotal) continue;
        const uint32_t bit = 1u << (r & 31);
        if (negate) atomicAnd(allow + (r >> 5), ~bit);
        else atomicOr(allow + (r >> 5), bit);
    }
}

__global__ void __launch_bounds__(kFilterThreads)
masked_bias_kernel(const float* __restrict__ norms, const uint32_t* __restrict__ allow, int64_t ntotal, float* __restrict__ bias) {
    for (int64_t r = (int64_t)blockIdx.x * kFilterThreads + threadIdx.x; r < ntotal; r += (int64_t)gridDim.x * kFilterThreads)
        bias[r] = ((allow[r >> 5] >> (r & 31)) & 1) ? norms[r] : __int_as_float(0x7fffffff);
}

int grid_for(int64_t items) {
    const int64_t b = (items + kFilterThreads - 1) / kFilterThreads;
    const int64_t cap = (int64_t)kNumSMs * 8;
    return (int)(b < 1 ? 1 : (b < cap ? b : cap));
}

}  // namespace

int check_selector(const b2f_selector* sel) {
    if (!sel) return B2F_OK;
    if (sel->kind != B2F_SEL_RANGE && sel->kind != B2F_SEL_BATCH && sel->kind != B2F_SEL_BITMAP) {
        set_error("selector: unknown kind %d", (int)sel->kind);
        return B2F_EINVAL;
    }
    if (sel->kind != B2F_SEL_RANGE && (sel->n < 0 || (sel->n > 0 && !sel->data))) {
        set_error("selector: n = %lld with data %p", (long long)sel->n, sel->data);
        return B2F_EINVAL;
    }
    return B2F_OK;
}

FilterWindow filter_window(const b2f_selector& sel, int64_t ntotal, int64_t id_offset) {
    FilterWindow w{0, 0};
    if (sel.kind == B2F_SEL_BATCH) {
        w.hi = sel.n;
    } else if (sel.kind == B2F_SEL_BITMAP && ntotal > 0) {
        // the bytes that hold the labels id_offset .. id_offset + ntotal - 1, clipped to the bitmap
        const int64_t first = id_offset > 0 ? id_offset : 0, last = id_offset + ntotal - 1;
        if (last >= 0) {
            w.lo = first >> 3 < sel.n ? first >> 3 : sel.n;
            w.hi = (last >> 3) + 1 < sel.n ? (last >> 3) + 1 : sel.n;
        }
    }
    return w;
}

size_t filter_staged_bytes(const b2f_selector& sel, int64_t ntotal, int64_t id_offset) {
    const FilterWindow w = filter_window(sel, ntotal, id_offset);
    return (size_t)(w.hi - w.lo) * (sel.kind == B2F_SEL_BATCH ? 8 : 1);
}

int launch_allow_bitmap(const b2f_selector& sel, int32_t mem, int64_t ntotal, int64_t id_offset, void* staged, uint32_t* allow,
                        cudaStream_t st) {
    if (ntotal <= 0) return B2F_OK;
    const FilterWindow w = filter_window(sel, ntotal, id_offset);
    const size_t esize = sel.kind == B2F_SEL_BATCH ? 8 : 1;
    const char* data = static_cast<const char*>(sel.data) + (size_t)w.lo * esize;
    if (w.hi > w.lo && mem == B2F_MEM_HOST) {
        B2F_CUDA(cudaMemcpyAsync(staged, data, (size_t)(w.hi - w.lo) * esize, cudaMemcpyHostToDevice, st));
        data = static_cast<const char*>(staged);
    }
    const int64_t nwords = (ntotal + 31) / 32;
    allow_fill_kernel<<<grid_for(nwords), kFilterThreads, 0, st>>>(sel.kind, sel.negate != 0, sel.imin, sel.imax,
                                                                   reinterpret_cast<const uint8_t*>(data), w.lo, w.hi,
                                                                   id_offset, ntotal, nwords, allow);
    B2F_CUDA(cudaGetLastError());
    if (sel.kind == B2F_SEL_BATCH && w.hi > 0) {
        allow_scatter_kernel<<<grid_for(w.hi), kFilterThreads, 0, st>>>(reinterpret_cast<const int64_t*>(data), w.hi, id_offset,
                                                                        ntotal, sel.negate != 0, allow);
        B2F_CUDA(cudaGetLastError());
    }
    return B2F_OK;
}

int launch_masked_bias(const float* norms, const uint32_t* allow, int64_t ntotal, float* bias, cudaStream_t st) {
    if (ntotal <= 0) return B2F_OK;
    masked_bias_kernel<<<grid_for(ntotal), kFilterThreads, 0, st>>>(norms, allow, ntotal, bias);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

}  // namespace b2f
