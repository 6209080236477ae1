// remove.cuh -- row removal (index.remove_ids): the run list, where each row goes, the compaction's tiles (host and
// device), and the launchers.  Kept out of common.cuh so that the search kernels' translation units do not change.
#pragma once
#include <vector>

#include "common.cuh"

namespace b2f {

// ---- row removal (index.remove_ids; remove.cu) ---------------------------------------------------------------------
// The rows one removal takes out: sorted disjoint runs [start[j], end[j]), j < nruns; cum[j] = rows in runs 0..j-1
// (cum[nruns]: all of them).  One device (or host) array holds start, end and cum in that order.
struct RemoveRuns {
    const int64_t* start;
    const int64_t* end;
    const int64_t* cum;
    int64_t nruns;
};
// first j in [lo, hi) with v[j] > x (strict) or >= x, else hi
__host__ __device__ inline int64_t remove_search(const int64_t* v, int64_t x, int64_t lo, int64_t hi, bool strict) {
    while (lo < hi) {
        const int64_t m = (lo + hi) >> 1;
        if (strict ? v[m] <= x : v[m] < x) lo = m + 1;
        else hi = m;
    }
    return lo;
}
// removed rows below row x
__host__ __device__ inline int64_t removed_before(const RemoveRuns& r, int64_t x) {
    const int64_t j = remove_search(r.start, x, 0, r.nruns, false);   // runs 0..j-1 start below x
    if (j == 0) return 0;
    const int64_t e = r.end[j - 1] < x ? r.end[j - 1] : x;
    return r.cum[j - 1] + e - r.start[j - 1];
}
// Where row s goes: its new row number, or -1 when it is removed.  [lo, hi): runs known to hold every run that starts at
// or below s and ends above it (the whole list: 0, nruns); every run below lo ends at or below s.
__host__ __device__ inline int64_t remove_dest(const RemoveRuns& r, int64_t s, int64_t lo, int64_t hi) {
    const int64_t j = remove_search(r.start, s, lo, hi, true);   // runs 0..j-1 start at or below s
    if (j > 0 && s < r.end[j - 1]) return -1;
    return s - r.cum[j];
}
// Tile t of the compaction: source rows [s0, s1) of [first, ntotal) in tiles of tile_rows rows.  Its survivors land on
// [dlo, dhi) in order; before storing there it waits for tiles [w0, w1) -- every tile whose source rows meet [dlo, dhi),
// all below t -- to have read their rows.  Runs [j0, j1) are those that meet [s0, s1).
struct RemoveSpan {
    int64_t s0, s1, dlo, dhi, w0, w1, j0, j1;
};
__host__ __device__ inline RemoveSpan remove_tile_span(const RemoveRuns& r, int64_t first, int64_t ntotal, int64_t tile_rows, int64_t t) {
    RemoveSpan sp;
    sp.s0 = first + t * tile_rows;
    sp.s1 = sp.s0 + tile_rows < ntotal ? sp.s0 + tile_rows : ntotal;
    sp.dlo = sp.s0 - removed_before(r, sp.s0);
    sp.dhi = sp.s1 - removed_before(r, sp.s1);
    sp.j0 = remove_search(r.end, sp.s0, 0, r.nruns, true);   // first run that ends above s0
    sp.j1 = remove_search(r.start, sp.s1, sp.j0, r.nruns, false);   // first run that starts at or above s1
    sp.w0 = sp.w1 = t;
    if (sp.dhi > sp.dlo) {   // no row moves up, and every removed row is at or above first: first <= dlo <= s0
        sp.w0 = (sp.dlo - first) / tile_rows;
        const int64_t last = (sp.dhi - 1 - first) / tile_rows + 1;
        sp.w1 = last < t ? last : t;
    }
    return sp;
}
constexpr int64_t kRemoveTileBytes = 32 << 10;   // shared memory a tile's rows take (a row of more: one row per tile)
int64_t remove_tile_rows(int64_t row_bytes);
// tiles of the compaction of [first, ntotal) for rows of row_bytes bytes
inline int64_t remove_tiles(int64_t first, int64_t ntotal, int64_t row_bytes) {
    const int64_t tr = remove_tile_rows(row_bytes);
    return ntotal > first ? (ntotal - first + tr - 1) / tr : 0;
}
// Compacts the rows (row_bytes each, a multiple of 4) of [first, ntotal) of the array at base in place: survivors move to
// remove_dest.  spans: device scratch for remove_tiles(...) spans; flags: 1 + remove_tiles(...) words, word 0 the tile
// ticket; epoch: a value no earlier launch on these flags used.  Two launches on st, the second cooperative.
int launch_remove_compact(void* base, int64_t row_bytes, const RemoveRuns& runs, int64_t first, int64_t ntotal, RemoveSpan* spans,
                          uint32_t* flags, uint32_t epoch, cudaStream_t st);
// stats[0..1] = max over rows [0, n) of a bf16-storage scan copy, as ingest_kernel computes them (stats zeroed first)
int launch_scan_stats(const __nv_bfloat16* scan, int64_t n, int d, int64_t dpad, const float* mu, float* stats, cudaStream_t st);

// ids (any order; duplicates and ids outside [0, ntotal) ignored) -> sorted disjoint runs, flattened (a0, b0, a1, b1, ...)
std::vector<int64_t> remove_runs_from_ids(int64_t ntotal, int64_t n, const int64_t* ids);
// flattened runs -> the one-array layout of RemoveRuns (start, end, cum), and a view of such an array
void remove_runs_layout(const std::vector<int64_t>& runs, std::vector<int64_t>& words);
RemoveRuns remove_runs_view(const int64_t* words, int64_t nruns);

}  // namespace b2f
