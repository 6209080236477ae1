// index.cu -- host side of the C ABI (include/b200flat.h): device storage, ingest, the search
// pipelines (K1 scan | K2 tensor scan -> K3 merge -> K4 re-rank -> finalize), FAISS-compatible
// file I/O.  No CPU compute path exists here: without a usable sm_100 device every compute entry
// point returns B2F_ENOGPU.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <new>
#include <vector>

#include "remove.cuh"

namespace b2f {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

std::mutex& launch_cache_mutex() {
    static std::mutex m;
    return m;
}

}  // namespace b2f

using namespace b2f;

// What searches teach an index about its data.  It goes with the data: b2f_index_reset starts it over.
struct Adapt {
    int slack_boost = 0;           // extra candidates per query, raised when too many queries fail certification
    bool range_mode = false;       // earlier batches left many queries uncertified: run the range pass (one host sync per search)
    int32_t range_ran_seq = 0;     // the search (sequence number) whose range pass served range_ran_nfail queries
    int range_ran_nfail = 0;
    int range_futile = 0;          // consecutive range passes that left most of their queries to the exact scan anyway
    int range_ban = 0;             // searches to wait before the range pass may be switched on again
    int range_quiet = 0;           // consecutive range-mode searches whose first pass certified everything
    // Order-robust mode.  A batch whose candidate lists overflowed en masse (rows stored so that a query's best rows sit in
    // one or two lists: the shared thresholds never tighten) switches the index to per-thread heaps for the first pass
    // (plan_tensor_scan's force_heap) plus the range pass for what the heaps cannot certify; LIST mode is tried again after
    // heap_span searches, and the span doubles every time it fails again.
    int heap_left = 0;             // searches still to run in this mode
    int heap_span = 64;

    // Folds in what finished search s counted: c0 uncertified queries, c1 of them with an overflowed list, of a batch of nqb.
    void learn(int32_t s, int c0, int c1, int nqb, int certify) {
        // The slack that certification needs grows with the neighbour density at rank k (i.e. with the database
        // size and the data distribution): when too many queries of a batch had to fall back, keep more candidates
        // per query from now on.  "Too many" is where the exact scans cost more than the wider tensor pass would: the
        // fallback walks the database once per four queries (F / 4 x n d 4 B at ~5.5 TB/s) while the batch's tensor
        // pass costs 2 nq n d flop at ~1.3 PFLOP/s and grows by < 10 % with 32 more candidates -- break-even at
        // F ~ nq / 1200; the boost waits for 0.5 % because the range pass below is cheaper still.  (Round 1 waited for 2 % of
        // the batch: BASELINE config 5 on 2 GPUs spent 9 of its 34 ms per search in exact scans for 0.5 % of the queries.)
        if (certify && c0 - c1 > (nqb / 200 > 2 ? nqb / 200 : 2) && slack_boost < 224) slack_boost += 32;
        // Well before that (F > nq / 1000) the range pass takes over: a second TENSOR pass over the uncertified queries with a
        // fixed threshold per query, one database pass for all of them instead of one exact scan per four (range_pass).
        // ... unless it does not help: neighbourhoods so dense that the fixed-threshold lists overflow too (thousands of
        // near-duplicates) leave its queries to the exact scan anyway; two such searches in a row switch it off for a while.
        if (range_ban > 0) range_ban--;
        if (range_mode && range_ran_seq == s) {
            if (2 * c0 > range_ran_nfail) {
                if (++range_futile >= 2) {
                    range_mode = false;
                    range_futile = 0;
                    range_ban = 256;
                }
            } else {
                range_futile = 0;
            }
        }
        if (certify && c1 > (nqb / 8 > 8 ? nqb / 8 : 8) && heap_left == 0) {
            heap_left = heap_span;
            if (heap_span < 4096) heap_span *= 2;
            if (range_ban == 0) {
                range_mode = true;   // the heaps find the k' best whatever the row order; dense neighbourhoods still need the range pass
                range_quiet = 0;
            }
        }
        if (certify && !range_mode && range_ban == 0 && c0 - c1 > (nqb / 1000 > 2 ? nqb / 1000 : 2)) {
            range_mode = true;
            range_quiet = 0;
        }
    }
    // A range-mode search whose first pass left nfail queries uncertified
    void first_pass_failed(int nfail) {
        if (nfail == 0) {
            if (++range_quiet >= 8) range_mode = false;   // the data (or the adaptive slack) no longer needs it
        } else {
            range_quiet = 0;
        }
    }
};

struct b2f_index {
    int d = 0, metric = 1, storage = 0, device = 0;
    int64_t ntotal = 0, cap = 0, dpad = 0;
    float* rows_f32 = nullptr;        // [cap, d]      authoritative rows (B2F_STORE_F32)
    __nv_bfloat16* scan = nullptr;    // [cap, dpad]   bf16 scan copy (authoritative for B2F_STORE_BF16)
    float* norms = nullptr;           // [cap]         |bf16 row|^2 in fp32
    float* stats = nullptr;           // [2] device    max |x~|^2, max |x - x~|^2
    cudaStream_t stream = nullptr;
    char* ws = nullptr;               // device workspace (grow only)
    size_t ws_bytes = 0;
    char* pinned = nullptr;           // host staging
    size_t pinned_bytes = 0;
    std::vector<cudaEvent_t> ev;      // profiling events
    std::mutex mu;
    b2f_stats st{};
    float host_stats[2] = {0.f, 0.f};
    bool stats_dirty = true;
    float* qpool = nullptr;           // pooled query batch of search_pooled (grow only)
    size_t qpool_bytes = 0;
    float* centre = nullptr;          // [d] device: centre of the scan copy (fp32 storage; see ingest_kernel), fixed at the first add
    bool mu_set = false;
    float mu_norm = 0.f;              // |mu| (host copy, refreshed with host_stats)
    int32_t* host_flag = nullptr;     // mapped pinned memory [16]: counters of the latest finished tensor-path search + its seq
    int32_t seq = 0;
    uint32_t scan_launches = 0;       // launch parity of the scan's cross-CTA bounds
    int32_t harvested_seq = 0;        // last seq whose counters were folded into the host-side statistics
    Adapt adapt;
    unsigned long long* totals = nullptr;  // device [4]: fallback queries, overflowed queries, rescued queries (running totals)
    cudaEvent_t ev_done = nullptr;    // recorded at the end of every search (searches return without synchronising)
    cudaStream_t last_stream = nullptr;
    bool search_recorded = false;
    cudaEvent_t ev_ingest = nullptr;  // recorded behind every add (and removal) on the stream it was enqueued on
    cudaStream_t last_add_stream = nullptr;
    bool add_recorded = false;
    uint32_t* rm_flags = nullptr;     // device, grow-only, zeroed once: the compaction's ticket + per-tile "read" flags
    int64_t rm_flag_words = 0;
    uint32_t rm_epoch = 0;            // the flag value of the latest compaction launch (one new value per launch)
    // profiling: a ring of event sets so that timing never forces a host synchronisation inside a search
    struct ProfSlot {
        cudaEvent_t t0 = nullptr, t1 = nullptr;
        std::vector<cudaEvent_t> m;   // 2 per launch of the dominant kernel
        int n_main = 0;
        bool pending = false;
    };
    static constexpr int kProfSlots = 16;
    ProfSlot prof[kProfSlots];
    int prof_head = 0;
};

namespace {

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

int check_device(int device) {
    // cached: cudaGetDeviceProperties costs milliseconds and this runs on per-search entry points
    static std::mutex cache_mu;   // indexes on several devices may be created from several threads
    static int cached_count = -1;
    static int cached_major[64];
    std::lock_guard<std::mutex> cache_lk(cache_mu);
    if (cached_count < 0) {
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if (e != cudaSuccess || n <= 0) {
            cudaGetLastError();
            set_error("no CUDA device available (%s); this engine has no CPU path", e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
            return B2F_ENOGPU;
        }
        if (n > 64) n = 64;
        for (int i = 0; i < n; i++) {
            int major = 0;
            if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) != cudaSuccess) {
                cudaGetLastError();
                major = 0;
            }
            cached_major[i] = major;
        }
        cached_count = n;
    }
    if (device < 0 || device >= cached_count) {
        set_error("device %d out of range [0,%d)", device, cached_count);
        return B2F_EINVAL;
    }
    if (cached_major[device] != 10) {
        set_error("device %d is not sm_100 (Blackwell B200); kernels are built for sm_100a only", device);
        return B2F_ENOGPU;
    }
    return B2F_OK;
}

// Bump allocator over the index workspace of `size` bytes.  Over a null base it only measures: the same carve that lays
// the buffers out then gives the bytes they need.  A carve that passes the end leaves fits() false.
struct Bump {
    char* base;
    size_t size;
    size_t off = 0;
    Bump(char* b, size_t n) : base(b), size(n) {}
    template <typename T>
    T* take(size_t count) {
        off = align_up(off, 256);
        T* p = reinterpret_cast<T*>(reinterpret_cast<uintptr_t>(base) + off);
        off += count * sizeof(T);
        return p;
    }
    bool fits() const { return off <= size; }
};

// rows of d floats that fit `bytes` (at least one)
int64_t rows_in(size_t bytes, int d) {
    const int64_t r = (int64_t)(bytes / ((size_t)d * 4));
    return r > 0 ? r : 1;
}

int ensure_ws(b2f_index* ix, size_t bytes) {
    if (bytes <= ix->ws_bytes) return B2F_OK;
    if (ix->ws) {
        B2F_CUDA(cudaStreamSynchronize(ix->stream));
        B2F_CUDA(cudaDeviceSynchronize());
        B2F_CUDA(cudaFree(ix->ws));
        ix->ws = nullptr;
        ix->ws_bytes = 0;
    }
    bytes = align_up(bytes + (bytes >> 2), 1 << 20);
    cudaError_t e = cudaMalloc(&ix->ws, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("workspace cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
        return B2F_ENOMEM;
    }
    ix->ws_bytes = bytes;
    return B2F_OK;
}

int ensure_pinned(b2f_index* ix, size_t bytes) {
    if (bytes <= ix->pinned_bytes) return B2F_OK;
    if (ix->pinned) {
        B2F_CUDA(cudaStreamSynchronize(ix->stream));
        B2F_CUDA(cudaFreeHost(ix->pinned));
        ix->pinned = nullptr;
        ix->pinned_bytes = 0;
    }
    cudaError_t e = cudaMallocHost(&ix->pinned, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(e));
        return B2F_ENOMEM;
    }
    ix->pinned_bytes = bytes;
    return B2F_OK;
}

// Lays one call's buffers out in the workspace.  carve(Bump&) takes them in one fixed order: over a null base it measures
// them, then the workspace grows to max(measured, min_bytes) bytes and the same carve lays them out there.  *grew: a
// workspace the call found had to be replaced (which waits for the device).
template <class Carve>
int carve_ws(b2f_index* ix, size_t min_bytes, Carve&& carve, const char* what, bool* grew = nullptr) {
    Bump layout(nullptr, SIZE_MAX);
    carve(layout);
    const size_t need = std::max(layout.off, min_bytes);
    if (grew) *grew = need > ix->ws_bytes && ix->ws;
    B2F_TRY(ensure_ws(ix, need));
    Bump bump(ix->ws, ix->ws_bytes);
    carve(bump);
    if (!bump.fits()) {
        set_error("%s workspace: the layout needs %zu bytes, the workspace has %zu", what, bump.off, bump.size);
        return B2F_ECUDA;
    }
    return B2F_OK;
}

// The centre of the scan copy (either storage; null before the first add): what ingest subtracts from a row and the query
// preparation from a query before the bf16 rounding, and what bf16 storage adds back to a stored row.
const float* scan_centre(const b2f_index* ix) { return ix->mu_set ? ix->centre : nullptr; }

// The rows as the exact kernels read them.  Their centre is the one added back to a stored bf16 row: bf16 storage only.
StoredRows stored_rows(const b2f_index* ix) {
    const bool f32 = ix->storage == B2F_STORE_F32;
    return StoredRows{f32 ? ix->rows_f32 : nullptr, ix->scan, ix->dpad, f32 ? nullptr : scan_centre(ix), ix->ntotal, ix->d, ix->metric};
}

// kernel launches of a search: the running total and the latest search's count
void count_launches(b2f_index* ix, int n) {
    ix->st.launches += n;
    ix->st.last_launches += n;
}

// Adds are enqueued on the caller's stream (a device-tensor add / add_pooled runs behind the encoder on torch's
// stream) and return without synchronising.  Everything that reads rows, norms, stats or the centre on ANOTHER
// stream -- searches, write, reconstruct, the stats refresh, the growth copies -- first waits for the latest add.
int wait_ingest(b2f_index* ix, cudaStream_t st) {
    if (ix->add_recorded && ix->last_add_stream != st) B2F_CUDA(cudaStreamWaitEvent(st, ix->ev_ingest, 0));
    return B2F_OK;
}
int record_ingest(b2f_index* ix, cudaStream_t st) {
    if (!ix->ev_ingest) B2F_CUDA(cudaEventCreateWithFlags(&ix->ev_ingest, cudaEventDisableTiming));
    // an add on a new stream is ordered behind the previous add (both write stats / may share the workspace)
    B2F_CUDA(cudaEventRecord(ix->ev_ingest, st));
    ix->last_add_stream = st;
    ix->add_recorded = true;
    return B2F_OK;
}
// recorded behind every search and range search on the stream it was enqueued on (they return without synchronising)
int record_search(b2f_index* ix, cudaStream_t st) {
    if (!ix->ev_done) B2F_CUDA(cudaEventCreateWithFlags(&ix->ev_done, cudaEventDisableTiming));
    B2F_CUDA(cudaEventRecord(ix->ev_done, st));
    ix->last_stream = st;
    ix->search_recorded = true;
    return B2F_OK;
}

// The start of every entry point that works on the index's buffers from stream st: the device must be usable, a search
// still running on another stream must be done with the workspace (searches return without synchronising), and the
// latest add must have landed.
int enter_stream(b2f_index* ix, const DeviceGuard& g, cudaStream_t st) {
    if (!g.ok) {
        set_error("cudaSetDevice(%d) failed", ix->device);
        return B2F_ENOGPU;
    }
    if (ix->search_recorded && ix->last_stream != st) B2F_CUDA(cudaStreamWaitEvent(st, ix->ev_done, 0));
    return wait_ingest(ix, st);
}

int ensure_capacity(b2f_index* ix, int64_t need) {
    if (need <= ix->cap) return B2F_OK;
    if (need > (int64_t)INT32_MAX - 64) {
        set_error("a single index holds at most 2^31-65 rows (row-shard across GPUs beyond that)");
        return B2F_EINVAL;
    }
    int64_t ncap = ix->cap + ix->cap / 2;
    if (ncap < need) ncap = need;
    if (ncap < 1024) ncap = 1024;
    float* nrows = nullptr;
    __nv_bfloat16* nscan = nullptr;
    float* nnorm = nullptr;
    cudaError_t e = cudaSuccess;
    if (ix->storage == B2F_STORE_F32) e = cudaMalloc(&nrows, (size_t)ncap * ix->d * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&nscan, (size_t)ncap * ix->dpad * sizeof(__nv_bfloat16));
    if (e == cudaSuccess) e = cudaMalloc(&nnorm, (size_t)ncap * sizeof(float));
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaFree(nrows);
        cudaFree(nscan);
        cudaFree(nnorm);
        set_error("device allocation for %lld rows failed: %s", (long long)ncap, cudaGetErrorString(e));
        return B2F_ENOMEM;
    }
    if (ix->ntotal > 0) {
        // an ingest may still be pending on a caller stream (e.g. behind an encoder forward): its rows must have landed
        // before they are copied into the new buffers
        B2F_TRY(wait_ingest(ix, ix->stream));
        if (nrows) B2F_CUDA(cudaMemcpyAsync(nrows, ix->rows_f32, (size_t)ix->ntotal * ix->d * sizeof(float), cudaMemcpyDeviceToDevice, ix->stream));
        B2F_CUDA(cudaMemcpyAsync(nscan, ix->scan, (size_t)ix->ntotal * ix->dpad * sizeof(__nv_bfloat16), cudaMemcpyDeviceToDevice, ix->stream));
        B2F_CUDA(cudaMemcpyAsync(nnorm, ix->norms, (size_t)ix->ntotal * sizeof(float), cudaMemcpyDeviceToDevice, ix->stream));
    }
    B2F_CUDA(cudaStreamSynchronize(ix->stream));
    B2F_CUDA(cudaDeviceSynchronize());  // other streams may still be searching the old buffers
    cudaFree(ix->rows_f32);
    cudaFree(ix->scan);
    cudaFree(ix->norms);
    ix->rows_f32 = nrows;
    ix->scan = nscan;
    ix->norms = nnorm;
    ix->cap = ncap;
    ix->st.bytes_rows = nrows ? (int64_t)ncap * ix->d * 4 : (int64_t)ncap * ix->dpad * 2;
    ix->st.bytes_scan = (nrows ? (int64_t)ncap * ix->dpad * 2 : 0) + (int64_t)ncap * 4;
    return B2F_OK;
}

cudaEvent_t get_event(b2f_index* ix, size_t i) {
    while (ix->ev.size() <= i) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
        ix->ev.push_back(e);
    }
    return ix->ev[i];
}

int refresh_host_stats(b2f_index* ix, cudaStream_t st) {
    if (!ix->stats_dirty) return B2F_OK;
    B2F_CUDA(cudaMemcpyAsync(ix->host_stats, ix->stats, 2 * sizeof(float), cudaMemcpyDeviceToHost, st));
    std::vector<float> m((size_t)ix->d, 0.f);
    if (const float* mu = scan_centre(ix)) B2F_CUDA(cudaMemcpyAsync(m.data(), mu, (size_t)ix->d * sizeof(float), cudaMemcpyDeviceToHost, st));
    B2F_CUDA(cudaStreamSynchronize(st));
    double s2 = 0.0;
    for (float v : m) s2 += (double)v * v;
    ix->mu_norm = (float)(sqrt(s2) * (1.0 + 1e-6));
    ix->stats_dirty = false;
    return B2F_OK;
}

// make `st` wait for everything queued so far on the index's own stream (ingest) and vice versa
int order_after(cudaStream_t waiter, cudaStream_t producer, b2f_index* ix) {
    if (waiter == producer) return B2F_OK;
    cudaEvent_t e = get_event(ix, 0);
    if (!e) {
        set_error("cudaEventCreate failed");
        return B2F_ECUDA;
    }
    B2F_CUDA(cudaEventRecord(e, producer));
    B2F_CUDA(cudaStreamWaitEvent(waiter, e, 0));
    return B2F_OK;
}

// ---- K1: one cooperative launch (scan + merge + faiss formatting) for any number of queries ----------
// qsel / nsel_dev (optional, device): the list of query rows to process and its length -- the tensor path's
// uncertified queries, which the host never counts.  counters != null marks the closing kernel of a
// tensor-path search: it also publishes the search's counters.
int enqueue_scan(b2f_index* ix, const float* qd, const int32_t* qsel, const int32_t* nsel_dev, int nsel, int k, float* Dd,
                 int64_t* Id, int64_t id_offset, void* scratch, int32_t* counters, int32_t seq, int nq_batch, int certify,
                 const uint32_t* allow, cudaStream_t st) {
    ScanArgs a{};
    a.rows = stored_rows(ix);
    a.k = k;
    a.q = qd;
    a.qsel = qsel;
    a.nsel_dev = nsel_dev;
    a.nsel = nsel;
    a.D = Dd;
    a.I = Id;
    a.id_offset = id_offset;
    a.scratch = scratch;
    a.counters = counters;
    a.totals = counters ? ix->totals : nullptr;
    a.host_flag = counters ? ix->host_flag : nullptr;
    a.seq = seq;
    a.nq_batch = nq_batch;
    a.certify = certify;
    a.tub = reinterpret_cast<uint32_t*>(ix->totals + 4);
    a.parity = (int32_t)(ix->scan_launches++ & 1);
    a.allow = allow;
    B2F_TRY(launch_scan(a, st));
    count_launches(ix, 1);
    return B2F_OK;
}

// Folds the counters the latest finished tensor-path search left in mapped host memory into the host-side
// view (never blocks; a search that is still running is simply picked up later).
void harvest_flag(b2f_index* ix) {
    volatile int32_t* hf = ix->host_flag;
    const int32_t s = hf[4];
    if (s == 0 || s == ix->harvested_seq) return;
    std::atomic_thread_fence(std::memory_order_acquire);
    const int32_t c0 = hf[0], c1 = hf[1], c2 = hf[2], c3 = hf[3], nqb = hf[6], certify = hf[7];
    std::atomic_thread_fence(std::memory_order_acquire);
    if (hf[4] != s) return;  // a later search is publishing right now: take that one next time
    ix->harvested_seq = s;
    ix->st.last_list_entries = (int64_t)(((uint64_t)(uint32_t)c3 << 32) | (uint32_t)c2);
    ix->adapt.learn(s, c0, c1, nqb, certify);
}

void harvest_prof_slot(b2f_index* ix, b2f_index::ProfSlot& sl) {
    if (!sl.pending) return;
    sl.pending = false;
    if (cudaEventSynchronize(sl.t1) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    float ms = 0.f, tot = 0.f;
    for (int i = 0; i < sl.n_main; i++) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, sl.m[2 * (size_t)i], sl.m[2 * (size_t)i + 1]) == cudaSuccess) ms += t;
    }
    if (cudaEventElapsedTime(&tot, sl.t0, sl.t1) != cudaSuccess) tot = 0.f;
    cudaGetLastError();
    ix->st.last_main_ms = ms;
    ix->st.last_total_ms = tot;
    ix->st.last_main_launches = sl.n_main;
    ix->st.prof_main_ms_sum += ms;
    ix->st.prof_total_ms_sum += tot;
    ix->st.prof_main_launches += sl.n_main;
    ix->st.prof_searches += 1;
}

cudaEvent_t prof_main_event(b2f_index::ProfSlot& sl, size_t i) {
    while (sl.m.size() <= i) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
        sl.m.push_back(e);
    }
    return sl.m[i];
}

// Candidates kept per query by the tensor pass.  The slack above k must cover the rows whose coarse
// (bf16) key can fall inside the rounding band around the k-th result; that count grows with k (the
// neighbour density at rank k), hence ~0.9 k with a floor of 22.  32 / 64 are also the heap sizes of HEAP
// mode; larger values (multiples of 8, up to 256) exist in LIST mode only.  0 = k too large for K2.
int tensor_kprime(int k, int slack) {
    int extra = slack > 0 ? slack : ((9 * k + 9) / 10 > 22 ? (9 * k + 9) / 10 : 22);
    int kp = k + extra;
    if (kp <= 32) return 32;
    if (kp <= 64) return 64;
    kp = (kp + 7) / 8 * 8;
    return kp <= 256 ? kp : 0;
}

// Query chunking of the tensor path.  A batch is processed in several passes for feasibility only: more query tile
// units than units (one wave), or a big k' with so many tiles that a tile is left with too few voucher lists for the
// shared threshold (j <= 16).  Balance is no longer a reason: a pass's work is shared equally among the units whatever
// the tile count is (k2::Seg), so 16 pair tiles over 74 pairs cost 16/74 of the database per unit in ONE pass (before:
// tiles got 4 or 5 whole units, and two passes of 8 tiles were cheaper than one of 16).
// The planner still evaluates 1..8 equal passes and a few fixed pass sizes with a small cost model (tensor time per
// unit, floored by the HBM time of one database pass, plus a fixed per-pass overhead) and returns the cheapest.
// force_heap: as plan_tensor_scan's.
int plan_tensor_chunked(int nq, int64_t n, int d, int kp, bool force_heap, TensorScanPlan* plan) {
    int feasible = nq;
    while (true) {
        if (plan_tensor_scan(feasible, n, d, kp, force_heap, plan) == B2F_OK) break;
        if (feasible <= 128) return 0;
        feasible = ((feasible / 2 + 127) / 128) * 128;
    }
    const double dpad = (double)((d + 63) / 64 * 64);
    const double kSmRate = 10.0e12, kHbm = 6.0e12, kPassOverhead = 20e-6;
    const double t_hbm = (double)n * dpad * 2.0 / kHbm;
    int best_chunk = feasible;
    double best_cost = 1e30;
    // candidates: 1..8 equal passes, and the fixed pass sizes that fill one wave of pairs (74 / 37 pair tiles) or
    // give every tile many splits -- so that very large batches are cut into LIST-mode passes instead of falling
    // into the multi-wave HEAP selection (the first version of K2, ~6x slower per query)
    int cands[12];
    int nc = 0;
    for (int m = 1; m <= 8; m++) {
        int chunk = (nq + m - 1) / m;
        chunk = (chunk + 255) / 256 * 256;   // whole pair tiles
        if (chunk > feasible) chunk = m == 1 ? feasible : 0;
        if (chunk >= 256 || m == 1) cands[nc++] = chunk;
    }
    const int fixed[4] = {74 * 256, 37 * 256, 4096, 2048};
    for (int i = 0; i < 4; i++)
        if (fixed[i] < nq && fixed[i] <= feasible) cands[nc++] = fixed[i];
    for (int i = 0; i < nc; i++) {
        const int chunk = cands[i];
        if (chunk <= 0) continue;
        TensorScanPlan p{};
        if (plan_tensor_scan(chunk, n, d, kp, force_heap, &p) != B2F_OK) continue;
        const int passes = (nq + chunk - 1) / chunk;
        const double waves = p.list_mode ? 1.0 : (double)((p.units + kNumSMs - 1) / kNumSMs);
        // rows every unit streams: LIST mode shares the pass equally (tile_units / units of the database per unit,
        // whatever the two numbers are), HEAP mode splits every tile nsplits ways
        const double rows_per_unit = p.list_mode ? (double)n * p.tile_units / p.units : (double)n / p.nsplits;
        double t_mma = rows_per_unit * 128.0 * dpad * 2.0 / kSmRate * waves;  // per SM
        if (!p.list_mode) t_mma *= 6.0;   // per-thread heaps instead of shared-threshold lists
        const double cost = passes * ((t_mma > t_hbm ? t_mma : t_hbm) + kPassOverhead);
        if (cost < best_cost * 0.97) {  // a new candidate has to buy at least 3%
            best_cost = cost;
            best_chunk = chunk;
        }
    }
    if (plan_tensor_scan(best_chunk, n, d, kp, force_heap, plan) != B2F_OK) return 0;
    return best_chunk;
}

}  // namespace

// =================================================================================================
extern "C" {

int b2f_version(void) { return B2F_VERSION; }

const char* b2f_last_error(void) { return g_err; }

int b2f_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    int ok = 0;
    for (int i = 0; i < n; i++) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ok++;
    }
    return ok;
}

int b2f_index_create(int32_t d, int32_t metric, int32_t storage, int32_t device, b2f_index** out) {
    if (!out) {
        set_error("out is NULL");
        return B2F_EINVAL;
    }
    *out = nullptr;
    if (d <= 0 || d > 16384) {
        set_error("d=%d out of range [1,16384]", d);
        return B2F_EINVAL;
    }
    if (metric != B2F_METRIC_L2 && metric != B2F_METRIC_INNER_PRODUCT) {
        set_error("metric %d not supported (0 = inner product, 1 = L2)", metric);
        return B2F_EINVAL;
    }
    if (storage != B2F_STORE_F32 && storage != B2F_STORE_BF16) {
        set_error("storage %d not supported", storage);
        return B2F_EINVAL;
    }
    B2F_TRY(check_device(device));
    DeviceGuard g(device);
    b2f_index* ix = new (std::nothrow) b2f_index();
    if (!ix) return B2F_ENOMEM;
    ix->d = d;
    ix->metric = metric;
    ix->storage = storage;
    ix->device = device;
    ix->dpad = (int64_t)align_up((size_t)d, 64);
    cudaError_t e = cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&ix->stats, 2 * sizeof(float));
    if (e == cudaSuccess) e = cudaMemset(ix->stats, 0, 2 * sizeof(float));
    // centre [d] floats, then (8-byte aligned) d 64-bit words and d floats: the fixed-point accumulators its mean is summed
    // in and the per-column magnitudes that choose their scale
    const size_t centre_bytes = (((size_t)d * sizeof(float) + 7) & ~(size_t)7) + (size_t)d * 12;
    if (e == cudaSuccess) e = cudaMalloc(&ix->centre, centre_bytes);
    if (e == cudaSuccess) e = cudaMemset(ix->centre, 0, centre_bytes);
    if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void**>(&ix->host_flag), 64, cudaHostAllocMapped | cudaHostAllocPortable);
    if (e == cudaSuccess) memset(ix->host_flag, 0, 64);
    if (e == cudaSuccess) e = cudaMalloc(&ix->totals, 4 * sizeof(unsigned long long) + kScanTubWords * 4);
    if (e == cudaSuccess) e = cudaMemset(ix->totals, 0, 4 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemset(ix->totals + 4, 0xff, kScanTubWords * 4);  // the scan's cross-CTA bounds, idle = all ones
    if (e != cudaSuccess) {
        set_error("index init failed: %s", cudaGetErrorString(e));
        delete ix;
        return B2F_ECUDA;
    }
    *out = ix;
    return B2F_OK;
}

int b2f_index_destroy(b2f_index* ix) {
    if (!ix) return B2F_OK;
    DeviceGuard g(ix->device);
    cudaDeviceSynchronize();
    cudaFree(ix->rows_f32);
    cudaFree(ix->scan);
    cudaFree(ix->norms);
    cudaFree(ix->stats);
    cudaFree(ix->centre);
    cudaFree(ix->qpool);
    cudaFree(ix->ws);
    if (ix->pinned) cudaFreeHost(ix->pinned);
    if (ix->host_flag) cudaFreeHost(ix->host_flag);
    cudaFree(ix->totals);
    cudaFree(ix->rm_flags);
    for (cudaEvent_t e : ix->ev) cudaEventDestroy(e);
    if (ix->ev_done) cudaEventDestroy(ix->ev_done);
    if (ix->ev_ingest) cudaEventDestroy(ix->ev_ingest);
    for (auto& sl : ix->prof) {
        if (sl.t0) cudaEventDestroy(sl.t0);
        if (sl.t1) cudaEventDestroy(sl.t1);
        for (cudaEvent_t e : sl.m) cudaEventDestroy(e);
    }
    if (ix->stream) cudaStreamDestroy(ix->stream);
    delete ix;
    return B2F_OK;
}

int b2f_index_reset(b2f_index* ix) {
    if (!ix) {
        set_error("index is NULL");
        return B2F_EINVAL;
    }
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    ix->ntotal = 0;
    ix->mu_set = false;
    ix->adapt = {};
    if (ix->search_recorded) B2F_CUDA(cudaEventSynchronize(ix->ev_done));
    if (ix->add_recorded) B2F_CUDA(cudaEventSynchronize(ix->ev_ingest));
    B2F_CUDA(cudaMemsetAsync(ix->stats, 0, 2 * sizeof(float), ix->stream));
    B2F_CUDA(cudaStreamSynchronize(ix->stream));
    ix->stats_dirty = true;
    return B2F_OK;
}

int b2f_index_reserve(b2f_index* ix, int64_t nrows) {
    if (!ix) {
        set_error("index is NULL");
        return B2F_EINVAL;
    }
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    return ensure_capacity(ix, nrows);
}

int64_t b2f_index_ntotal(const b2f_index* ix) { return ix ? ix->ntotal : -1; }
int32_t b2f_index_d(const b2f_index* ix) { return ix ? ix->d : -1; }
int32_t b2f_index_metric(const b2f_index* ix) { return ix ? ix->metric : -1; }
int32_t b2f_index_storage(const b2f_index* ix) { return ix ? ix->storage : -1; }
int32_t b2f_index_device(const b2f_index* ix) { return ix ? ix->device : -1; }

int b2f_plan_describe(int64_t nq, int64_t n, int32_t d, int64_t k, int32_t slack, int32_t out[12]) {
    if (!out || nq <= 0 || n <= 0 || d <= 0 || k <= 0 || nq > (1 << 24)) {
        set_error("plan_describe: bad arguments");
        return B2F_EINVAL;
    }
    for (int i = 0; i < 12; i++) out[i] = 0;
    const int kp = k <= 1024 ? tensor_kprime((int)k, slack) : 0;
    if (kp <= 0) return B2F_OK;
    TensorScanPlan plan{};
    const int chunk = plan_tensor_chunked((int)nq, n, d, kp, false, &plan);
    if (chunk <= 0) return B2F_OK;
    out[0] = kp;
    out[1] = chunk;
    out[2] = (int32_t)((nq + chunk - 1) / chunk);
    out[3] = plan.list_mode;
    out[4] = plan.pair_mode;
    out[5] = plan.units;
    out[6] = plan.nsplits;
    out[7] = plan.nlists;
    out[8] = plan.list_j;
    out[9] = plan.list_cap;
    out[10] = plan.nq_tiles;
    out[11] = plan.round_tiles;
    return B2F_OK;
}

int b2f_plan_unit_work(int32_t tile_units, int32_t units, int32_t round_tiles, int64_t db_tiles, int32_t kprime, int32_t unit,
                       int32_t seg_info[14], int64_t* tiles, int64_t cap, int32_t counts[2]) {
    const int rc = plan_unit_work(tile_units, units, round_tiles, db_tiles, kprime, unit, seg_info, tiles, cap, counts);
    if (rc < 0) set_error("plan_unit_work: bad arguments");
    return rc < 0 ? B2F_EINVAL : rc;
}

int b2f_index_stats(const b2f_index* cix, b2f_stats* out) {
    if (!cix || !out) {
        set_error("NULL argument");
        return B2F_EINVAL;
    }
    // searches return without synchronising and keep their counters on the device: settle them first
    b2f_index* ix = const_cast<b2f_index*>(cix);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    if (g.ok && ix->totals) {
        if (ix->search_recorded) B2F_CUDA(cudaEventSynchronize(ix->ev_done));
        unsigned long long t[4] = {0, 0, 0, 0};
        B2F_CUDA(cudaMemcpy(t, ix->totals, sizeof(t), cudaMemcpyDeviceToHost));
        ix->st.fallback_queries = (int64_t)t[0];
        ix->st.overflow_queries = (int64_t)t[1];
        ix->st.rescued_queries = (int64_t)t[2];
        harvest_flag(ix);
        for (int i = 0; i < b2f_index::kProfSlots; i++)
            harvest_prof_slot(ix, ix->prof[(ix->prof_head + i) % b2f_index::kProfSlots]);  // oldest first
    }
    *out = ix->st;
    return B2F_OK;
}

// ---- add -------------------------------------------------------------------------------------------
// The scan copy is taken around the mean of the first rows the index sees, fixed from then on: any centre is correct, a
// representative one makes the bf16 pass far more decisive on embeddings that share a large common component.  bf16
// storage keeps the same centred copy as its ONLY copy: the authoritative row is then fl32(mu + bf16(x - mu)) -- closer
// to x than bf16(x) on such data, and the tensor pass certifies as on fp32 storage.
// Which rows: the first min(n, 65536) rows of the FIRST add call, on every route (device rows, host rows, pooled,
// generated, read from a file), whatever the route's staging -- so that the same rows give the same centre, and the same
// bf16-storage index, bit for bit.  Every route calls take_centre before it ingests its first rows.  A route that stages
// its rows through a smaller buffer passes its piece size (>= 64 rows) and stage(r0, rows, &src), which puts rows
// [r0, r0 + rows) of the call on the device in stream order; both passes of the mean walk every piece, so such a route
// stages the first <= 65536 rows once more (they fit one piece) or twice more, once per index.
static const int64_t kCentreRows = 65536;

extern "C++" {   // (a template inside the extern "C" block)
template <class Stage>
static int take_centre(b2f_index* ix, int64_t n, int64_t piece, cudaStream_t st, Stage&& stage) {
    if (ix->mu_set || ix->ntotal != 0 || n <= 0) return B2F_OK;
    const int64_t m = n < kCentreRows ? n : kCentreRows;
    piece = piece >= m ? m : piece / 64 * 64;
    if (piece <= 0) {
        set_error("centre: staging piece of %lld rows is below one 64-row block", (long long)piece);
        return B2F_EINVAL;
    }
    unsigned long long* acc = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(ix->centre) + (((size_t)ix->d * sizeof(float) + 7) & ~(size_t)7));
    B2F_TRY(launch_mean_begin(ix->d, acc, st));
    const float* src = nullptr;
    for (int pass = 0; pass < 2; pass++)
        for (int64_t r0 = 0; r0 < m; r0 += piece) {
            const int64_t rows = m - r0 < piece ? m - r0 : piece;
            if (pass == 0 || piece < m) B2F_TRY(stage(r0, rows, &src));   // (one piece: pass 1 reads it again in place)
            B2F_TRY(launch_mean_pass(src, r0, rows, m, ix->d, acc, pass, st));
            ix->st.launches++;
        }
    B2F_TRY(launch_mean_finish(m, ix->d, ix->centre, acc, st));
    ix->st.launches++;
    ix->mu_set = true;
    return B2F_OK;
}
static int add_device_rows(b2f_index* ix, const float* src_dev, int64_t n, cudaStream_t st) {
    // src_dev: [n, d] fp32 on the device (may alias the tail of rows_f32); the centre is set (take_centre) beforehand
    float* rows_out = nullptr;
    if (ix->storage == B2F_STORE_F32) {
        float* dst = ix->rows_f32 + ix->ntotal * ix->d;
        if (src_dev != dst) rows_out = dst;
    }
    B2F_TRY(launch_ingest(src_dev, n, ix->d, rows_out, ix->scan + ix->ntotal * ix->dpad, ix->dpad,
                          ix->norms + ix->ntotal, ix->stats, scan_centre(ix),
                          ix->metric == B2F_METRIC_INNER_PRODUCT ? 1 : 0, ix->storage == B2F_STORE_BF16 ? 1 : 0, st));
    ix->st.launches++;
    return B2F_OK;
}

// One add call of n rows, on every route.  Rows already on the device (dev) are ingested where they are.  Any other route
// stages them in pieces of `piece` rows: stage(r0, rows, dst) puts rows [r0, r0 + rows) of the call into dst in stream
// order -- their final place on fp32 storage (the ingest then derives the scan copy in place), the workspace on bf16
// storage, whose only copy is the scan copy.  A call that fits one piece is staged once and gives the centre from those
// rows; a longer one lets take_centre stage the centre's rows first.
template <class Stage>
static int ingest_call(b2f_index* ix, int64_t n, int64_t piece, const float* dev, cudaStream_t st, Stage&& stage) {
    const int64_t base = ix->ntotal;
    const bool via_ws = !dev && ix->storage == B2F_STORE_BF16;
    if (via_ws) B2F_TRY(ensure_ws(ix, (size_t)(n < piece ? n : piece) * ix->d * 4 + 4096));
    auto put = [&](int64_t r0, int64_t rows, const float** src) -> int {
        if (dev) {
            *src = dev + r0 * ix->d;
            return B2F_OK;
        }
        float* dst = via_ws ? reinterpret_cast<float*>(ix->ws) : ix->rows_f32 + (base + r0) * ix->d;
        *src = dst;
        return stage(r0, rows, dst);
    };
    if (piece >= n) {
        const float* src = nullptr;
        B2F_TRY(put(0, n, &src));
        B2F_TRY(take_centre(ix, n, n, st, [&](int64_t r0, int64_t, const float** s) {
            *s = src + r0 * ix->d;
            return B2F_OK;
        }));
        B2F_TRY(add_device_rows(ix, src, n, st));
        ix->ntotal += n;
    } else {
        B2F_TRY(take_centre(ix, n, piece, st, put));
        for (int64_t r0 = 0; r0 < n; r0 += piece) {
            const int64_t rows = n - r0 < piece ? n - r0 : piece;
            const float* src = nullptr;
            B2F_TRY(put(r0, rows, &src));
            B2F_TRY(add_device_rows(ix, src, rows, st));
            ix->ntotal += rows;
        }
    }
    ix->stats_dirty = true;
    return record_ingest(ix, st);
}
}  // extern "C++"

int b2f_index_add(b2f_index* ix, int64_t n, const float* x, int32_t mem, void* stream) {
    if (!ix || n < 0 || (n > 0 && !x)) {
        set_error("add: bad arguments");
        return B2F_EINVAL;
    }
    if (n == 0) return B2F_OK;
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : ix->stream;
    B2F_TRY(enter_stream(ix, g, st));
    B2F_TRY(ensure_capacity(ix, ix->ntotal + n));
    if (mem == B2F_MEM_DEVICE) return ingest_call(ix, n, n, x, st, [](int64_t, int64_t, float*) { return B2F_OK; });
    // host rows: one copy of all of them on fp32 storage, 64 MB pieces on bf16 storage
    const int64_t piece = ix->storage == B2F_STORE_F32 ? n : rows_in(64u << 20, ix->d);
    B2F_TRY(ingest_call(ix, n, piece, nullptr, st, [&](int64_t r0, int64_t m, float* dst) {
        B2F_CUDA(cudaMemcpyAsync(dst, x + r0 * ix->d, (size_t)m * ix->d * 4, cudaMemcpyHostToDevice, st));
        return B2F_OK;
    }));
    B2F_CUDA(cudaStreamSynchronize(st));
    return B2F_OK;
}

int b2f_index_add_synth(b2f_index* ix, uint64_t seed, int64_t row0, int64_t nrows, int32_t normalize) {
    if (!ix || nrows < 0) {
        set_error("add_synth: bad arguments");
        return B2F_EINVAL;
    }
    if (nrows == 0) return B2F_OK;
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = ix->stream;
    B2F_TRY(enter_stream(ix, g, st));
    B2F_TRY(ensure_capacity(ix, ix->ntotal + nrows));
    const int64_t piece = ix->storage == B2F_STORE_F32 ? nrows : rows_in(256u << 20, ix->d);
    B2F_TRY(ingest_call(ix, nrows, piece, nullptr, st, [&](int64_t r0, int64_t m, float* dst) {
        B2F_TRY(launch_synth(seed, row0 + r0, m, ix->d, normalize, dst, st));
        ix->st.launches++;
        return B2F_OK;
    }));
    B2F_CUDA(cudaStreamSynchronize(st));
    return B2F_OK;
}

int b2f_index_add_pooled(b2f_index* ix, const float* hidden, const int64_t* mask, int64_t B, int64_t T, int32_t pool,
                         int32_t normalize, void* stream) {
    if (!ix || B < 0 || (B > 0 && !hidden)) {
        set_error("add_pooled: bad arguments");
        return B2F_EINVAL;
    }
    if (B == 0) return B2F_OK;
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : ix->stream;
    B2F_TRY(enter_stream(ix, g, st));
    B2F_TRY(ensure_capacity(ix, ix->ntotal + B));
    // The pooled rows go through the SAME ingest kernel every other add uses: it derives the scan copy, the per-row
    // bias of the tensor pass (L2: |x~'|^2, IP: -mu.x -- NOT a norm) and the stats for either storage mode and metric.
    const int64_t piece = ix->storage == B2F_STORE_F32 ? B : rows_in(64u << 20, ix->d);
    return ingest_call(ix, B, piece, nullptr, st, [&](int64_t b0, int64_t m, float* dst) {
        B2F_TRY(launch_pool(hidden + b0 * T * ix->d, mask ? mask + b0 * T : nullptr, m, T, ix->d, pool, normalize, dst, st));
        ix->st.launches++;
        return B2F_OK;
    });
}

int b2f_pool_normalize(const float* hidden, const int64_t* mask, int64_t B, int64_t T, int32_t d, int32_t pool,
                       int32_t normalize, float* out, int32_t device, void* stream) {
    if (B < 0 || d <= 0 || (B > 0 && (!hidden || !out))) {
        set_error("pool_normalize: bad arguments");
        return B2F_EINVAL;
    }
    B2F_TRY(check_device(device));
    DeviceGuard g(device);
    return launch_pool(hidden, mask, B, T, d, pool, normalize, out, (cudaStream_t)stream);
}

int b2f_synth_rows(uint64_t seed, int64_t row0, int64_t nrows, int32_t d, int32_t normalize, float* out, int32_t device,
                   void* stream) {
    if (nrows < 0 || d <= 0 || (nrows > 0 && !out)) {
        set_error("synth_rows: bad arguments");
        return B2F_EINVAL;
    }
    B2F_TRY(check_device(device));
    DeviceGuard g(device);
    return launch_synth(seed, row0, nrows, d, normalize, out, (cudaStream_t)stream);
}

int b2f_merge_topk_strided(int32_t metric, int64_t nq, int64_t k, int32_t nparts, const float* D_parts, const int64_t* I_parts,
                           int64_t part_stride_bytes, float* D, int64_t* I, int32_t device, void* stream) {
    if (nq < 0 || k <= 0 || !D_parts || !I_parts || !D || !I || part_stride_bytes <= 0 || (part_stride_bytes & 7)) {
        set_error("merge_topk: bad arguments");
        return B2F_EINVAL;
    }
    B2F_TRY(check_device(device));
    DeviceGuard g(device);
    return launch_merge_faiss(metric, nq, k, nparts, D_parts, I_parts, part_stride_bytes, D, I, (cudaStream_t)stream);
}

int b2f_merge_range_strided(int64_t nq, int32_t nparts, const int64_t* lims_parts, const float* D_parts,
                            const int64_t* I_parts, int64_t part_stride_bytes, float* D, int64_t* I, int32_t device,
                            void* stream) {
    // the hit count lives in the device lims, so with nq > 0 every hit pointer must be usable
    const bool misaligned = ((uintptr_t)lims_parts | (uintptr_t)I_parts | (uintptr_t)I) & 7 || ((uintptr_t)D_parts | (uintptr_t)D) & 3;
    if (nq < 0 || nparts < 1 || nparts > 32 || !lims_parts || part_stride_bytes <= 0 || (part_stride_bytes & 15) ||
        (nq > 0 && (!D_parts || !I_parts || !D || !I)) || misaligned) {
        set_error("merge_range: bad arguments");
        return B2F_EINVAL;
    }
    B2F_TRY(check_device(device));
    DeviceGuard g(device);
    return launch_merge_range(nq, nparts, lims_parts, D_parts, I_parts, part_stride_bytes, D, I, (cudaStream_t)stream);
}

}  // extern "C"

// ---- search workspace ------------------------------------------------------------------------------
// The query side of one tensor pass: bf16 copy, |q~|^2, e_q and the per-query constant
struct PassQueries {
    __nv_bfloat16* qb;
    float* qnorm;
    float* qerr;
    float* qconst;
};
static PassQueries take_queries(Bump& b, size_t rows, int64_t dpad) {
    PassQueries p;
    p.qb = b.take<__nv_bfloat16>(rows * dpad);
    p.qnorm = b.take<float>(rows);
    p.qerr = b.take<float>(rows);
    p.qconst = b.take<float>(rows);
    return p;
}

// LIST-mode scratch of a tensor pass planned as p
static TensorScanLists take_lists(Bump& b, const TensorScanPlan& p) {
    const size_t nq_pad = (size_t)p.nq_tiles * 128, words = nq_pad * p.nlists;
    TensorScanLists l{};
    l.shared_thr = b.take<float>(words);
    l.counts = b.take<int32_t>(words);
    l.final_thr = b.take<float>(words);
    l.cand = b.take<uint2>(words * p.list_cap);
    l.big_flag = b.take<uint8_t>(nq_pad);   // warp-merge pass-on flags
    return l;
}

// A filtered search's buffers: the allow bitmap, the masked row bias of the tensor pass, and the device copy of host-memory
// selector data
struct FilterWs {
    uint32_t* allow = nullptr;
    float* bias = nullptr;
    void* staged = nullptr;
};

static FilterWs carve_filter(Bump& b, const b2f_index* ix, const b2f_selector* sel, int64_t id_offset, bool host, bool tensor) {
    FilterWs f;
    if (!sel || ix->ntotal == 0) return f;
    f.allow = b.take<uint32_t>((size_t)(ix->ntotal + 31) / 32);
    if (tensor) f.bias = b.take<float>((size_t)ix->ntotal);
    if (host) f.staged = b.take<char>(filter_staged_bytes(*sel, ix->ntotal, id_offset));
    return f;
}

// Builds a filtered call's allow bitmap (and, for the tensor pass, its masked bias) on st; *launches: kernels launched
static int build_filter(const b2f_index* ix, const b2f_selector* sel, int32_t mem, int64_t id_offset, const FilterWs& f,
                        cudaStream_t st, int* launches) {
    *launches = 0;
    if (!f.allow) return B2F_OK;
    B2F_TRY(launch_allow_bitmap(*sel, mem, ix->ntotal, id_offset, f.staged, f.allow, st));
    *launches = (sel->kind == B2F_SEL_BATCH && sel->n > 0) ? 2 : 1;
    if (f.bias) {
        B2F_TRY(launch_masked_bias(ix->norms, f.allow, ix->ntotal, f.bias, st));
        ++*launches;
    }
    return B2F_OK;
}

// the row bias the tensor pass reads: a filtered search's masked copy, else the index's own
static const float* tensor_bias(const b2f_index* ix, const FilterWs& f) { return f.bias ? f.bias : ix->norms; }

// What one search carves from the workspace, in one order (carve_ws measures it, then lays it out).
struct SearchWs {
    float* q = nullptr;              // host buffers: device copies of the queries and the results
    float* D = nullptr;
    int64_t* I = nullptr;
    void* scan_scratch = nullptr;
    PassQueries pq{};                // tensor path from here on
    TensorScanLists lists{};         // LIST mode
    float* pk = nullptr;             // HEAP mode: partial lists, merged coarse candidates
    int32_t* pi = nullptr;
    float* ck = nullptr;
    int32_t* ci = nullptr;
    int32_t* fail_list = nullptr;
    float* fail_tau = nullptr;       // range mode
    // [0] uncertified queries, [1] of which list overflows, [2..3] u64 list entries, [4] rescued by the extended pass,
    // [8..11] ticket counters of K2's die-aware unit assignment
    int32_t* counters = nullptr;
    FilterWs filter{};               // filtered search
};

static SearchWs carve_search(Bump& b, const b2f_index* ix, int nq, int k, bool host, bool tensor, const TensorScanPlan& plan,
                             int chunk_nq, int kp, const b2f_selector* sel, int64_t id_offset) {
    SearchWs w;
    w.filter = carve_filter(b, ix, sel, id_offset, host, tensor);
    if (host) {
        w.q = b.take<float>((size_t)nq * ix->d);
        w.D = b.take<float>((size_t)nq * k);
        w.I = b.take<int64_t>((size_t)nq * k);
    }
    w.scan_scratch = b.take<char>(scan_scratch_bytes(k));
    if (!tensor) return w;
    const size_t nq_pad = (size_t)plan.nq_tiles * 128;
    w.pq = take_queries(b, nq_pad, ix->dpad);
    if (plan.list_mode) {
        w.lists = take_lists(b, plan);
    } else {
        w.pk = b.take<float>(nq_pad * plan.nsplits * kp);
        w.pi = b.take<int32_t>(nq_pad * plan.nsplits * kp);
        w.ck = b.take<float>((size_t)chunk_nq * kp);
        w.ci = b.take<int32_t>((size_t)chunk_nq * kp);
    }
    w.fail_list = b.take<int32_t>(nq);
    if (ix->adapt.range_mode) w.fail_tau = b.take<float>(nq);
    w.counters = b.take<int32_t>(16);
    w.lists.die_ctr = w.counters + 8;
    return w;
}

// The re-rank of one tensor pass over the nq queries q (pq: their tensor-pass buffers): results go to D / I in faiss
// layout, the queries it cannot certify to fail_list / fail_count
static RerankArgs rerank_args(const b2f_index* ix, const float* q, const PassQueries& pq, int nq, int k, int kp, float* D,
                              int64_t* I, int64_t id_offset, int32_t* fail_list, int32_t* fail_count) {
    RerankArgs a{};
    a.rows = stored_rows(ix);
    a.q = q;
    a.qnorm = pq.qnorm;
    a.qerr = pq.qerr;
    a.qconst = pq.qconst;
    a.mu_norm = ix->mu_norm;
    a.nq = nq;
    a.kp = kp;
    a.k = k;
    a.max_row_norm = sqrtf(ix->host_stats[0]);
    // fp32 storage: the bf16 rounding of the centred row; bf16 storage: what fl32(mu + x~') loses (0 uncentred)
    a.max_row_err = sqrtf(ix->host_stats[1]);
    a.certify = 1;
    a.D = D;
    a.I = I;
    a.id_offset = id_offset;
    a.fail_list = fail_list;
    a.fail_count = fail_count;
    return a;
}

// ---- range pass (second tensor pass over uncertified queries) -----------------------------------------
constexpr int kRangeCap = 1024;   // failed queries one range pass holds; more go to the exact scan
constexpr int kRangeListCap = 256;

static int plan_range_pass(int nfail, int64_t n, int d, int kp, TensorScanPlan* plan) {
    if (plan_tensor_scan(nfail, n, d, kp, false, plan) != B2F_OK || !plan->list_mode) return B2F_EINVAL;
    if (plan->list_cap < kRangeListCap) plan->list_cap = kRangeListCap;   // lists are not pruned: every row at or below the threshold
    return B2F_OK;
}

// What a range pass carves behind the search's own buffers: its queries hold kRangeCap rows whatever the failed count,
// its lists follow its plan
struct RangeWs {
    float* q;                        // the failed queries, gathered
    PassQueries pq;
    float* tau;
    float* thr;
    int32_t* out_map;
    int32_t* fail_list;
    int32_t* counters;               // [0..7] as SearchWs::counters, [8..11] K2's tickets, [16] compacted queries
    TensorScanLists lists;
};

static RangeWs carve_range(Bump& b, const b2f_index* ix, int nq, const TensorScanPlan& rp) {
    RangeWs r;
    r.q = b.take<float>((size_t)kRangeCap * ix->d);
    r.pq = take_queries(b, kRangeCap, ix->dpad);
    r.tau = b.take<float>(kRangeCap);
    r.thr = b.take<float>(kRangeCap);
    r.out_map = b.take<int32_t>(kRangeCap);
    r.fail_list = b.take<int32_t>(nq);
    r.counters = b.take<int32_t>(32);
    r.lists = take_lists(b, rp);
    r.lists.die_ctr = r.counters + 8;
    r.lists.range_thr = r.thr;
    return r;
}

// Where a range pass carved behind the search's buffers (carve_search(Bump&) lays them out) ends at most.  The list
// geometry depends on the number of failed queries, known only after the host sync: take the largest over 128..kRangeCap
// of them.
template <class Carve>
static size_t range_end(Carve&& carve_search, const b2f_index* ix, int nq, int kp) {
    Bump search(nullptr, SIZE_MAX);
    carve_search(search);
    size_t end = search.off;
    for (int f = 128; f <= kRangeCap; f *= 2) {
        TensorScanPlan p{};
        if (plan_range_pass(f, ix->ntotal, ix->d, kp, &p) != B2F_OK) continue;
        Bump b = search;
        carve_range(b, ix, nq, p);
        if (b.off > end) end = b.off;
    }
    return end;
}

// Range pass.  Earlier batches on this index left many queries uncertified (data denser than the bf16 band even after
// centring): instead of one exact scan per four of them, ONE more tensor pass serves them all.  For a failed query the
// first pass found an exact k-th key tau, an upper bound of the true one; every true top-k row therefore has a coarse key
// <= thr(tau) (the certification bound, inverted), so a pass that lists EVERY row at or below that fixed threshold and
// re-ranks all of them is exact.  The host must know how many queries failed to plan the pass: the one synchronisation
// inside a search, paid only by indexes in this mode.
// *served: the queries the pass served (0: it did not run); *scan_list / *scan_counters: what the closing scan reads.
static int range_pass(b2f_index* ix, Bump& bump, const SearchWs& w, const float* q, int nq, int k, int kp, float* D, int64_t* I,
                      int64_t id_offset, cudaStream_t st, int32_t** scan_list, int32_t** scan_counters, int* served) {
    volatile int32_t* hf = ix->host_flag + 12;
    B2F_CUDA(cudaMemcpyAsync(const_cast<int32_t*>(hf), w.counters, 4, cudaMemcpyDeviceToHost, st));
    B2F_CUDA(cudaStreamSynchronize(st));
    const int nfail = hf[0];
    ix->adapt.first_pass_failed(nfail);
    TensorScanPlan rp{};
    const int nr = nfail < kRangeCap ? nfail : kRangeCap;
    if (nfail < 8 || plan_range_pass(nr, ix->ntotal, ix->d, kp, &rp) != B2F_OK) return B2F_OK;
    const RangeWs r = carve_range(bump, ix, nq, rp);
    if (!bump.fits()) return B2F_OK;   // a layout the workspace was not sized for: the exact scan serves these queries
    const int nq_pad = rp.nq_tiles * 128;
    B2F_CUDA(cudaMemsetAsync(r.counters, 0, 32 * 4, st));
    B2F_CUDA(cudaMemsetAsync(r.out_map, 0xff, (size_t)kRangeCap * 4, st));
    B2F_CUDA(cudaMemsetAsync(r.q, 0, (size_t)nq_pad * ix->d * 4, st));
    B2F_TRY(launch_gather_failed(q, ix->d, w.fail_list, w.fail_tau, w.counters, nfail, nr, r.q, r.tau, r.out_map, r.counters + 16,
                                 r.fail_list, r.counters, st));
    B2F_TRY(launch_prep_queries(r.q, nr, nq_pad, ix->d, r.pq.qb, ix->dpad, r.pq.qnorm, r.pq.qerr, r.pq.qconst, scan_centre(ix), nullptr,
                                0, reinterpret_cast<uint32_t*>(r.lists.shared_thr), (int64_t)nq_pad * rp.nlists, st));
    B2F_TRY(launch_range_thresholds(r.tau, 0.f, r.out_map, nr, ix->d, ix->metric, r.pq.qnorm, r.pq.qerr, r.pq.qconst,
                                    sqrtf(ix->host_stats[0]), sqrtf(ix->host_stats[1]), ix->mu_norm, r.thr, st));
    B2F_TRY(launch_tensor_scan(ix->scan, ix->dpad, tensor_bias(ix, w.filter), ix->ntotal, ix->metric, r.pq.qb, nr, nq_pad, rp, nullptr,
                               nullptr, r.lists, st));
    RerankArgs ra = rerank_args(ix, r.q, r.pq, nr, k, kp, D, I, id_offset, r.fail_list, r.counters);
    ra.out_map = r.out_map;
    ra.range = 1;
    B2F_TRY(launch_merge_lists(r.lists, nr, rp, nullptr, ra, st));
    // the statistics the closing kernel publishes: what the first pass counted, with the final fallback count
    B2F_CUDA(cudaMemcpyAsync(r.counters + 1, w.counters + 1, 7 * 4, cudaMemcpyDeviceToDevice, st));
    count_launches(ix, 5);
    ix->st.range_queries += nr;
    *served = nr;
    *scan_list = r.fail_list;
    *scan_counters = r.counters;
    return B2F_OK;
}

// ---- search ----------------------------------------------------------------------------------------
// The caller holds ix->mu (search_pooled pools the queries into the index's buffer and searches them under ONE
// lock, so a second thread cannot overwrite or re-allocate that buffer in between).
static int search_locked(b2f_index* ix, int64_t nq64, const float* q, int64_t k64, float* D, int64_t* I, int32_t mem,
                         void* stream, const b2f_search_params* params, const b2f_selector* sel) {
    if (k64 <= 0) {
        set_error("k must be > 0 (faiss asserts k > 0)");
        return B2F_EINVAL;
    }
    if (k64 > 1024) {
        set_error("k=%lld > 1024 is not supported by the GPU selection kernels", (long long)k64);
        return B2F_EINVAL;
    }
    if (nq64 < 0 || nq64 > (1 << 24) || (nq64 > 0 && (!q || !D || !I))) {
        set_error("search: bad arguments");
        return B2F_EINVAL;
    }
    if (nq64 == 0) return B2F_OK;
    const int nq = (int)nq64, k = (int)k64;
    b2f_search_params P{};
    if (params) P = *params;
    DeviceGuard g(ix->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : ix->stream;
    B2F_TRY(enter_stream(ix, g, st));
    B2F_TRY(order_after(st, ix->stream, ix));
    const bool host = mem == B2F_MEM_HOST;
    const bool profile = P.profile != 0;
    harvest_flag(ix);

    // ---- plan ----------------------------------------------------------------------------------
    int algo = P.algo;
    // AUTO: fp32 storage serves the reference's own batch size (nq = 1) with the fp32 streaming scan -- the
    // reference's arithmetic, 90% of HBM on the fp32 rows.  bf16 storage has nothing to gain from it (both paths
    // read the same bf16 rows; the tensor path streams them at the full HBM rate, the CUDA-core scan at half
    // of it because of the unpacking), so every batch size goes to the tensor path there.
    const int scan_max = P.scan_max_nq > 0 ? P.scan_max_nq : (ix->storage == B2F_STORE_BF16 ? 0 : 1);
    int kp = tensor_kprime(k, P.slack);
    if (kp > 0 && P.slack <= 0 && ix->adapt.slack_boost > 0) {  // adaptive slack learned from earlier searches on this index
        int boosted = ((kp + ix->adapt.slack_boost + 7) / 8) * 8;
        if (boosted > 64) kp = boosted <= 256 ? boosted : 256;
    }
    TensorScanPlan plan{};
    const bool heap_first = ix->adapt.heap_left > 0 && P.certify >= 0;
    const int chunk_nq = (kp > 0 && ix->ntotal > 0) ? plan_tensor_chunked(nq, ix->ntotal, ix->d, kp, heap_first, &plan) : 0;
    const bool tensor_ok = chunk_nq > 0;
    if (algo == B2F_ALGO_AUTO) algo = (nq <= scan_max || !tensor_ok) ? B2F_ALGO_SCAN : B2F_ALGO_TENSOR;
    // an explicit TENSOR request on a shape the tensor path cannot plan (k' > 256, or a database of a few rows with
    // k' other than 32 / 64) is served by the exact scan, like AUTO would; stats().last_algo tells
    if (algo == B2F_ALGO_TENSOR && !tensor_ok) algo = B2F_ALGO_SCAN;
    const bool tensor = algo == B2F_ALGO_TENSOR;
    const int certify = P.certify >= 0 ? 1 : 0;
    if (tensor && heap_first) ix->adapt.heap_left--;

    // ---- workspace -----------------------------------------------------------------------------
    SearchWs w;
    Bump bump(nullptr, 0);   // the workspace behind w: a range pass carves its buffers there
    const auto carve = [&](Bump& b) {
        w = carve_search(b, ix, nq, k, host, tensor, plan, chunk_nq, kp, sel, P.id_offset);
        bump = b;
    };
    B2F_TRY(carve_ws(ix, tensor && ix->adapt.range_mode ? range_end(carve, ix, nq, kp) : 0, carve, "search"));
    const float* qd = host ? w.q : q;
    float* Dd = host ? w.D : D;
    int64_t* Id = host ? w.I : I;
    if (host) B2F_CUDA(cudaMemcpyAsync(w.q, q, (size_t)nq * ix->d * 4, cudaMemcpyHostToDevice, st));
    ix->st.searches++;
    ix->st.last_launches = 0;
    ix->st.last_algo = algo;
    ix->st.last_kprime = 0;
    int filter_launches = 0;
    B2F_TRY(build_filter(ix, sel, mem, P.id_offset, w.filter, st, &filter_launches));
    count_launches(ix, filter_launches);
    int n_main = 0;
    b2f_index::ProfSlot* slot = nullptr;
    if (profile) {
        slot = &ix->prof[ix->prof_head % b2f_index::kProfSlots];
        ix->prof_head++;
        harvest_prof_slot(ix, *slot);  // blocks only when the host is a whole ring of searches ahead
        if (!slot->t0) B2F_CUDA(cudaEventCreate(&slot->t0));
        if (!slot->t1) B2F_CUDA(cudaEventCreate(&slot->t1));
        B2F_CUDA(cudaEventRecord(slot->t0, st));
    }
    auto main_event = [&](int which) -> int {  // which: 0 = before, 1 = after the dominant kernel's launch
        if (!slot) return B2F_OK;
        cudaEvent_t e = prof_main_event(*slot, 2 * (size_t)n_main + which);
        if (!e) {
            set_error("cudaEventCreate failed");
            return B2F_ECUDA;
        }
        B2F_CUDA(cudaEventRecord(e, st));
        return B2F_OK;
    };

    if (ix->ntotal == 0) {
        B2F_TRY(launch_fill_empty(nq, k, ix->metric, Dd, Id, st));
        count_launches(ix, 1);
    } else if (!tensor) {
        B2F_TRY(main_event(0));
        B2F_TRY(enqueue_scan(ix, qd, nullptr, nullptr, nq, k, Dd, Id, P.id_offset, w.scan_scratch, nullptr, 0, nq, 0, w.filter.allow,
                             st));
        B2F_TRY(main_event(1));
        n_main++;
    } else {
        const int nq_pad = plan.nq_tiles * 128;
        ix->st.last_kprime = kp;
        B2F_TRY(refresh_host_stats(ix, st));
        for (int c0 = 0; c0 < nq; c0 += chunk_nq) {
            const int cn = nq - c0 < chunk_nq ? nq - c0 : chunk_nq;  // queries in this pass (the plan covers chunk_nq)
            const float* qc = qd + (int64_t)c0 * ix->d;
            // one launch: bf16 copy / norms of the queries, reset the shared thresholds, clear the counters (first pass)
            B2F_TRY(launch_prep_queries(qc, cn, nq_pad, ix->d, w.pq.qb, ix->dpad, w.pq.qnorm, w.pq.qerr, w.pq.qconst, scan_centre(ix),
                                        reinterpret_cast<uint32_t*>(w.counters), c0 == 0 ? 16 : 0,
                                        reinterpret_cast<uint32_t*>(w.lists.shared_thr),
                                        plan.list_mode ? (int64_t)nq_pad * plan.nlists : 0, st));
            B2F_TRY(main_event(0));
            B2F_TRY(launch_tensor_scan(ix->scan, ix->dpad, tensor_bias(ix, w.filter), ix->ntotal, ix->metric, w.pq.qb, cn, nq_pad, plan,
                                       w.pk, w.pi, w.lists, st));
            B2F_TRY(main_event(1));
            n_main++;
            // the re-rank writes faiss-formatted results directly (no finalize launch)
            RerankArgs ra = rerank_args(ix, qc, w.pq, cn, k, kp, Dd + (int64_t)c0 * k, Id + (int64_t)c0 * k, P.id_offset,
                                        w.fail_list, w.counters);
            ra.cand_key = w.ck;
            ra.cand_id = w.ci;
            ra.certify = certify;
            ra.fail_tau = w.fail_tau;
            ra.q_base = c0;
            if (plan.list_mode) {
                // K3b + K4 + finalize fused: per query, merge the lists, re-rank exactly, certify, write (D, I)
                B2F_TRY(launch_merge_lists(w.lists, cn, plan, reinterpret_cast<unsigned long long*>(w.counters + 2), ra, st));
                count_launches(ix, 3);
            } else {
                B2F_TRY(launch_merge_parts(w.pk, w.pi, cn, plan.nsplits, kp, kp, w.ck, w.ci, st));
                B2F_TRY(launch_rerank(ra, st));
                count_launches(ix, 4);
            }
        }  // query chunks
        int32_t* scan_list = w.fail_list;
        int32_t* scan_counters = w.counters;
        int range_served = 0;
        if (ix->adapt.range_mode && certify && w.fail_tau)
            B2F_TRY(range_pass(ix, bump, w, qd, nq, k, kp, Dd, Id, P.id_offset, st, &scan_list, &scan_counters, &range_served));
        // Closing kernel: the exact scan over the queries that could not be certified.  The count lives on the
        // device -- with none (the usual case) the kernel publishes the counters and exits -- so the host never
        // waits inside a search and consecutive searches run back to back on the GPU.
        B2F_TRY(enqueue_scan(ix, qd, scan_list, scan_counters, 0, k, Dd, Id, P.id_offset, w.scan_scratch, scan_counters, ++ix->seq, nq,
                             certify, w.filter.allow, st));
        if (range_served) {
            ix->adapt.range_ran_seq = ix->seq;
            ix->adapt.range_ran_nfail = range_served;
        }
    }
    if (slot) {
        B2F_CUDA(cudaEventRecord(slot->t1, st));
        slot->n_main = n_main;
        slot->pending = true;
    }
    if (host) {
        B2F_CUDA(cudaMemcpyAsync(D, Dd, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, st));
        B2F_CUDA(cudaMemcpyAsync(I, Id, (size_t)nq * k * 8, cudaMemcpyDeviceToHost, st));
    }
    B2F_TRY(record_search(ix, st));
    if (host) {
        B2F_CUDA(cudaStreamSynchronize(st));  // faiss semantics: results are in the caller's arrays on return
        harvest_flag(ix);
    }
    return B2F_OK;
}

// ---- range search ----------------------------------------------------------------------------------
// The result of one range search: lims on the host, the hits in buffers the library owns (faiss's RangeSearchResult).
// D / I grow while the chunks are counted; a buffer they outgrow may still be read by copies in flight, so it is freed
// with the others when the result is destroyed.
struct b2f_range_result {
    int device = 0;
    std::vector<int64_t> lims;
    float* D = nullptr;
    int64_t* I = nullptr;
    int64_t cap = 0;
    std::vector<void*> retired;
    cudaStream_t st = nullptr;       // the stream the search ran on
    cudaEvent_t done = nullptr;      // recorded behind the last write to, or device copy from, D / I
    int64_t info[5] = {0, 0, 0, 0, 0};
};

// A range search plans its tensor pass for the threshold alone: nothing is pruned or vouched for, so k' only sizes the
// (unused) voucher state.  Every row at or below a query's threshold must fit its lists, and a query whose lists hold more
// than kRangeHitsMax entries goes to the exact range scan anyway: lists of 2 x kRangeHitsMax / nlists entries, at least
// kRangeListCap.
constexpr int kRangeSearchKp = 32;

static int plan_range_search(int nq, int64_t n, int d, TensorScanPlan* plan) {
    if (plan_tensor_scan(nq, n, d, kRangeSearchKp, false, plan) != B2F_OK || !plan->list_mode) return B2F_EINVAL;
    int cap = (int)align_up((size_t)(2 * kRangeHitsMax / plan->nlists), 64);
    if (cap < kRangeListCap) cap = kRangeListCap;
    plan->list_cap = cap < 1024 ? cap : 1024;
    return B2F_OK;
}

// What one chunk of a range search carves from the workspace, in one order (measured over a null base first)
struct RangeSearchWs {
    float* q = nullptr;              // host queries: the chunk's device copy
    int32_t* count = nullptr;        // [chunk] hits per query
    int32_t* staged = nullptr;       // [chunk] hits the tensor path staged per query
    int32_t* scan_list = nullptr;    // [chunk] queries left to the exact range scan
    int64_t* lims = nullptr;         // [chunk + 1] chunk-local offsets
    int32_t* tile_counts = nullptr;  // [chunk][ntiles] the exact range scan's hits per row tile
    PassQueries pq{};                // tensor path from here on
    float* thr = nullptr;
    int32_t* counters = nullptr;     // [0] queries in scan_list, [8..11] K2's tickets
    TensorScanLists lists{};
    float* skey = nullptr;           // [chunk][kRangeHitsMax] staged hits: exact key, row id
    int32_t* sid = nullptr;
    FilterWs filter{};               // filtered search
};

static RangeSearchWs carve_range_search(Bump& b, const b2f_index* ix, int cn, bool host, bool tensor, const TensorScanPlan& plan,
                                        int ntiles, const b2f_selector* sel, int64_t id_offset) {
    RangeSearchWs w;
    w.filter = carve_filter(b, ix, sel, id_offset, host, tensor);
    if (host) w.q = b.take<float>((size_t)cn * ix->d);
    w.count = b.take<int32_t>(cn);
    w.staged = b.take<int32_t>(cn);
    w.scan_list = b.take<int32_t>(cn);
    w.lims = b.take<int64_t>((size_t)cn + 1);
    w.tile_counts = b.take<int32_t>((size_t)cn * ntiles);
    if (!tensor) return w;
    const size_t nq_pad = (size_t)plan.nq_tiles * 128;
    w.pq = take_queries(b, nq_pad, ix->dpad);
    w.thr = b.take<float>(nq_pad);
    w.counters = b.take<int32_t>(16);
    w.lists = take_lists(b, plan);
    w.lists.die_ctr = w.counters + 8;
    w.lists.range_thr = w.thr;
    w.skey = b.take<float>((size_t)cn * kRangeHitsMax);
    w.sid = b.take<int32_t>((size_t)cn * kRangeHitsMax);
    return w;
}

// D / I of r hold at least `need` hits (contents kept)
static int range_result_reserve(b2f_range_result* r, int64_t need, cudaStream_t st) {
    if (need <= r->cap) return B2F_OK;
    int64_t cap = 2 * r->cap > need ? 2 * r->cap : need;
    float* D = nullptr;
    int64_t* I = nullptr;
    cudaError_t e = cudaMalloc(&D, (size_t)cap * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&I, (size_t)cap * sizeof(int64_t));
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaFree(D);
        set_error("range search: %lld hits (%.2f GB of distances and labels) do not fit device memory: %s", (long long)need,
                  (double)need * 12 / 1e9, cudaGetErrorString(e));
        return B2F_ENOMEM;
    }
    if (r->cap > 0) {
        B2F_CUDA(cudaMemcpyAsync(D, r->D, (size_t)r->cap * sizeof(float), cudaMemcpyDeviceToDevice, st));
        B2F_CUDA(cudaMemcpyAsync(I, r->I, (size_t)r->cap * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    }
    if (r->D) r->retired.push_back(r->D);
    if (r->I) r->retired.push_back(r->I);
    r->D = D;
    r->I = I;
    r->cap = cap;
    return B2F_OK;
}

// The batch in chunks of at most kRangeCap queries.  A chunk goes to the tensor path when a LIST-mode pass can be planned
// for it (halving the chunk until one can); with none even for one query, the chunk goes to the exact range scan.  Per chunk:
// [tensor: prep, thresholds, K2 listing every row at or below thr(tau), collect] -> exact range scan count pass over what
// the lists could not answer (or over the whole chunk) -> offsets -> ONE host sync for the chunk's lims -> emit.
static int range_search_locked(b2f_index* ix, int nq, const float* q, float radius, int32_t mem, void* stream,
                               const b2f_search_params* params, const b2f_selector* sel, b2f_range_result* r) {
    b2f_search_params P{};
    if (params) P = *params;
    const bool l2 = ix->metric == B2F_METRIC_L2;
    r->lims.assign((size_t)nq + 1, 0);
    if (nq == 0 || ix->ntotal == 0 || (l2 && !(radius > 0.f))) return B2F_OK;   // nothing can be a hit
    DeviceGuard g(ix->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : ix->stream;
    r->st = st;
    B2F_TRY(enter_stream(ix, g, st));
    B2F_TRY(order_after(st, ix->stream, ix));
    const bool host = mem == B2F_MEM_HOST;
    const float tau = l2 ? radius : -radius;   // hit <=> exact key < tau
    int64_t launches = 0, syncs = ix->stats_dirty ? 1 : 0;
    B2F_TRY(refresh_host_stats(ix, st));
    const float max_row_norm = sqrtf(ix->host_stats[0]), max_row_err = sqrtf(ix->host_stats[1]);
    // the threshold is the certification bound inverted: with a non-finite row in the index it bounds nothing
    const bool bound_ok = isfinite(max_row_norm) && isfinite(max_row_err) && isfinite(ix->mu_norm);
    const bool want_tensor = bound_ok && P.algo != B2F_ALGO_SCAN && !(P.algo == B2F_ALGO_AUTO && nq <= P.scan_max_nq);
    RerankArgs a{};
    a.rows = stored_rows(ix);
    const RangeScanGeometry geo = range_scan_geometry(ix->ntotal);
    B2F_TRY(ensure_pinned(ix, ((size_t)kRangeCap + 2) * sizeof(int64_t)));
    int64_t* lims_h = reinterpret_cast<int64_t*>(ix->pinned);
    int64_t base = 0;
    for (int c0 = 0; c0 < nq;) {
        int cn = nq - c0 < kRangeCap ? nq - c0 : kRangeCap;
        TensorScanPlan plan{};
        bool tensor = false;
        for (int m = cn; want_tensor && !tensor; m = (m + 1) / 2) {
            if (plan_range_search(m, ix->ntotal, ix->d, &plan) == B2F_OK) {
                tensor = true;
                cn = m;
            } else if (m == 1) {
                break;
            }
        }
        RangeSearchWs w;
        bool grew = false;
        B2F_TRY(carve_ws(ix, 0, [&](Bump& b) { w = carve_range_search(b, ix, cn, host, tensor, plan, geo.ntiles, sel, P.id_offset); },
                         "range search", &grew));
        syncs += grew;
        const float* qc = host ? w.q : q + (int64_t)c0 * ix->d;
        if (host) B2F_CUDA(cudaMemcpyAsync(w.q, q + (int64_t)c0 * ix->d, (size_t)cn * ix->d * 4, cudaMemcpyHostToDevice, st));
        a.q = qc;
        // (built per chunk: a later chunk may re-allocate the workspace)
        int filter_launches = 0;
        B2F_TRY(build_filter(ix, sel, mem, P.id_offset, w.filter, st, &filter_launches));
        launches += filter_launches;
        a.allow = w.filter.allow;
        if (tensor) {
            const int nq_pad = plan.nq_tiles * 128;
            B2F_TRY(launch_prep_queries(qc, cn, nq_pad, ix->d, w.pq.qb, ix->dpad, w.pq.qnorm, w.pq.qerr, w.pq.qconst, scan_centre(ix),
                                        reinterpret_cast<uint32_t*>(w.counters), 16, nullptr, 0, st));
            B2F_TRY(launch_range_thresholds(nullptr, tau, nullptr, cn, ix->d, ix->metric, w.pq.qnorm, w.pq.qerr, w.pq.qconst,
                                            max_row_norm, max_row_err, ix->mu_norm, w.thr, st));
            B2F_TRY(launch_tensor_scan(ix->scan, ix->dpad, tensor_bias(ix, w.filter), ix->ntotal, ix->metric, w.pq.qb, cn, nq_pad, plan,
                                       nullptr, nullptr, w.lists, st));
            B2F_TRY(launch_range_collect(w.lists, cn, plan, tau, a, w.skey, w.sid, w.staged, w.count, w.scan_list, w.counters, st));
            launches += 4;
        } else {
            B2F_CUDA(cudaMemsetAsync(w.count, 0, (size_t)cn * 4, st));
        }
        const int32_t* list = tensor ? w.scan_list : nullptr;
        const int32_t* nlist = tensor ? w.counters : nullptr;
        B2F_TRY(launch_range_scan(a, tau, list, nlist, cn, w.tile_counts, w.count, nullptr, 0, nullptr, nullptr, 0, false, st));
        B2F_TRY(launch_range_offsets(w.count, cn, w.lims, st));
        launches += 2;
        B2F_CUDA(cudaMemcpyAsync(lims_h, w.lims, ((size_t)cn + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        if (tensor) B2F_CUDA(cudaMemcpyAsync(lims_h + kRangeCap + 1, w.counters, 4, cudaMemcpyDeviceToHost, st));
        B2F_CUDA(cudaStreamSynchronize(st));
        syncs++;
        const int64_t hits = lims_h[cn];
        const int nscan = tensor ? *reinterpret_cast<const int32_t*>(lims_h + kRangeCap + 1) : cn;
        for (int i = 0; i <= cn; i++) r->lims[(size_t)c0 + i] = base + lims_h[i];
        if (hits > 0) {
            B2F_TRY(range_result_reserve(r, base + hits, st));
            if (tensor) {
                B2F_TRY(launch_range_emit(w.skey, w.sid, w.staged, w.lims, cn, base, ix->metric, r->D, r->I, P.id_offset, st));
                launches++;
            }
            if (nscan > 0) {
                B2F_TRY(launch_range_scan(a, tau, list, nlist, cn, w.tile_counts, w.count, w.lims, base, r->D, r->I, P.id_offset, true, st));
                launches++;
            }
        }
        r->info[1] += cn - nscan;
        r->info[2] += nscan;
        base += hits;
        c0 += cn;
    }
    r->info[0] = base;
    r->info[3] = launches;
    r->info[4] = syncs;
    ix->st.launches += launches;
    if (!r->done) B2F_CUDA(cudaEventCreateWithFlags(&r->done, cudaEventDisableTiming));
    B2F_CUDA(cudaEventRecord(r->done, st));
    return record_search(ix, st);
}

extern "C" {

int b2f_range_result_destroy(b2f_range_result* r) {
    if (!r) return B2F_OK;
    DeviceGuard g(r->device);
    if (r->done) {
        cudaEventSynchronize(r->done);
        cudaEventDestroy(r->done);
    } else if (r->st) {
        cudaStreamSynchronize(r->st);   // a search that failed half way may still write D / I
    }
    cudaGetLastError();
    cudaFree(r->D);
    cudaFree(r->I);
    for (void* p : r->retired) cudaFree(p);
    delete r;
    return B2F_OK;
}

int b2f_index_range_search(b2f_index* ix, int64_t nq, const float* q, float radius, int32_t mem, void* stream,
                           const b2f_search_params* params, b2f_range_result** out) {
    return b2f_index_range_search_filtered(ix, nq, q, radius, mem, stream, params, nullptr, out);
}

int b2f_index_range_search_filtered(b2f_index* ix, int64_t nq, const float* q, float radius, int32_t mem, void* stream,
                                    const b2f_search_params* params, const b2f_selector* sel, b2f_range_result** out) {
    if (!out) {
        set_error("range_search: out is NULL");
        return B2F_EINVAL;
    }
    *out = nullptr;
    B2F_TRY(check_selector(sel));
    if (!ix) {
        set_error("index is NULL");
        return B2F_EINVAL;
    }
    if (nq < 0 || nq > (1 << 24) || (nq > 0 && !q)) {
        set_error("range_search: bad arguments (nq=%lld)", (long long)nq);
        return B2F_EINVAL;
    }
    if (radius != radius) {
        set_error("range_search: radius is NaN");
        return B2F_EINVAL;
    }
    b2f_range_result* r = new (std::nothrow) b2f_range_result();
    if (!r) {
        set_error("range_search: out of host memory");
        return B2F_ENOMEM;
    }
    r->device = ix->device;
    int rc;
    {
        std::lock_guard<std::mutex> lk(ix->mu);
        rc = range_search_locked(ix, (int)nq, q, radius, mem, stream, params, sel, r);
    }
    if (rc != B2F_OK) {
        b2f_range_result_destroy(r);
        return rc;
    }
    *out = r;
    return B2F_OK;
}

int b2f_range_result_lims(const b2f_range_result* r, int64_t* lims) {
    if (!r || !lims) {
        set_error("range_result_lims: NULL argument");
        return B2F_EINVAL;
    }
    memcpy(lims, r->lims.data(), r->lims.size() * sizeof(int64_t));
    return B2F_OK;
}

int b2f_range_result_fetch(b2f_range_result* r, float* D, int64_t* I, int32_t mem, void* stream) {
    const int64_t hits = r ? r->lims.back() : 0;
    if (!r || (hits > 0 && (!D || !I))) {
        set_error("range_result_fetch: NULL argument");
        return B2F_EINVAL;
    }
    if (hits == 0) return B2F_OK;
    DeviceGuard g(r->device);
    if (mem == B2F_MEM_HOST) {
        B2F_CUDA(cudaEventSynchronize(r->done));
        B2F_CUDA(cudaMemcpy(D, r->D, (size_t)hits * sizeof(float), cudaMemcpyDeviceToHost));
        B2F_CUDA(cudaMemcpy(I, r->I, (size_t)hits * sizeof(int64_t), cudaMemcpyDeviceToHost));
        return B2F_OK;
    }
    cudaStream_t st = stream ? (cudaStream_t)stream : r->st;
    B2F_CUDA(cudaStreamWaitEvent(st, r->done, 0));
    B2F_CUDA(cudaMemcpyAsync(D, r->D, (size_t)hits * sizeof(float), cudaMemcpyDeviceToDevice, st));
    B2F_CUDA(cudaMemcpyAsync(I, r->I, (size_t)hits * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    B2F_CUDA(cudaEventRecord(r->done, st));   // destroy waits for these copies
    return B2F_OK;
}

int b2f_range_result_info(const b2f_range_result* r, int64_t out[5]) {
    if (!r || !out) {
        set_error("range_result_info: NULL argument");
        return B2F_EINVAL;
    }
    for (int i = 0; i < 5; i++) out[i] = r->info[i];
    return B2F_OK;
}

}  // extern "C"

extern "C" {

int b2f_index_search(b2f_index* ix, int64_t nq, const float* q, int64_t k, float* D, int64_t* I, int32_t mem, void* stream,
                     const b2f_search_params* params) {
    return b2f_index_search_filtered(ix, nq, q, k, D, I, mem, stream, params, nullptr);
}

int b2f_index_search_filtered(b2f_index* ix, int64_t nq, const float* q, int64_t k, float* D, int64_t* I, int32_t mem,
                              void* stream, const b2f_search_params* params, const b2f_selector* sel) {
    B2F_TRY(check_selector(sel));
    if (!ix) {
        set_error("index is NULL");
        return B2F_EINVAL;
    }
    std::lock_guard<std::mutex> lk(ix->mu);
    return search_locked(ix, nq, q, k, D, I, mem, stream, params, sel);
}

int b2f_index_search_pooled(b2f_index* ix, const float* hidden, const int64_t* mask, int64_t B, int64_t T, int32_t pool,
                            int32_t normalize, int64_t k, float* D, int64_t* I, void* stream, const b2f_search_params* params) {
    if (!ix || B < 0 || (B > 0 && (!hidden || !D || !I))) {
        set_error("search_pooled: bad arguments");
        return B2F_EINVAL;
    }
    if (B == 0) return B2F_OK;
    float* qbuf = nullptr;
    std::lock_guard<std::mutex> lk(ix->mu);   // held across pooling AND the search: the pooled queries live in ix->qpool
    {
        DeviceGuard g(ix->device);
        cudaStream_t st = stream ? (cudaStream_t)stream : ix->stream;
        B2F_TRY(enter_stream(ix, g, st));
        // pooled queries live in their own grow-only buffer (the search below carves the workspace itself)
        const size_t need = (size_t)B * ix->d * sizeof(float);
        if (need > ix->qpool_bytes) {
            if (ix->search_recorded) B2F_CUDA(cudaEventSynchronize(ix->ev_done));
            cudaFree(ix->qpool);
            ix->qpool = nullptr;
            ix->qpool_bytes = 0;
            if (cudaMalloc(&ix->qpool, need + (need >> 2)) != cudaSuccess) {
                cudaGetLastError();
                set_error("search_pooled: cudaMalloc(%zu) failed", need);
                return B2F_ENOMEM;
            }
            ix->qpool_bytes = need + (need >> 2);
        }
        qbuf = ix->qpool;
        B2F_TRY(launch_pool(hidden, mask, B, T, ix->d, pool, normalize, qbuf, st));
        ix->st.launches++;
    }
    return search_locked(ix, B, qbuf, k, D, I, B2F_MEM_DEVICE, stream, params, nullptr);
}

int b2f_index_reconstruct(b2f_index* ix, int64_t i0, int64_t n, float* out, int32_t mem, void* stream) {
    if (!ix || !out || n < 0) {
        set_error("reconstruct: bad arguments");
        return B2F_EINVAL;
    }
    if (i0 < 0 || i0 + n > ix->ntotal) {
        set_error("reconstruct: rows [%lld, %lld) out of range [0, %lld)", (long long)i0, (long long)(i0 + n), (long long)ix->ntotal);
        return B2F_ERANGE;
    }
    if (n == 0) return B2F_OK;
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : ix->stream;
    B2F_TRY(enter_stream(ix, g, st));
    B2F_TRY(order_after(st, ix->stream, ix));
    const size_t bytes = (size_t)n * ix->d * 4;
    if (ix->storage == B2F_STORE_F32) {
        B2F_CUDA(cudaMemcpyAsync(out, ix->rows_f32 + i0 * ix->d, bytes, mem == B2F_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, st));
    } else if (mem == B2F_MEM_DEVICE) {
        B2F_TRY(launch_bf16_to_f32(ix->scan + i0 * ix->dpad, ix->dpad, n, ix->d, scan_centre(ix), out, st));
        ix->st.launches++;
    } else {
        B2F_TRY(ensure_ws(ix, bytes + 4096));
        B2F_TRY(launch_bf16_to_f32(ix->scan + i0 * ix->dpad, ix->dpad, n, ix->d, scan_centre(ix), reinterpret_cast<float*>(ix->ws), st));
        ix->st.launches++;
        B2F_CUDA(cudaMemcpyAsync(out, ix->ws, bytes, cudaMemcpyDeviceToHost, st));
    }
    if (mem == B2F_MEM_HOST) B2F_CUDA(cudaStreamSynchronize(st));
    return B2F_OK;
}

// ---- remove_ids -------------------------------------------------------------------------------------
// faiss IndexFlatCodes::remove_ids: the rows of `runs` (sorted, disjoint, inside [0, ntotal)) go, the survivors keep their
// order and are renumbered from 0.  Every surviving row keeps its bits in all three arrays; the centre stays; the stats are
// taken again over the survivors, so a removed non-finite row no longer spoils certification; Adapt stays (speed only).
static int remove_runs_locked(b2f_index* ix, const std::vector<int64_t>& runs, int64_t* nremoved) {
    const int64_t nr = (int64_t)runs.size() / 2;
    int64_t removed = 0;
    for (int64_t j = 0; j < nr; j++) removed += runs[2 * j + 1] - runs[2 * j];
    if (nremoved) *nremoved = removed;
    if (removed == 0) return B2F_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = ix->stream;
    B2F_TRY(enter_stream(ix, g, st));
    // Until now rows were only ever appended.  A search, range search, device reconstruct or write may still be reading
    // them on any stream: all of it finishes before a row is overwritten (as before ensure_capacity's copies).
    B2F_CUDA(cudaDeviceSynchronize());
    const int64_t first = runs[0], n_new = ix->ntotal - removed;
    if (ix->ntotal - first > removed) {   // survivors above the first removed row: they move
        struct Arr {
            void* base;
            int64_t row_bytes;
        } arrs[3] = {{ix->rows_f32, (int64_t)ix->d * 4}, {ix->scan, ix->dpad * 2}, {ix->norms, 4}};
        int64_t tiles = 0;
        for (const Arr& a : arrs)
            if (a.base) tiles = std::max(tiles, remove_tiles(first, ix->ntotal, a.row_bytes));
        std::vector<int64_t> words;
        remove_runs_layout(runs, words);
        int64_t* runs_dev = nullptr;
        RemoveSpan* spans = nullptr;
        B2F_TRY(carve_ws(ix, 0, [&](Bump& b) {
            runs_dev = b.take<int64_t>(words.size());
            spans = b.take<RemoveSpan>((size_t)tiles);
        }, "remove"));
        B2F_CUDA(cudaMemcpyAsync(runs_dev, words.data(), words.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        const RemoveRuns rr = remove_runs_view(runs_dev, nr);
        const int64_t need = 1 + tiles;
        if (need > ix->rm_flag_words) {
            cudaFree(ix->rm_flags);
            ix->rm_flags = nullptr;
            ix->rm_flag_words = 0;
            cudaError_t e = cudaMalloc(&ix->rm_flags, (size_t)need * 4);
            if (e == cudaSuccess) e = cudaMemset(ix->rm_flags, 0, (size_t)need * 4);
            if (e != cudaSuccess) {
                cudaGetLastError();
                set_error("remove: %lld flag words: %s", (long long)need, cudaGetErrorString(e));
                return B2F_ENOMEM;
            }
            ix->rm_flag_words = need;
            ix->rm_epoch = 0;
        }
        for (const Arr& a : arrs) {
            if (!a.base) continue;   // bf16 storage keeps no fp32 rows
            if (++ix->rm_epoch == 0) ix->rm_epoch = 1;   // 0 is what fresh flags hold
            B2F_TRY(launch_remove_compact(a.base, a.row_bytes, rr, first, ix->ntotal, spans, ix->rm_flags, ix->rm_epoch, st));
            ix->st.launches += 2;
        }
    }
    B2F_CUDA(cudaMemsetAsync(ix->stats, 0, 2 * sizeof(float), st));
    const float* mu = scan_centre(ix);
    if (n_new > 0) {
        if (ix->storage == B2F_STORE_F32)   // ingest's own arithmetic over the fp32 rows, writing nothing but the stats
            B2F_TRY(launch_ingest(ix->rows_f32, n_new, ix->d, nullptr, nullptr, ix->dpad, nullptr, ix->stats, mu, 0, 0, st));
        else
            B2F_TRY(launch_scan_stats(ix->scan, n_new, ix->d, ix->dpad, mu, ix->stats, st));
        ix->st.launches++;
    }
    ix->ntotal = n_new;
    ix->stats_dirty = true;
    B2F_TRY(record_ingest(ix, st));
    B2F_CUDA(cudaStreamSynchronize(st));   // faiss semantics: done on return
    return B2F_OK;
}

int b2f_index_remove_ids(b2f_index* ix, int64_t n, const int64_t* ids, int64_t* nremoved) {
    if (nremoved) *nremoved = 0;
    if (!ix || n < 0 || (n > 0 && !ids)) {
        set_error("remove_ids: bad arguments");
        return B2F_EINVAL;
    }
    std::lock_guard<std::mutex> lk(ix->mu);
    return remove_runs_locked(ix, remove_runs_from_ids(ix->ntotal, n, ids), nremoved);
}

int b2f_index_remove_range(b2f_index* ix, int64_t imin, int64_t imax, int64_t* nremoved) {
    if (nremoved) *nremoved = 0;
    if (!ix) {
        set_error("index is NULL");
        return B2F_EINVAL;
    }
    std::lock_guard<std::mutex> lk(ix->mu);
    const int64_t a = imin > 0 ? imin : 0, b = imax < ix->ntotal ? imax : ix->ntotal;
    std::vector<int64_t> runs;
    if (a < b) runs = {a, b};
    return remove_runs_locked(ix, runs, nremoved);
}

int b2f_remove_plan(int64_t ntotal, int64_t n, const int64_t* ids, int64_t row_bytes, int64_t* runs, int64_t* nruns, int64_t* dest,
                    int64_t* tiles, int64_t cap, int64_t* ntiles) {
    if (ntotal < 0 || n < 0 || (n > 0 && !ids) || row_bytes <= 0 || !nruns || !ntiles || cap < 0) {
        set_error("remove_plan: bad arguments");
        return B2F_EINVAL;
    }
    const std::vector<int64_t> r = remove_runs_from_ids(ntotal, n, ids);
    const int64_t nr = (int64_t)r.size() / 2;
    *nruns = nr;
    if (runs) memcpy(runs, r.data(), r.size() * sizeof(int64_t));
    std::vector<int64_t> words;
    remove_runs_layout(r, words);
    const RemoveRuns rr = remove_runs_view(words.data(), nr);
    if (dest)
        for (int64_t s = 0; s < ntotal; s++) dest[s] = remove_dest(rr, s, 0, nr);
    *ntiles = 0;
    if (nr == 0) return B2F_OK;
    const int64_t first = r[0], tr = remove_tile_rows(row_bytes);
    *ntiles = remove_tiles(first, ntotal, row_bytes);
    for (int64_t t = 0; tiles && t < *ntiles && t < cap; t++) {
        const RemoveSpan sp = remove_tile_span(rr, first, ntotal, tr, t);
        tiles[3 * t] = sp.s0;
        tiles[3 * t + 1] = sp.w0;
        tiles[3 * t + 2] = sp.w1;
    }
    return B2F_OK;
}

// ---- file I/O (FAISS IndexFlat layout; see include/b200flat.h) --------------------------------------
static const size_t kIoChunk = 32u << 20;

int b2f_index_write(b2f_index* ix, const char* path) {
    if (!ix || !path) {
        set_error("write: bad arguments");
        return B2F_EINVAL;
    }
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    B2F_TRY(enter_stream(ix, g, ix->stream));
    FILE* f = fopen(path, "wb");
    if (!f) {
        set_error("could not open %s for writing", path);
        return B2F_EIO;
    }
    const char* cc = ix->metric == B2F_METRIC_L2 ? "IxF2" : "IxFI";
    const int32_t d32 = ix->d, mt = ix->metric;
    const int64_t nt = ix->ntotal, dummy = 1 << 20;
    const uint8_t tr = 1;
    const uint64_t sz = (uint64_t)ix->ntotal * ix->d;
    bool ok = fwrite(cc, 1, 4, f) == 4 && fwrite(&d32, 4, 1, f) == 1 && fwrite(&nt, 8, 1, f) == 1 &&
              fwrite(&dummy, 8, 1, f) == 1 && fwrite(&dummy, 8, 1, f) == 1 && fwrite(&tr, 1, 1, f) == 1 &&
              fwrite(&mt, 4, 1, f) == 1 && fwrite(&sz, 8, 1, f) == 1;
    int rc = B2F_OK;
    if (ok && ix->ntotal > 0) {
        const int64_t rows_per = (int64_t)(kIoChunk / ((size_t)ix->d * 4)) > 0 ? (int64_t)(kIoChunk / ((size_t)ix->d * 4)) : 1;
        const size_t cbytes = (size_t)rows_per * ix->d * 4;
        rc = ensure_pinned(ix, 2 * cbytes);
        if (rc == B2F_OK && ix->storage == B2F_STORE_BF16) rc = ensure_ws(ix, 2 * cbytes + 4096);
        cudaEvent_t evs[2] = {get_event(ix, 1), get_event(ix, 2)};
        int64_t pending_rows[2] = {0, 0};
        int slot = 0;
        // double-buffered: D2H of chunk i+1 overlaps fwrite of chunk i
        for (int64_t r0 = 0; rc == B2F_OK && ok && r0 < ix->ntotal + rows_per; r0 += rows_per, slot ^= 1) {
            if (r0 < ix->ntotal) {
                const int64_t m = ix->ntotal - r0 < rows_per ? ix->ntotal - r0 : rows_per;
                char* hbuf = ix->pinned + (size_t)slot * cbytes;
                cudaError_t e;
                if (ix->storage == B2F_STORE_F32) {
                    e = cudaMemcpyAsync(hbuf, ix->rows_f32 + r0 * ix->d, (size_t)m * ix->d * 4, cudaMemcpyDeviceToHost, ix->stream);
                } else {
                    float* dbuf = reinterpret_cast<float*>(ix->ws + (size_t)slot * cbytes);
                    rc = launch_bf16_to_f32(ix->scan + r0 * ix->dpad, ix->dpad, m, ix->d, scan_centre(ix), dbuf, ix->stream);
                    ix->st.launches++;
                    e = cudaMemcpyAsync(hbuf, dbuf, (size_t)m * ix->d * 4, cudaMemcpyDeviceToHost, ix->stream);
                }
                if (e == cudaSuccess) e = cudaEventRecord(evs[slot], ix->stream);
                if (e != cudaSuccess) {
                    set_error("write: device read failed: %s", cudaGetErrorString(e));
                    rc = B2F_ECUDA;
                }
                pending_rows[slot] = m;
            } else {
                pending_rows[slot] = 0;
            }
            const int prev = slot ^ 1;
            if (rc == B2F_OK && r0 > 0 && pending_rows[prev] > 0) {
                if (cudaEventSynchronize(evs[prev]) != cudaSuccess) {
                    set_error("write: event sync failed");
                    rc = B2F_ECUDA;
                } else {
                    const size_t cnt = (size_t)pending_rows[prev] * ix->d;
                    ok = fwrite(ix->pinned + (size_t)prev * cbytes, 4, cnt, f) == cnt;
                    pending_rows[prev] = 0;
                }
            }
        }
    }
    if (fclose(f) != 0) ok = false;
    if (rc != B2F_OK) return rc;
    if (!ok) {
        set_error("short write to %s", path);
        return B2F_EIO;
    }
    return B2F_OK;
}

int b2f_index_read(const char* path, int32_t storage, int32_t device, b2f_index** out) {
    if (!path || !out) {
        set_error("read: bad arguments");
        return B2F_EINVAL;
    }
    *out = nullptr;
    FILE* f = fopen(path, "rb");
    if (!f) {
        set_error("could not open %s for reading", path);
        return B2F_EIO;
    }
    char cc[4];
    int32_t d32 = 0, mt = 0;
    int64_t nt = 0, dm[2];
    uint8_t tr = 0;
    uint64_t sz = 0;
    bool ok = fread(cc, 1, 4, f) == 4;
    if (ok && memcmp(cc, "IxF2", 4) != 0 && memcmp(cc, "IxFI", 4) != 0 && memcmp(cc, "IxFl", 4) != 0) {
        fclose(f);
        set_error("%s is not an IndexFlat file (fourcc %.4s)", path, cc);
        return B2F_EFORMAT;
    }
    ok = ok && fread(&d32, 4, 1, f) == 1 && fread(&nt, 8, 1, f) == 1 && fread(dm, 8, 2, f) == 2 &&
         fread(&tr, 1, 1, f) == 1 && fread(&mt, 4, 1, f) == 1;
    if (ok && mt > 1) {
        float arg;
        ok = fread(&arg, 4, 1, f) == 1;
    }
    ok = ok && fread(&sz, 8, 1, f) == 1;
    if (!ok || d32 <= 0 || nt < 0 || sz != (uint64_t)nt * (uint64_t)d32) {
        fclose(f);
        set_error("%s: truncated or inconsistent IndexFlat header", path);
        return B2F_EFORMAT;
    }
    if (mt != B2F_METRIC_L2 && mt != B2F_METRIC_INNER_PRODUCT) {
        fclose(f);
        set_error("%s: metric_type %d is not supported (only L2 and inner product)", path, mt);
        return B2F_EFORMAT;
    }
    b2f_index* ix = nullptr;
    int rc = b2f_index_create(d32, mt, storage, device, &ix);
    if (rc != B2F_OK) {
        fclose(f);
        return rc;
    }
    {
        DeviceGuard g(device);
        rc = ensure_capacity(ix, nt);
        const int64_t piece = rows_in(kIoChunk, d32);
        const size_t cbytes = (size_t)piece * d32 * 4;
        if (rc == B2F_OK && nt > 0) rc = ensure_pinned(ix, 2 * cbytes);
        // The rows are ingested as one add of nt rows, through two pinned slots: the fread of a piece overlaps the H2D and
        // ingest of the one before.  The centre's rows are read once more first (take_centre), so every piece seeks to its rows.
        const long payload = ftell(f);
        cudaEvent_t evs[2] = {get_event(ix, 1), get_event(ix, 2)};
        int64_t pieces = 0;
        if (rc == B2F_OK && nt > 0)
            rc = ingest_call(ix, nt, piece, nullptr, ix->stream, [&](int64_t r0, int64_t m, float* dst) {
                const int slot = (int)(pieces++ & 1);
                char* hbuf = ix->pinned + (size_t)slot * cbytes;
                if (pieces > 2) B2F_CUDA(cudaEventSynchronize(evs[slot]));   // the slot's previous H2D has finished
                const size_t cnt = (size_t)m * d32;
                if (fseek(f, payload + (long)((size_t)r0 * d32 * 4), SEEK_SET) != 0 || fread(hbuf, 4, cnt, f) != cnt) {
                    set_error("%s: truncated payload", path);
                    return B2F_EFORMAT;
                }
                B2F_CUDA(cudaMemcpyAsync(dst, hbuf, cnt * 4, cudaMemcpyHostToDevice, ix->stream));
                B2F_CUDA(cudaEventRecord(evs[slot], ix->stream));
                return B2F_OK;
            });
        if (rc == B2F_OK && cudaStreamSynchronize(ix->stream) != cudaSuccess) {
            set_error("read: stream sync failed");
            rc = B2F_ECUDA;
        }
    }
    fclose(f);
    if (rc != B2F_OK) {
        b2f_index_destroy(ix);
        return rc;
    }
    *out = ix;
    return B2F_OK;
}

}  // extern "C"
