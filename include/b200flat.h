/*
 * b200flat.h -- C ABI of the B200-native flat (exact) vector-search engine.
 *
 * This is the drop-in boundary for the one hot path of luzbetak/rag-faiss-embedding: everything its
 * Python delegates to faiss-cpu's IndexFlatL2 / IndexFlatIP through the SWIG module `faiss`.
 * Each entry point names the reference call site(s) it replaces (paths relative to the reference
 * repository root).  Plain pointers and sizes only; no C++ or torch types cross this line.
 *
 * Conventions
 *   - every function returns 0 on success or a negative B2F_E* code; b2f_last_error() returns the
 *     thread-local message of the last failure.  Nothing throws or aborts across the ABI.
 *   - `mem` says where the caller's buffers live: B2F_MEM_HOST (numpy) or B2F_MEM_DEVICE (a CUDA
 *     pointer on the index's device, e.g. torch.Tensor.data_ptr()).
 *   - `stream` is a cudaStream_t passed as void*; NULL = the index's own (non-blocking) stream; pass
 *     cudaStreamLegacy (0x1) to mean the legacy default stream.  With host buffers
 *     every call is synchronous on return (faiss semantics).  With device buffers the work is
 *     enqueued on `stream` and the call returns without synchronising: nothing inside a search waits
 *     for the GPU (uncertified queries are re-run by a kernel that reads their count on the device),
 *     so back-to-back searches keep the GPU busy.  b2f_index_stats() settles all pending work.
 *   - the caller allocates D / I (as faiss's search_c does); the library owns all device storage
 *     behind the handle.
 *   - there is NO CPU fallback: every compute entry point fails with B2F_ENOGPU when no sm_100 device
 *     is usable.
 */
#ifndef B200FLAT_H
#define B200FLAT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2F_VERSION 1

#if defined(__GNUC__)
#define B2F_API __attribute__((visibility("default")))
#else
#define B2F_API
#endif

/* faiss MetricType values (faiss.METRIC_INNER_PRODUCT = 0, faiss.METRIC_L2 = 1) */
#define B2F_METRIC_INNER_PRODUCT 0
#define B2F_METRIC_L2 1

/* what the index keeps as its authoritative rows */
#define B2F_STORE_F32 0  /* fp32 rows (faiss IndexFlat layout) + derived bf16 scan copy */
#define B2F_STORE_BF16 1 /* rows rounded to bf16 at add(); fp32 arithmetic on the rounded values */

#define B2F_MEM_HOST 0
#define B2F_MEM_DEVICE 1

/* search algorithm selector (b2f_search_params.algo) */
#define B2F_ALGO_AUTO 0   /* nq <= scan_max_nq -> streaming scan, else tensor path */
#define B2F_ALGO_SCAN 1   /* K1: fp32 exact-difference streaming scan on CUDA cores (any nq, in groups) */
#define B2F_ALGO_TENSOR 2 /* K2: tcgen05/TMEM bf16 contraction + fused top-k, then exact fp32 re-rank (shapes it cannot
                             plan -- k' > 256, a few-row database -- are served by the scan; b2f_stats.last_algo tells) */

/* pooling modes of the fused encoder epilogue */
#define B2F_POOL_CLS 0  /* last_hidden_state[:, 0]  (the reference: vectorization.py:44) */
#define B2F_POOL_MEAN 1 /* attention-mask weighted mean over tokens */

/* error codes */
#define B2F_OK 0
#define B2F_EINVAL -1   /* bad argument (faiss: AssertionError, e.g. d mismatch, k <= 0) */
#define B2F_ENOGPU -2   /* no usable sm_100 device / CUDA runtime failure at init */
#define B2F_ECUDA -3    /* a CUDA call or kernel failed */
#define B2F_EIO -4      /* file could not be read / written */
#define B2F_EFORMAT -5  /* not an IndexFlat file */
#define B2F_ENOMEM -6   /* device or host allocation failed */
#define B2F_ERANGE -7   /* row index out of range */

typedef struct b2f_index b2f_index;

typedef struct b2f_search_params {
    int32_t algo;          /* B2F_ALGO_* */
    int32_t scan_max_nq;   /* AUTO: largest nq served by the streaming scan (0 = default: 1, the reference's nq,
                              for fp32 storage; none for bf16 storage, where the tensor path is always faster) */
    int32_t slack;         /* tensor path: extra coarse candidates per query kept for the exact re-rank
                              (0 = default: k' = k + max(22, ceil(0.9 k)), rounded up to 32 / 64 / a multiple of 8, <= 256) */
    int32_t certify;       /* tensor path: 1 (default when 0 is passed via NULL params) = prove from the
                              bf16 rounding bound that no non-candidate can beat the k-th re-ranked
                              result; queries that fail are answered exactly another way: by the range pass (one more
                              tensor pass with a fixed threshold per query) once an index has seen more than 0.1 % of
                              a batch fail, else by the exact scan.  The index also adapts to what its data does to the
                              candidate lists: +32 candidates per query after batches with > 0.5 % exact scans,
                              per-thread heaps instead of shared-threshold lists after mass list overflows.
                              All of it changes speed only -- results are exact either way.  -1 = certification off */
    int64_t id_offset;     /* added to every returned label (row-sharded indexes: the shard's first row) */
    int32_t profile;       /* 1 = record CUDA events around the dominant kernel (see b2f_stats) */
    int32_t reserved;
} b2f_search_params;

typedef struct b2f_stats {
    int64_t launches;          /* kernels launched by the library on behalf of this index so far */
    int64_t searches;          /* search calls so far */
    int64_t fallback_queries;  /* queries re-run through the exact scan after failing certification */
    int32_t last_algo;         /* B2F_ALGO_SCAN / B2F_ALGO_TENSOR actually used by the last search */
    int32_t last_kprime;       /* candidates per query kept by the last tensor-path search */
    float last_main_ms;        /* CUDA-event time of the dominant kernel of the last search (profile=1) */
    float last_total_ms;       /* CUDA-event time of the whole device pipeline of the last search */
    int32_t last_main_launches;/* how many launches last_main_ms covers */
    int32_t last_launches;     /* kernels launched by the last search */
    int64_t bytes_rows;        /* device bytes held: authoritative rows */
    int64_t bytes_scan;        /* device bytes held: bf16 scan copy + norms */
    int64_t overflow_queries;  /* subset of fallback_queries caused by a candidate-list overflow */
    int64_t last_list_entries; /* rows that survived the fused threshold filter in the last tensor-path search */
    double prof_main_ms_sum;   /* profile=1: running sums over searches, so a benchmark reads them once */
    double prof_total_ms_sum;
    int64_t prof_main_launches;
    int64_t prof_searches;
    int64_t rescued_queries;   /* tensor path: queries certified only after re-ranking every list entry (no database pass) */
    int64_t range_queries;     /* tensor path: uncertified queries served by the range pass (a second tensor pass with a fixed
                                  threshold per query) instead of the exact scan */
} b2f_stats;

/* ---- lifecycle -------------------------------------------------------------------------------
 * faiss.IndexFlatL2(d) / IndexFlatIP(d) / IndexFlat(d, metric):
 *   faiss_store.py:29, faiss_store.py:126, rag_datastore_manager.py:138                          */
B2F_API int b2f_index_create(int32_t d, int32_t metric, int32_t storage, int32_t device, b2f_index** out);
B2F_API int b2f_index_destroy(b2f_index* idx);
/* index.reset(): faiss_store.py:124-128 re-creates the index; same effect */
B2F_API int b2f_index_reset(b2f_index* idx);
/* capacity hint so that large ingests do not re-allocate (no reference counterpart) */
B2F_API int b2f_index_reserve(b2f_index* idx, int64_t nrows);

/* ---- attributes: index.ntotal (faiss_store.py:53,115), index.d, index.metric_type ------------- */
B2F_API int64_t b2f_index_ntotal(const b2f_index* idx);
B2F_API int32_t b2f_index_d(const b2f_index* idx);
B2F_API int32_t b2f_index_metric(const b2f_index* idx);
B2F_API int32_t b2f_index_storage(const b2f_index* idx);
B2F_API int32_t b2f_index_device(const b2f_index* idx);

/* ---- index.add(x): faiss_store.py:46, rag_datastore_manager.py:173 ----------------------------
 * x: [n, d] fp32 row-major contiguous.  Appends; labels are implicit row numbers.               */
B2F_API int b2f_index_add(b2f_index* idx, int64_t n, const float* x, int32_t mem, void* stream);

/* ---- index.search(q, k): faiss_store.py:64, rag_datastore_manager.py:218 (THE hot call) -------
 * q: [nq, d] fp32; D: [nq, k] fp32; I: [nq, k] int64.
 * L2: k smallest SQUARED distances ascending; IP: k largest inner products descending;
 * fewer than k rows -> label -1 and distance +FLT_MAX (L2) / -FLT_MAX (IP).
 * params may be NULL (all defaults).                                                             */
B2F_API int b2f_index_search(b2f_index* idx, int64_t nq, const float* q, int64_t k, float* D, int64_t* I,
                     int32_t mem, void* stream, const b2f_search_params* params);

/* ---- index.range_search(q, radius): every row closer than a radius (faiss IndexFlat range search) ----------------
 * L2: radius is on SQUARED distances, a row is a hit when dist < radius (strict); an L2 radius <= 0 returns nothing.
 * IP: a row is a hit when ip > radius (strict).  NaN distances are never hits; a NaN radius is B2F_EINVAL.
 * Distances are the engine's exact fp32 values -- L2 in the exact-difference form, IP the fp32 dot product, both to the
 * authoritative rows (bf16 storage: fl32(mu + x~')) -- computed by the same code on every path, so a row's membership
 * and its distance bits do not depend on the path that served the query, the batch size or the chunking.
 * Within a query the hits are in ascending label order (label = row + params->id_offset).
 * Layout of faiss's RangeSearchResult: lims [nq + 1] with lims[0] = 0, D [lims[nq]] fp32, I [lims[nq]] int64; query i
 * owns [lims[i], lims[i+1]).
 * params: algo AUTO / TENSOR use the tensor pass with a fixed per-query threshold wherever it can be planned (nq = 1
 * included), SCAN forces the exact range scan; scan_max_nq > 0 sends AUTO batches of at most that many queries to the
 * exact range scan (default: none); id_offset is added to every label; slack, certify and profile are ignored.
 * A range search changes nothing top-k searches learn or report (b2f_stats: only `launches` grows).
 * The result size is known only after the GPU has counted, so the library owns the result behind a handle. */
typedef struct b2f_range_result b2f_range_result;
/* index.range_search(x, radius): q [nq, d] fp32 in `mem`.  Returns once lims are known (host sync(s) inside); the
 * hits may still be in flight on `stream`.  A result too large for device memory is B2F_ENOMEM. */
B2F_API int b2f_index_range_search(b2f_index* idx, int64_t nq, const float* q, float radius, int32_t mem, void* stream,
                                   const b2f_search_params* params, b2f_range_result** out);
B2F_API int b2f_range_result_lims(const b2f_range_result* r, int64_t* lims /* host, nq + 1 */);
/* D [lims[nq]] fp32, I [lims[nq]] int64 in `mem`; device: enqueued on `stream`, host: synchronous */
B2F_API int b2f_range_result_fetch(b2f_range_result* r, float* D, int64_t* I, int32_t mem, void* stream);
/* out[0] hits, [1] queries answered from tensor-pass lists, [2] queries answered by the exact range scan,
 * [3] kernels launched, [4] host synchronisations */
B2F_API int b2f_range_result_info(const b2f_range_result* r, int64_t out[5]);
/* waits for the result's pending copies, then frees it */
B2F_API int b2f_range_result_destroy(b2f_range_result* r);

/* ---- index.remove_ids(sel): faiss IndexFlat::remove_ids (no reference call site) ---------------------------------
 * Removes the named rows; the survivors keep their order and are renumbered 0 .. ntotal' - 1 (labels above a removed
 * row shift down).  *nremoved (may be NULL) = rows removed.  Ids outside [0, ntotal) and duplicates are ignored; removing
 * nothing launches nothing.  Every surviving row keeps its stored bits (fp32 rows; bf16 storage: fl32(mu + x~'), its
 * scan copy and bias too), and the centre mu stays until reset -- removing every row is not a reset.  The certification
 * bound is taken again over the survivors, so removing a non-finite row gives the tensor path back.  Synchronous on
 * return; searches still in flight on any stream finish first.  The device work is an in-place compaction of the rows
 * above the first removed one: each moved byte read once and written once, no second copy of the rows.             */
/* ids: host int64 [n], any order */
B2F_API int b2f_index_remove_ids(b2f_index* idx, int64_t n, const int64_t* ids, int64_t* nremoved);
/* IDSelectorRange(imin, imax): rows imin <= i < imax */
B2F_API int b2f_index_remove_range(b2f_index* idx, int64_t imin, int64_t imax, int64_t* nremoved);

/* ---- index.reconstruct(i) / reconstruct_n(i0, n) (SURVEY 8b shim surface) ---------------------- */
B2F_API int b2f_index_reconstruct(b2f_index* idx, int64_t i0, int64_t n, float* out, int32_t mem, void* stream);

/* ---- faiss.write_index(index, path): faiss_store.py:91, rag_datastore_manager.py:186 ----------
 * ---- faiss.read_index(path):         faiss_store.py:106, rag_datastore_manager.py:205 ----------
 * Byte-compatible with FAISS's IndexFlat serialisation ("IxF2"/"IxFI" | i32 d | i64 ntotal |
 * i64 2^20 | i64 2^20 | u8 is_trained | i32 metric | u64 nfloats | fp32 rows).  Streams through
 * pinned chunks, so a 100+ GB index never needs a host copy.  Reading into B2F_STORE_BF16
 * re-ingests the file's fp32 rows as a first add would: a new centre from the file's first rows,
 * each row rounded around it.                                                                    */
B2F_API int b2f_index_write(b2f_index* idx, const char* path);
B2F_API int b2f_index_read(const char* path, int32_t storage, int32_t device, b2f_index** out);

/* ---- multi-GPU: merge per-shard top-k lists after the all-gather (SURVEY 8e) -------------------
 * D_parts/I_parts: [nparts, nq, k] (the all_gather_into_tensor layout); out: [nq, k].
 * Keeps faiss ordering and -1 padding.  Device buffers only.  1 <= nparts <= 32 (else B2F_EINVAL). */
B2F_API int b2f_merge_topk(int32_t metric, int64_t nq, int64_t k, int32_t nparts, const float* D_parts,
                   const int64_t* I_parts, float* D, int64_t* I, int32_t device, void* stream);
/* Same merge over parts that are `part_stride_bytes` apart (D_parts / I_parts point at part 0): lets each rank
 * ship its distances and labels in ONE packed all-gather message instead of two.                      */
B2F_API int b2f_merge_topk_strided(int32_t metric, int64_t nq, int64_t k, int32_t nparts, const float* D_parts,
                   const int64_t* I_parts, int64_t part_stride_bytes, float* D, int64_t* I, int32_t device,
                   void* stream);
/* Merge nparts per-shard range-search results into one, query by query, hits in ascending label order.
 * lims_parts: device int64 [nparts][nq + 1], part p's own lims (any base: part p's hits of query q are its
 * elements lims_parts[p][q] - lims_parts[p][0] .. lims_parts[p][q+1] - lims_parts[p][0]);
 * part p's D (fp32) at D_parts + p * part_stride_bytes, its I (int64) at I_parts + p * part_stride_bytes
 * (the packed all-gather layout [D | pad | I], as b2f_merge_topk_strided).
 * Within a part and a query the labels must be strictly ascending; different parts hold disjoint labels.
 * Output: D [total], I [total], total = sum over p of the parts' hit counts, query q at offset
 * sum_p (lims_parts[p][q] - lims_parts[p][0]).  Distances are copied bit for bit.  1 <= nparts <= 32.
 * Device buffers only; enqueued on `stream` without a host synchronisation (the hit count is read on the device), so
 * with nq > 0 the hit pointers must not be NULL even when every part is empty.  part_stride_bytes: a multiple of 16. */
B2F_API int b2f_merge_range_strided(int64_t nq, int32_t nparts, const int64_t* lims_parts, const float* D_parts,
                                    const int64_t* I_parts, int64_t part_stride_bytes, float* D, int64_t* I,
                                    int32_t device, void* stream);

/* ---- multi-GPU over NVLink peer memory: the exchange + merge above as ONE kernel (no NCCL call, no second launch).
 * One process per GPU.  create() allocates this rank's receive buffers (two generations x world slots of
 * slot_bytes) and returns a 64-byte IPC handle; the host exchanges the handles of all ranks (any side channel,
 * e.g. torch.distributed.all_gather_object) and passes them, rank-ordered, to connect().  merge() is collective:
 * every rank calls it once per search with its own message `msg` = [D (nq*k fp32) | pad | I (nq*k int64) at off_i],
 * msg_bytes a multiple of 16 and <= slot_bytes.  The kernel pushes the message into every peer's slot with
 * 16-byte stores, signals with a system-scope release flag, waits for all ranks' flags and merges the world
 * parts into (D, I) [nq, k] on `stream`.  Device buffers only.                                          */
typedef struct b2f_exchange b2f_exchange;
B2F_API int b2f_exchange_create(int32_t device, int32_t rank, int32_t world, int64_t slot_bytes, b2f_exchange** out,
                        void* handle_out_64_bytes);
B2F_API int b2f_exchange_connect(b2f_exchange* ex, const void* handles_world_x_64_bytes);
B2F_API int64_t b2f_exchange_slot_bytes(const b2f_exchange* ex);
B2F_API int b2f_exchange_merge(b2f_exchange* ex, const void* msg, int64_t msg_bytes, int32_t metric, int64_t nq, int64_t k,
                       int64_t off_i, float* D, int64_t* I, void* stream);
/* The whole sharded step (SURVEY 8e) behind ONE call: search this rank's shard (labels + params->id_offset) straight into
 * the exchange's own message buffer, then the push + flag + merge kernel above, all enqueued on `stream` -- no host
 * allocation, no second library call.  Collective: every rank calls it once per search with the same nq / k.
 * q: [nq, d] fp32, D: [nq, k] fp32, I: [nq, k] int64, device buffers.                                     */
B2F_API int b2f_exchange_search(b2f_exchange* ex, b2f_index* idx, int64_t nq, const float* q, int64_t k, float* D,
                        int64_t* I, void* stream, const b2f_search_params* params);
B2F_API int b2f_exchange_destroy(b2f_exchange* ex);

/* ---- fused encoder epilogue (replaces vectorization.py:44-47, rag_datastore_manager.py:129-132:
 *      last_hidden_state[:,0].cpu().numpy() -> list -> np.array) ---------------------------------
 * hidden: [B, T, d] fp32 device; mask: [B, T] int64 device (HF attention_mask) or NULL.
 * pool = B2F_POOL_CLS reproduces the reference; normalize != 0 divides by the L2 norm.
 * b2f_pool_normalize writes [B, d] to `out` (device); b2f_index_add_pooled appends straight into
 * the index storage (rows, bf16 scan copy and norms in the same kernel, no host bounce).          */
B2F_API int b2f_pool_normalize(const float* hidden, const int64_t* mask, int64_t B, int64_t T, int32_t d,
                       int32_t pool, int32_t normalize, float* out, int32_t device, void* stream);
B2F_API int b2f_index_add_pooled(b2f_index* idx, const float* hidden, const int64_t* mask, int64_t B, int64_t T,
                         int32_t pool, int32_t normalize, void* stream);

/* Query side of the same hand-off (replaces the encode -> .cpu().numpy() -> np.array -> index.search chain of
 * vectorization.py:38-47 + faiss_store.py:56-64): pools (+ normalises) the encoder output of a query batch on the
 * device and searches it, all on `stream`; D: [B, k] fp32, I: [B, k] int64, device buffers.              */
B2F_API int b2f_index_search_pooled(b2f_index* idx, const float* hidden, const int64_t* mask, int64_t B, int64_t T,
                            int32_t pool, int32_t normalize, int64_t k, float* D, int64_t* I, void* stream,
                            const b2f_search_params* params);

/* ---- synthetic rows for benchmarks: same bits as oracle/flat_oracle.c orc_synth_rows ----------- */
B2F_API int b2f_synth_rows(uint64_t seed, int64_t row0, int64_t nrows, int32_t d, int32_t normalize, float* out,
                   int32_t device, void* stream);
/* append synthetic rows generated on the device (no host staging; for 10^7..10^8-row configs) */
B2F_API int b2f_index_add_synth(b2f_index* idx, uint64_t seed, int64_t row0, int64_t nrows, int32_t normalize);

/* ---- diagnostics ------------------------------------------------------------------------------ */
/* How the tensor path would run a search of nq queries, k neighbours, on n rows of dimension d (pure host logic,
 * no GPU needed): out[0] = k' (0: tensor path unavailable), out[1] = queries per pass, out[2] = passes,
 * out[3] = 1 LIST / 0 HEAP selection, out[4] = 1 when CTA pairs are used, out[5] = units (CTAs or pairs) per pass,
 * out[6] = whole units per query tile unit (LIST: every unit gets tile units / units of a pass, balanced),
 * out[7] = candidate lists allocated per query, out[8] = j (rows each voucher list vouches for), out[9] = entries
 * per list, out[10] = 128-query tiles per pass, out[11] = database tiles per round of the interleaved sweep.   */
B2F_API int b2f_plan_describe(int64_t nq, int64_t n, int32_t d, int64_t k, int32_t slack, int32_t out[12]);
/* The work of unit `unit` (of `units`) under the balanced split of `tile_units` query tile units x `db_tiles` database
 * tiles with k' = kprime, as the kernel computes it: returns the number of segments (1 or 2), in the order the unit runs
 * them; seg_info[7 s ..] = query tile unit, list slot, voucher slots of that tile, in-tile range [p0, p1) in 1/units,
 * rows each list of the piece vouches for, voucher lists a thread consults; counts[s] = database tiles of segment s, the
 * first `cap` of which are written to tiles[s * cap ..] (tiles may be NULL).  Host logic only (tests).          */
B2F_API int b2f_plan_unit_work(int32_t tile_units, int32_t units, int32_t round_tiles, int64_t db_tiles, int32_t kprime,
                       int32_t unit, int32_t seg_info[14], int64_t* tiles, int64_t cap, int32_t counts[2]);
/* How b2f_index_remove_ids plans a removal of ids [n] from ntotal rows (host logic only, no GPU): the sorted disjoint
 * runs it removes, runs[2 j] <= row < runs[2 j + 1] (*nruns of them; runs: room for 2 n, or NULL); the new row of every
 * row, dest[ntotal] (-1: removed; or NULL); and the compaction tiles for rows of row_bytes bytes (*ntiles of them, the
 * first cap written to tiles[3 t ..]: first source row, then [first, last + 1) of the tiles it waits for).           */
B2F_API int b2f_remove_plan(int64_t ntotal, int64_t n, const int64_t* ids, int64_t row_bytes, int64_t* runs, int64_t* nruns,
                            int64_t* dest, int64_t* tiles, int64_t cap, int64_t* ntiles);
B2F_API int b2f_index_stats(const b2f_index* idx, b2f_stats* out);
B2F_API const char* b2f_last_error(void);
B2F_API int b2f_version(void);
/* number of usable sm_100 devices (0 on a CPU-only box; never fails) */
B2F_API int b2f_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* B200FLAT_H */
