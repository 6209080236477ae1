// exchange.cu -- K6': the multi-GPU exchange of SURVEY 8(e) as ONE kernel over NVLink peer memory.
//
// After the per-shard search every rank holds one message [D | I] (12 * nq * k bytes).  Instead of an NCCL
// all-gather followed by a merge launch, one kernel per rank
//   1. pushes its message into slot [rank] of every peer's receive buffer with 16-byte stores through the
//      peer mappings (cudaIpc; NVLink / NVSwitch),
//   2. the last CTA to finish pushing publishes this search's sequence number into every peer's flag word
//      (system-scope release),
//   3. every CTA waits until the flags of all PEER ranks show the sequence number (acquire), and
//   4. merges its share of the queries (one warp per query, faiss ordering, -1 padding) into the caller's
//      (D, I): the peers' parts straight out of the receive buffer, its own part straight out of its message.
// Receive buffers and flags are double buffered by the parity of the sequence number: a rank can only start
// search s + 2 after it merged s + 1, which needed every peer's push of s + 1, which those peers issued after
// their merge of s -- so no slot is overwritten while a slower peer still reads it.  Nothing here depends on
// co-residency of this rank's own grid: pushes never wait, a CTA waits for PEER flags only (its own part is
// local), so a co-running kernel that keeps some of this grid's CTAs off the SMs cannot stall the ones that run.
//
// b2f_exchange_search() is the whole sharded step behind one C call: the local search writes (D, I) straight into
// the exchange's own message buffer, then the kernel above runs on the same stream -- no allocation, no second
// library call on the host.
#include <string.h>

#include <new>
#include <vector>

#include "common.cuh"

using namespace b2f;

struct b2f_exchange {
    int device = 0, rank = 0, world = 1;
    int64_t slot_bytes = 0;            // capacity of one message
    char* local = nullptr;             // [2][world][slot_bytes] receive buffers, then flags [2][world] u32, then the push counter
    size_t local_bytes = 0;
    std::vector<char*> peer;           // peer[r] = base of rank r's allocation as mapped here (peer[rank] = local)
    char** peer_dev = nullptr;         // device copy of the table
    uint32_t seq = 0;
    bool connected = false;
    char* msg = nullptr;               // [2][slot_bytes] this rank's outgoing messages (b2f_exchange_search), by sequence parity
};

namespace {

struct ExArgs {
    char* const* peer;       // [world] bases
    int rank, world;
    int64_t slot_bytes, msg_bytes;
    int64_t flags_off, ctr_off;
    uint32_t seq;
    const char* src;         // this rank's message
    int l2;
    int64_t nq;
    int k;
    int64_t off_i;           // byte offset of the labels inside a message
    float* D;
    int64_t* I;
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(256) exchange_merge_kernel(const ExArgs a) {
    const int par = (int)(a.seq & 1u);
    const int64_t buf_off = (int64_t)par * a.world * a.slot_bytes;
    // ---- 1. push: my message into slot [rank] of every PEER's receive buffer -------------------------------
    {
        const int64_t nvec = a.msg_bytes >> 4;   // messages are padded to 16 bytes
        const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
        const uint4* s = reinterpret_cast<const uint4*>(a.src);
        for (int64_t i = tid; i < nvec; i += nth) {
            const uint4 v = s[i];
            for (int r = 1; r < a.world; r++) {              // peers only: this rank merges its own part from `src`
                const int dst = (a.rank + r) % a.world;   // spread the NVLink traffic: every rank starts at a different peer
                reinterpret_cast<uint4*>(a.peer[dst] + buf_off + (int64_t)a.rank * a.slot_bytes)[i] = v;
            }
        }
    }
    // ---- 2. the last CTA to finish pushing signals every peer ---------------------------------------------
    __shared__ int s_last;
    __threadfence_system();
    __syncthreads();
    uint32_t* ctr = reinterpret_cast<uint32_t*>(a.peer[a.rank] + a.ctr_off);
    if (threadIdx.x == 0) {
        const uint32_t prev = atomicAdd(ctr, 1u);
        s_last = prev == gridDim.x - 1;
        if (s_last) *ctr = 0u;   // self-cleaning for the next call (stream ordered)
    }
    __syncthreads();
    if (s_last && threadIdx.x < a.world && (int)threadIdx.x != a.rank) {
        __threadfence_system();
        uint32_t* f = reinterpret_cast<uint32_t*>(a.peer[threadIdx.x] + a.flags_off) + par * a.world + a.rank;
        st_release_sys(f, a.seq);
    }
    // ---- 3. wait for every PEER's push of this search (never for this rank's own grid) ------------------------
    if (threadIdx.x < a.world && (int)threadIdx.x != a.rank) {
        const uint32_t* f = reinterpret_cast<const uint32_t*>(a.peer[a.rank] + a.flags_off) + par * a.world + threadIdx.x;
        // bounded: a peer that died must surface as a CUDA error at the next synchronisation, not as a hung GPU
        const long long t0 = clock64();
        while (ld_acquire_sys(f) != a.seq) {
            __nanosleep(64);
            if (clock64() - t0 > 120000000000LL) __trap();   // ~60 s at 2 GHz
        }
    }
    __syncthreads();
    // ---- 4. merge: one warp per query over the world parts (lane l walks part l) ----------------------------
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    const char* base = a.peer[a.rank] + buf_off;
    for (int64_t q = (int64_t)blockIdx.x * wpb + (threadIdx.x >> 5); q < a.nq; q += (int64_t)gridDim.x * wpb) {
        const bool have = lane < a.world;
        const char* part = (have && lane != a.rank) ? base + (int64_t)lane * a.slot_bytes : a.src;   // own part: the message itself
        warp_merge_faiss<true>(a.l2, have, reinterpret_cast<const float*>(part) + q * a.k,
                         reinterpret_cast<const int64_t*>(part + a.off_i) + q * a.k, a.k, a.D + q * a.k, a.I + q * a.k, lane);
    }
}

int64_t flags_offset(const b2f_exchange* ex) { return 2 * (int64_t)ex->world * ex->slot_bytes; }

}  // namespace

extern "C" {

int b2f_exchange_create(int32_t device, int32_t rank, int32_t world, int64_t slot_bytes, b2f_exchange** out, void* handle_out) {
    if (!out || !handle_out || world < 1 || world > 32 || rank < 0 || rank >= world || slot_bytes <= 0) {
        set_error("exchange_create: bad arguments");
        return B2F_EINVAL;
    }
    *out = nullptr;
    if (cudaSetDevice(device) != cudaSuccess) {
        cudaGetLastError();
        set_error("exchange_create: cudaSetDevice(%d) failed", device);
        return B2F_ENOGPU;
    }
    b2f_exchange* ex = new (std::nothrow) b2f_exchange();
    if (!ex) return B2F_ENOMEM;
    ex->device = device;
    ex->rank = rank;
    ex->world = world;
    ex->slot_bytes = (slot_bytes + 255) / 256 * 256;
    ex->local_bytes = (size_t)flags_offset(ex) + 2 * (size_t)world * 4 + 64;
    cudaError_t e = cudaMalloc(&ex->local, ex->local_bytes);
    if (e == cudaSuccess) e = cudaMemset(ex->local, 0, ex->local_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&ex->peer_dev, sizeof(char*) * world);
    if (e == cudaSuccess) e = cudaMalloc(&ex->msg, 2 * (size_t)ex->slot_bytes);
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, ex->local);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("exchange_create: %s", cudaGetErrorString(e));
        cudaFree(ex->local);
        cudaFree(ex->peer_dev);
        cudaFree(ex->msg);
        delete ex;
        return B2F_ECUDA;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(handle_out, &h, 64);
    ex->peer.assign(world, nullptr);
    ex->peer[rank] = ex->local;
    *out = ex;
    return B2F_OK;
}

int b2f_exchange_connect(b2f_exchange* ex, const void* handles) {
    if (!ex || !handles) {
        set_error("exchange_connect: bad arguments");
        return B2F_EINVAL;
    }
    B2F_CUDA(cudaSetDevice(ex->device));
    for (int r = 0; r < ex->world; r++) {
        if (r == ex->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, static_cast<const char*>(handles) + 64 * (size_t)r, 64);
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_error("exchange_connect: cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e));
            return B2F_ECUDA;
        }
        ex->peer[r] = static_cast<char*>(p);
    }
    B2F_CUDA(cudaMemcpy(ex->peer_dev, ex->peer.data(), sizeof(char*) * ex->world, cudaMemcpyHostToDevice));
    ex->connected = true;
    return B2F_OK;
}

int64_t b2f_exchange_slot_bytes(const b2f_exchange* ex) { return ex ? ex->slot_bytes : -1; }

int b2f_exchange_merge(b2f_exchange* ex, const void* msg, int64_t msg_bytes, int32_t metric, int64_t nq, int64_t k, int64_t off_i,
                       float* D, int64_t* I, void* stream) {
    if (!ex || !ex->connected || !msg || !D || !I || nq < 0 || k <= 0 || msg_bytes <= 0 || (msg_bytes & 15) || (off_i & 7) ||
        msg_bytes > ex->slot_bytes || off_i + nq * k * 8 > msg_bytes) {
        set_error("exchange_merge: bad arguments (message %lld bytes, slot %lld)", (long long)msg_bytes, ex ? (long long)ex->slot_bytes : -1LL);
        return B2F_EINVAL;
    }
    B2F_CUDA(cudaSetDevice(ex->device));
    ExArgs a{};
    a.peer = ex->peer_dev;
    a.rank = ex->rank;
    a.world = ex->world;
    a.slot_bytes = ex->slot_bytes;
    a.msg_bytes = msg_bytes;
    a.flags_off = flags_offset(ex);
    a.ctr_off = a.flags_off + 2 * (int64_t)ex->world * 4;
    a.seq = ++ex->seq;
    a.src = static_cast<const char*>(msg);
    a.l2 = metric == B2F_METRIC_L2;
    a.nq = nq;
    a.k = (int)k;
    a.off_i = off_i;
    a.D = D;
    a.I = I;
    const int wpb = 8;
    int64_t blocks = (nq + wpb - 1) / wpb;
    if (blocks > 2 * kNumSMs) blocks = 2 * kNumSMs;
    if (blocks < 1) blocks = 1;
    exchange_merge_kernel<<<(unsigned)blocks, wpb * 32, 0, (cudaStream_t)stream>>>(a);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

int b2f_exchange_search(b2f_exchange* ex, b2f_index* idx, int64_t nq, const float* q, int64_t k, float* D, int64_t* I,
                        void* stream, const b2f_search_params* params) {
    if (!ex || !ex->connected || !idx || nq < 0 || k <= 0 || (nq > 0 && (!q || !D || !I))) {
        set_error("exchange_search: bad arguments");
        return B2F_EINVAL;
    }
    if (nq == 0) return B2F_OK;
    const int64_t off_i = (nq * k * 4 + 15) / 16 * 16;
    const int64_t msg_bytes = (off_i + nq * k * 8 + 15) / 16 * 16;
    if (msg_bytes > ex->slot_bytes) {
        set_error("exchange_search: message of %lld bytes exceeds the slot size %lld (re-create the exchange)", (long long)msg_bytes,
                  (long long)ex->slot_bytes);
        return B2F_EINVAL;
    }
    if (b2f_index_device(idx) != ex->device) {
        set_error("exchange_search: the index lives on device %d, the exchange on device %d", b2f_index_device(idx), ex->device);
        return B2F_EINVAL;
    }
    // the local search writes its faiss-formatted (D, I) straight into the outgoing message (double buffered by the
    // parity of the next sequence number, so a caller that alternates streams cannot overwrite a message in flight)
    char* msg = ex->msg + (size_t)((ex->seq + 1) & 1u) * (size_t)ex->slot_bytes;
    B2F_TRY(b2f_index_search(idx, nq, q, k, reinterpret_cast<float*>(msg), reinterpret_cast<int64_t*>(msg + off_i), B2F_MEM_DEVICE,
                             stream, params));
    return b2f_exchange_merge(ex, msg, msg_bytes, b2f_index_metric(idx), nq, k, off_i, D, I, stream);
}

int b2f_exchange_destroy(b2f_exchange* ex) {
    if (!ex) return B2F_OK;
    cudaSetDevice(ex->device);
    cudaDeviceSynchronize();
    for (int r = 0; r < ex->world; r++)
        if (r != ex->rank && ex->peer[r]) cudaIpcCloseMemHandle(ex->peer[r]);
    cudaFree(ex->local);
    cudaFree(ex->peer_dev);
    cudaFree(ex->msg);
    delete ex;
    return B2F_OK;
}

}  // extern "C"
