// rerank.cuh -- K4 as a block-level device function, shared by the standalone re-rank kernel (HEAP mode)
// and the fused list-merge + re-rank kernel (LIST mode).  See rerank.cu for the bound.
#pragma once
#include "common.cuh"

namespace b2f {

constexpr int kRerankThreads = 256;

// Exact fp32 key (L2: squared distance in exact-difference form; IP: negated dot product) of row `id` for the
// query vector qv, computed by the 8 lanes of a lane group (sl = lane & 7); every lane returns the total.
// The loads of a row are issued four 16-byte chunks at a time, so a lane group keeps 512 bytes in flight.
__device__ __forceinline__ float exact_key_8lanes(const StoredRows& a, const float* __restrict__ qv, int32_t id, int sl, bool l2) {
    float acc = 0.f;
    if (id >= 0) {
        if (a.f32 && (a.d & 3) == 0) {
            const float* x = a.f32 + (int64_t)id * a.d;
            for (int j0 = sl * 4; j0 < a.d; j0 += 128) {
                float4 xv[4], qq[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int j = j0 + 32 * u;
                    xv[u] = j < a.d ? __ldg(reinterpret_cast<const float4*>(x + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int j = j0 + 32 * u;
                    qq[u] = j < a.d ? __ldg(reinterpret_cast<const float4*>(qv + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    if (l2) {
                        const float t0 = xv[u].x - qq[u].x, t1 = xv[u].y - qq[u].y, t2 = xv[u].z - qq[u].z, t3 = xv[u].w - qq[u].w;
                        acc = fmaf(t0, t0, acc); acc = fmaf(t1, t1, acc); acc = fmaf(t2, t2, acc); acc = fmaf(t3, t3, acc);
                    } else {
                        acc = fmaf(xv[u].x, qq[u].x, acc); acc = fmaf(xv[u].y, qq[u].y, acc);
                        acc = fmaf(xv[u].z, qq[u].z, acc); acc = fmaf(xv[u].w, qq[u].w, acc);
                    }
                }
            }
        } else if (!a.f32 && (a.d & 7) == 0) {
            const __nv_bfloat16* x = a.bf16 + (int64_t)id * a.pitch;
            for (int j0 = sl * 8; j0 < a.d; j0 += 128) {
                uint4 w[2];
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const int j = j0 + 64 * u;
                    w[u] = j < a.d ? __ldg(reinterpret_cast<const uint4*>(x + j)) : make_uint4(0u, 0u, 0u, 0u);
                }
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const int j = j0 + 64 * u;
                    if (j < a.d) {
                        const uint32_t ww[4] = {w[u].x, w[u].y, w[u].z, w[u].w};
                        const float4 qa = __ldg(reinterpret_cast<const float4*>(qv + j));
                        const float4 qb = __ldg(reinterpret_cast<const float4*>(qv + j + 4));
                        const float qq[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
                        float mm[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                        if (a.centre) {   // the authoritative row: fl32(centre + stored bf16 value)
                            const float4 ma = __ldg(reinterpret_cast<const float4*>(a.centre + j));
                            const float4 mb = __ldg(reinterpret_cast<const float4*>(a.centre + j + 4));
                            mm[0] = ma.x; mm[1] = ma.y; mm[2] = ma.z; mm[3] = ma.w; mm[4] = mb.x; mm[5] = mb.y; mm[6] = mb.z; mm[7] = mb.w;
                        }
#pragma unroll
                        for (int h = 0; h < 4; h++) {
                            const float x0 = mm[2 * h] + __uint_as_float(ww[h] << 16), x1 = mm[2 * h + 1] + __uint_as_float(ww[h] & 0xffff0000u);
                            if (l2) {
                                const float t0 = x0 - qq[2 * h], t1 = x1 - qq[2 * h + 1];
                                acc = fmaf(t0, t0, acc); acc = fmaf(t1, t1, acc);
                            } else {
                                acc = fmaf(x0, qq[2 * h], acc); acc = fmaf(x1, qq[2 * h + 1], acc);
                            }
                        }
                    }
                }
            }
        } else {
            for (int j = sl; j < a.d; j += 8) {
                const float xv = a.f32 ? a.f32[(int64_t)id * a.d + j]
                                       : (a.centre ? a.centre[j] : 0.f) + __bfloat162float(a.bf16[(int64_t)id * a.pitch + j]);
                if (l2) {
                    const float t = xv - qv[j];
                    acc = fmaf(t, t, acc);
                } else {
                    acc = fmaf(xv, qv[j], acc);
                }
            }
        }
    }
    acc += __shfl_xor_sync(kFull, acc, 4);
    acc += __shfl_xor_sync(kFull, acc, 2);
    acc += __shfl_xor_sync(kFull, acc, 1);
    return l2 ? acc : -acc;
}

// The certification test.  tau: exact k-th best key among the re-ranked candidates (FLT_MAX when fewer than k are
// valid); bound: a coarse key that every row OUTSIDE the candidates is known to reach or exceed.  True when the bf16 /
// fp32 rounding bounds prove that no such row can beat tau.
__device__ __forceinline__ bool rerank_certified(const RerankArgs& a, int q, float tau, float bound) {
    const bool l2 = a.rows.metric == B2F_METRIC_L2;
    const float qn2 = a.qnorm[q];
    const float qn = sqrtf(qn2);
    const float eq = a.qerr[q];
    // fp32 accumulation slack: gamma_n * sum|q_i x_i| <= n u |q||x| per inner product (n = d + 16 guards
    // the tensor core's chunked accumulation order, u = 2^-24), doubled for non-IEEE accumulator rounding
    const float gam = 4.f * (float)(a.rows.d + 16) * 5.9604645e-8f;
    if (l2) {
        // c = |q~|^2 + |x~|^2 - 2<q~,x~>: the two norms are fp32 sums as well
        const float nu = gam * (2.f * qn * a.max_row_norm + qn2 + a.max_row_norm * a.max_row_norm);
        const float c = bound + qn2 - nu;
        const float L = sqrtf(fmaxf(c, 0.f)) - eq - a.max_row_err;
        return L > 0.f && L * L * (1.f - 4e-7f) > tau;
    }
    // keys are negated (centred inner product + mu.x): <q,x> = -key + qconst + rounding terms, so
    // non-candidates have <q,x> <= -bound + qconst + slack.  The fp32 sums mu.x and q.mu carry their own
    // rounding error.
    const float cq = a.qconst ? a.qconst[q] : 0.f;
    // mu.x and q.mu are accumulated in double, so they only carry the rounding of their fp32 results and
    // of the fp32 additions they enter (a few ulp of |mu| (|x| + |q|))
    const float xmax = a.max_row_norm + a.max_row_err + a.mu_norm;   // >= |x| of any row
    const float nu = gam * qn * a.max_row_norm + 2.4e-7f * (a.mu_norm * (xmax + qn + eq + a.mu_norm) + qn * a.max_row_norm);
    const float U = -bound + cq + nu + (qn + eq) * a.max_row_err + a.max_row_norm * eq;
    return U < -tau;
}

// ck/ci: the query's candidates (shared or global memory); nc of them are re-ranked.
// bound: a coarse key that every row OUTSIDE the nc candidates is known to reach or exceed.
// all_rows: the candidates are every row of the index (nothing to certify against).
// ek/ei: nc floats / ints of shared scratch.  All kRerankThreads threads of the block must call.
// Writes the best k (exact) to the outputs and returns whether the result is certified exact
// (block-uniform).  Nothing is recorded about a failure here: the caller decides (it may retry with
// more candidates first).
__device__ __forceinline__ bool rerank_block(const RerankArgs& a, int q, const float* ck, const int32_t* ci, int nc, float bound,
                                             bool all_rows, float* ek, int32_t* ei, float* tau_out = nullptr) {
    __shared__ float s_tau;
    __shared__ int s_cert;
    const int lane = threadIdx.x & 31;
    const float* qv = a.q + (int64_t)q * a.rows.d;
    const bool l2 = a.rows.metric == B2F_METRIC_L2;
    const int64_t orow = a.out_map ? (int64_t)a.out_map[q] : (int64_t)q;   // row of D / I this query answers
    if (threadIdx.x == 0) s_tau = FLT_MAX;
    __syncthreads();
    // 8 lanes per candidate, 32 candidates per pass of the block
    const int sl = lane & 7;
    for (int c0 = 0; c0 < nc; c0 += kRerankThreads / 8) {
        const int c = c0 + (threadIdx.x >> 3);
        int32_t id = c < nc ? ci[c] : -1;
        if ((int64_t)id >= a.rows.n) id = -1;  // never dereference a label outside the index
        const float key = exact_key_8lanes(a.rows, qv, id, sl, l2);
        if (sl == 0 && c < nc) {
            const bool ok = id >= 0 && !(key != key);  // NaN never enters (faiss heap semantics)
            ek[c] = ok ? key : FLT_MAX;
            ei[c] = ok ? id : -1;
        }
    }
    __syncthreads();
    // rank sort by (key, id, slot); ranks are a permutation of [0, nc); only the first k ranks are emitted
    for (int t = threadIdx.x; t < nc; t += kRerankThreads) {
        const float mk = ek[t];
        const int32_t mi = ei[t];
        int rank = 0;
        for (int j = 0; j < nc; j++) {
            const float ok_ = ek[j];
            const int32_t oi_ = ei[j];
            rank += (cand_less(ok_, oi_, mk, mi) || (ok_ == mk && oi_ == mi && j < t)) ? 1 : 0;
        }
        if (rank < a.k) {   // faiss conventions straight to the caller's buffers
            const int64_t o = orow * a.k + rank;
            a.D[o] = mi < 0 ? (l2 ? FLT_MAX : -FLT_MAX) : (l2 ? mk : -mk);
            a.I[o] = mi < 0 ? -1 : (int64_t)mi + a.id_offset;
        }
        if (rank == a.k - 1) s_tau = mk;
    }
    // fewer candidates than k: pad (faiss: label -1, distance +-FLT_MAX)
    for (int t = nc + threadIdx.x; t < a.k; t += kRerankThreads) {
        a.D[orow * a.k + t] = l2 ? FLT_MAX : -FLT_MAX;
        a.I[orow * a.k + t] = -1;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const bool certified = all_rows || rerank_certified(a, q, s_tau, bound);  // all_rows: every row of the index is already a candidate
        s_cert = certified ? 1 : 0;
        if (tau_out) *tau_out = s_tau;
    }
    __syncthreads();
    return s_cert != 0;
}

// Records an uncertified query for the exact scan that closes the search.
// tau: the exact k-th key of the candidates that WERE re-ranked (an upper bound of the true k-th key), FLT_MAX when
// nothing usable was found (list overflow, fewer than k valid candidates).
__device__ __forceinline__ void rerank_record_failure(const RerankArgs& a, int q, bool overflowed, float tau = FLT_MAX) {
    const int slot = atomicAdd(a.fail_count, 1);
    a.fail_list[slot] = a.out_map ? a.out_map[q] : q + a.q_base;
    if (a.fail_tau) a.fail_tau[slot] = tau;
    if (overflowed) atomicAdd(a.fail_count + 1, 1);
}

}  // namespace b2f
