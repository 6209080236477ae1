// ingest.cu -- K5 (add: fp32 rows -> authoritative rows + bf16 scan copy + norms, one pass),
// K7 (fused encoder epilogue: CLS / masked-mean pool, optional L2 normalise, written straight into
// index storage), query preparation for the tensor path, and the synthetic-row generator.
// All HBM-bound elementwise / row-reduction work: one warp (or CTA) per row, 16-byte accesses.
#include "remove.cuh"

namespace b2f {

// Non-negative floats order like their bit patterns, so integer atomicMax works.
__device__ __forceinline__ void atomic_max_nonneg(float* addr, float v) {
    atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) v += __shfl_xor_sync(kFull, v, s);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) v += __shfl_xor_sync(kFull, v, s);
    return v;
}

// bf16 storage: the authoritative element r = fl32(m + xb) of a stored (centred, rounded) element xb, and what the fp32
// addition loses, (r - m) - xb.  The ingest and the stats taken again after a removal (scan_stats_kernel) both use it.
__device__ __forceinline__ float auth_loss(float m, float xb, float& r) {
    r = m + xb;
    return (float)((double)r - ((double)m + (double)xb));
}

// Writes one element group of a row to every derived store and returns (bf16(x)^2, (x-bf16(x))^2).
// bf16_auth: the index keeps no fp32 rows -- the authoritative row IS r = fl32(m + bf16(x - m)); then the "rounding
// error" of the scan copy is what the fp32 addition loses, (r - m) - bf16(x - m), and r_out receives r.
__device__ __forceinline__ void emit_elem(float x, int64_t row, int col, int d, float* rows_f32,
                                          __nv_bfloat16* scan, int64_t dpad, float& nn, float& ee, float m,
                                          bool bf16_auth, float& r_out) {
    if (rows_f32) rows_f32[row * d + col] = x;
    const float xc = x - m;  // the scan copy holds the CENTRED row (see ingest_kernel)
    const __nv_bfloat16 b = __float2bfloat16_rn(xc);
    const float xb = __bfloat162float(b);
    if (scan) scan[row * dpad + col] = b;
    nn = fmaf(xb, xb, nn);
    float e = xc - xb;
    if (bf16_auth) e = auth_loss(m, xb, r_out);
    ee = fmaf(e, e, ee);
}

// mu[c] = (1/m) * sum of column c over rows [0, m): the centre the scan copy is taken around.  The same rows must give the
// same centre bit for bit -- bf16 storage rounds the stored rows around it, so a centre that moved in its last bit would
// give two indexes built from the same vectors rows that differ by a bf16 ulp here and there (float atomics did exactly
// that).  Every 64-row block sums its column in float32 in a fixed order and adds the sum to a 64-bit FIXED-POINT
// accumulator: integer addition is associative, the order in which the blocks arrive does not matter.
// The fixed-point scale is a power of two chosen PER COLUMN from the largest |block sum| of that column (a first pass;
// integer atomicMax on the float bits is order independent too): 2^e with nblocks * max|block sum| * 2^e <= 2^62, so the
// sum of every block fits the signed 64-bit word whatever the magnitude of the rows.  (A fixed 2^24 wrapped silently once
// |sum of the rows| passed 5.5e11 -- a column mean above 8.4e6 over 65536 rows -- and left a garbage centre.)  Scaling the
// rows by a power of two scales every block sum, the exponent and so the centre exactly: the centre is scale-equivariant.
// A block whose float32 sum is not finite -- a NaN or inf entry, or 64 rows whose sum overflows (same-sign entries above
// ~5e36) -- is left out of the sum of that column but still counts in m.
// The rows may arrive in pieces (a caller that stages them through a smaller buffer): every piece starts at a multiple of
// 64 rows, and the exponent uses the block count of all m rows, so the result does not depend on the staging.
__device__ __forceinline__ float block_col_sum(const float* __restrict__ src, int64_t rows, int d, int c) {
    const int64_t r0 = (int64_t)blockIdx.x * 64, r1 = r0 + 64 < rows ? r0 + 64 : rows;
    float a = 0.f;
    for (int64_t r = r0; r < r1; r++) a += src[r * d + c];
    return a;
}
__device__ __forceinline__ int mean_scale_exp(float amax, int64_t nblocks) {
    if (!(amax > 0.f)) return 0;   // every block sum of the column is 0 (or none is finite): any scale
    int ex;
    frexp((double)amax * (double)nblocks, &ex);   // exact product; nblocks * amax < 2^ex
    return 62 - ex;
}
// src: `rows` rows of the m; pass 0: colmax[c] = max |block sum| of column c; pass 1: acc[c] += block sum * 2^e(c)
__global__ void __launch_bounds__(256) mean_rows_kernel(const float* __restrict__ src, int64_t rows, int64_t m, int d,
                                                        float* __restrict__ colmax, unsigned long long* __restrict__ acc,
                                                        int pass) {
    const int64_t nblocks = (m + 63) / 64;
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
        const float a = block_col_sum(src, rows, d, c);
        if (!isfinite(a)) continue;   // the whole block is left out of this column (it still counts in m)
        if (pass == 0)
            atomic_max_nonneg(colmax + c, fabsf(a));
        else   // two's complement: signed sums
            atomicAdd(acc + c, (unsigned long long)__double2ll_rn(ldexp((double)a, mean_scale_exp(colmax[c], nblocks))));
    }
}
__global__ void mean_finish_kernel(const unsigned long long* __restrict__ acc, const float* __restrict__ colmax, int64_t m, int d,
                                   float* __restrict__ mu) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < d) mu[c] = (float)(ldexp((double)(long long)acc[c], -mean_scale_exp(colmax[c], (m + 63) / 64)) / (double)m);
}

// acc: d 64-bit words followed by d floats of device scratch
int launch_mean_begin(int d, unsigned long long* acc, cudaStream_t st) {
    B2F_CUDA(cudaMemsetAsync(acc, 0, (size_t)d * 12, st));
    return B2F_OK;
}
int launch_mean_pass(const float* src, int64_t row0, int64_t rows, int64_t m, int d, unsigned long long* acc, int pass,
                     cudaStream_t st) {
    if (rows <= 0) return B2F_OK;
    if (row0 % 64 != 0 || row0 + rows > m) {
        set_error("mean pass: piece [%lld, %lld) of %lld rows does not start on a 64-row block", (long long)row0,
                  (long long)(row0 + rows), (long long)m);
        return B2F_EINVAL;
    }
    mean_rows_kernel<<<(unsigned)((rows + 63) / 64), 256, 0, st>>>(src, rows, m, d, reinterpret_cast<float*>(acc + d), acc, pass);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}
int launch_mean_finish(int64_t m, int d, float* mu, unsigned long long* acc, cudaStream_t st) {
    if (m <= 0) return B2F_OK;
    mean_finish_kernel<<<(d + 255) / 256, 256, 0, st>>>(acc, reinterpret_cast<const float*>(acc + d), m, d, mu);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

// Centring.  With mu given, the scan copy is x~' = bf16(x - mu): distances are translation invariant
// (|q - x| = |(q - mu) - (x - mu)|), inner products split as q.x = (q - mu).(x - mu) + mu.x + (q.mu - mu.mu), so the
// tensor pass works on the centred vectors and the row term mu.x rides along as the per-row bias (L2: |x~'|^2,
// IP: -mu.x).  Embeddings share a large common component (the reference's own index: |x| ~ 7.7 with relative
// neighbour gaps of 1e-4; a random-init encoder: all cosines > 0.95), and bf16 rounding error scales with the
// magnitude of what is rounded: centred, the certification bound is 5-30x tighter on such data.
// stats[0] = max |x~'|^2, stats[1] = max |x' - x~'|^2 over every row ingested since the index was created or reset, or,
// after a removal, over the rows that survived it (taken again with this per-row arithmetic)
// bf16_auth (bf16 storage): there are no fp32 rows; the authoritative row is r = fl32(mu + x~'), so the IP bias is
// -mu.r and stats[1] bounds |(r - mu) - x~'| (what the fp32 addition loses: ~1e-7 |r|), not the bf16 rounding.
__global__ void __launch_bounds__(256)
ingest_kernel(const float* __restrict__ src, int64_t n, int d, float* __restrict__ rows_f32,
              __nv_bfloat16* __restrict__ scan, int64_t dpad, float* __restrict__ norms, float* __restrict__ stats,
              const float* __restrict__ mu, int ip_bias, int bf16_auth) {
    const int lane = threadIdx.x & 31;
    const int64_t wpg = (int64_t)gridDim.x * (blockDim.x >> 5);
    // running maxima of the warp's rows: ONE atomic pair per warp at the end (two atomics per row on the same
    // two addresses serialised the whole kernel: 2.8 ms for 1M rows, 21% of HBM)
    float max_nn = 0.f, max_ee = 0.f;
    for (int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < n; row += wpg) {
        float nn = 0.f, ee = 0.f;
        double mx = 0.0;  // mu.x in double: its rounding error would otherwise dominate the IP certification slack
        if ((d & 3) == 0) {
            for (int c = lane * 4; c < d; c += 128) {
                float4 x = ldg_stream(reinterpret_cast<const float4*>(src + row * d + c));
                if (rows_f32) *reinterpret_cast<float4*>(rows_f32 + row * d + c) = x;
                float4 m4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (mu) {
                    m4 = __ldg(reinterpret_cast<const float4*>(mu + c));
                    if (ip_bias && !bf16_auth) mx += (double)m4.x * x.x + (double)m4.y * x.y + (double)m4.z * x.z + (double)m4.w * x.w;
                    x.x -= m4.x; x.y -= m4.y; x.z -= m4.z; x.w -= m4.w;
                }
                const __nv_bfloat162 lo = __floats2bfloat162_rn(x.x, x.y), hi = __floats2bfloat162_rn(x.z, x.w);
                if (scan) {
                    uint2 pk;
                    pk.x = *reinterpret_cast<const uint32_t*>(&lo);
                    pk.y = *reinterpret_cast<const uint32_t*>(&hi);
                    *reinterpret_cast<uint2*>(scan + row * dpad + c) = pk;
                }
                const float b0 = __low2float(lo), b1 = __high2float(lo), b2 = __low2float(hi), b3 = __high2float(hi);
                nn = fmaf(b0, b0, nn); nn = fmaf(b1, b1, nn); nn = fmaf(b2, b2, nn); nn = fmaf(b3, b3, nn);
                float e0 = x.x - b0, e1 = x.y - b1, e2 = x.z - b2, e3 = x.w - b3;
                if (bf16_auth) {
                    // the authoritative row: r = fl32(mu + x~'); what matters is how far r - mu is from x~'
                    float r0, r1, r2, r3;
                    e0 = auth_loss(m4.x, b0, r0); e1 = auth_loss(m4.y, b1, r1);
                    e2 = auth_loss(m4.z, b2, r2); e3 = auth_loss(m4.w, b3, r3);
                    if (ip_bias) mx += (double)m4.x * r0 + (double)m4.y * r1 + (double)m4.z * r2 + (double)m4.w * r3;
                }
                ee = fmaf(e0, e0, ee); ee = fmaf(e1, e1, ee); ee = fmaf(e2, e2, ee); ee = fmaf(e3, e3, ee);
            }
        } else {
            for (int c = lane; c < d; c += 32) {
                const float x = src[row * d + c], m = mu ? mu[c] : 0.f;
                float r = x;
                emit_elem(x, row, c, d, rows_f32, scan, dpad, nn, ee, m, bf16_auth != 0, r);
                if (ip_bias) mx += (double)m * r;   // r = x (fp32 rows) or the authoritative rounded row (bf16 storage)
            }
        }
        if (scan)
            for (int c = d + lane; c < dpad; c += 32) scan[row * dpad + c] = __float2bfloat16_rn(0.f);
        nn = warp_sum(nn);
        ee = warp_sum(ee);
        if (ip_bias) mx = warp_sum(mx);
        if (lane == 0 && norms) norms[row] = ip_bias ? (float)(-mx) : nn;   // the row's bias in the tensor pass
        max_nn = fmaxf(max_nn, nn);
        max_ee = fmaxf(max_ee, ee);
    }
    if (lane == 0 && stats) {
        atomic_max_nonneg(stats, max_nn);
        atomic_max_nonneg(stats + 1, max_ee);
    }
}

int launch_ingest(const float* src, int64_t n, int d, float* rows_f32, __nv_bfloat16* scan, int64_t dpad, float* norms,
                  float* stats, const float* mu, int ip_bias, int bf16_auth, cudaStream_t st) {
    if (n <= 0) return B2F_OK;
    const int wpb = 8;
    int64_t blocks = (n + wpb - 1) / wpb;
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    ingest_kernel<<<(unsigned)blocks, wpb * 32, 0, st>>>(src, n, d, rows_f32, scan, dpad, norms, stats, mu, ip_bias, bf16_auth);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

// stats over the survivors of a bf16-storage index, from its scan copy: the per-row arithmetic of ingest_kernel's
// bf16_auth branch (same lanes, same fmaf order, the same auth_loss), so the maxima equal an ingest of the same rows
__global__ void __launch_bounds__(256)
scan_stats_kernel(const __nv_bfloat16* __restrict__ scan, int64_t n, int d, int64_t dpad, const float* __restrict__ mu,
                  float* __restrict__ stats) {
    const int lane = threadIdx.x & 31;
    const int64_t wpg = (int64_t)gridDim.x * (blockDim.x >> 5);
    float max_nn = 0.f, max_ee = 0.f;
    for (int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < n; row += wpg) {
        float nn = 0.f, ee = 0.f, r;
        if ((d & 3) == 0) {
            for (int c = lane * 4; c < d; c += 128) {
                const uint2 pk = *reinterpret_cast<const uint2*>(scan + row * dpad + c);
                const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162*>(&pk.x), hi = *reinterpret_cast<const __nv_bfloat162*>(&pk.y);
                const float4 m4 = mu ? __ldg(reinterpret_cast<const float4*>(mu + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
                const float b0 = __low2float(lo), b1 = __high2float(lo), b2 = __low2float(hi), b3 = __high2float(hi);
                nn = fmaf(b0, b0, nn); nn = fmaf(b1, b1, nn); nn = fmaf(b2, b2, nn); nn = fmaf(b3, b3, nn);
                const float e0 = auth_loss(m4.x, b0, r), e1 = auth_loss(m4.y, b1, r), e2 = auth_loss(m4.z, b2, r), e3 = auth_loss(m4.w, b3, r);
                ee = fmaf(e0, e0, ee); ee = fmaf(e1, e1, ee); ee = fmaf(e2, e2, ee); ee = fmaf(e3, e3, ee);
            }
        } else {
            for (int c = lane; c < d; c += 32) {
                const float xb = __bfloat162float(scan[row * dpad + c]);
                nn = fmaf(xb, xb, nn);
                const float e = auth_loss(mu ? mu[c] : 0.f, xb, r);
                ee = fmaf(e, e, ee);
            }
        }
        nn = warp_sum(nn);
        ee = warp_sum(ee);
        max_nn = fmaxf(max_nn, nn);
        max_ee = fmaxf(max_ee, ee);
    }
    if (lane == 0) {
        atomic_max_nonneg(stats, max_nn);
        atomic_max_nonneg(stats + 1, max_ee);
    }
}

int launch_scan_stats(const __nv_bfloat16* scan, int64_t n, int d, int64_t dpad, const float* mu, float* stats, cudaStream_t st) {
    if (n <= 0) return B2F_OK;
    int64_t blocks = (n + 7) / 8;
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    scan_stats_kernel<<<(unsigned)blocks, 256, 0, st>>>(scan, n, d, dpad, mu, stats);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

// K7.  One CTA per sequence.  hidden [B,T,d] fp32, mask [B,T] int64 (may be null = all ones).
// CLS: row = hidden[b,0,:] (vectorization.py:44).  MEAN: sum_t mask*h / max(sum_t mask, 1e-9).
// normalize: row /= max(|row|, 1e-12).  The result goes to out_f32 [B,d]: staged index rows, which the ingest
// kernel then takes like any other add's, or a plain output.
__global__ void __launch_bounds__(256)
pool_kernel(const float* __restrict__ hidden, const int64_t* __restrict__ mask, int64_t T, int d, int pool, int normalize,
            float* __restrict__ out_f32) {
    extern __shared__ float srow[];  // [d]
    __shared__ float red[8];
    const int64_t b = blockIdx.x;
    const float* h = hidden + b * T * d;
    float cnt = 1.f;
    if (pool == B2F_POOL_MEAN) {
        float c = 0.f;
        for (int64_t t = 0; t < T; t++) c += mask ? (float)mask[b * T + t] : 1.f;  // uniform, L1-broadcast
        cnt = fmaxf(c, 1e-9f);
    }
    float ss = 0.f;
    if (pool == B2F_POOL_MEAN && (d & 3) == 0 && d / 4 <= (int)blockDim.x) {
        // 16-byte loads: a thread owns one group of four columns and every nth-th token (d = 384: 96 column
        // groups x 2 token phases), four tokens in flight; the partial sums of the phases meet in shared
        // memory (psum [nth][d] behind srow).  Masked-out tokens are skipped, as in the scalar path.
        float* psum = srow + d;
        const int ncg = d / 4, nth = (int)blockDim.x / ncg;
        const int cg = (int)threadIdx.x % ncg, th = (int)threadIdx.x / ncg;
        float4* const part = reinterpret_cast<float4*>(psum + th * d + cg * 4);   // this thread's partial sums
        if (th < nth) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int64_t t0 = th; t0 < T; t0 += 4 * nth) {
                float4 v[4];
                float mk[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int64_t t = t0 + (int64_t)u * nth;
                    mk[u] = t < T ? (mask ? (float)mask[b * T + t] : 1.f) : 0.f;
                    v[u] = mk[u] != 0.f ? ldg_stream(reinterpret_cast<const float4*>(h + t * d + cg * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    acc.x = fmaf(mk[u], v[u].x, acc.x); acc.y = fmaf(mk[u], v[u].y, acc.y);
                    acc.z = fmaf(mk[u], v[u].z, acc.z); acc.w = fmaf(mk[u], v[u].w, acc.w);
                }
            }
            *part = acc;
        }
        __syncthreads();
        for (int c = threadIdx.x; c < d; c += blockDim.x) {
            float a = 0.f;
            for (int p2 = 0; p2 < nth; p2++) a += psum[p2 * d + c];
            const float v = a / cnt;
            srow[c] = v;
            ss = fmaf(v, v, ss);
        }
    } else {
        for (int c = threadIdx.x; c < d; c += blockDim.x) {
            float v;
            if (pool == B2F_POOL_CLS) {
                v = h[c];
            } else {
                float acc = 0.f;
                for (int64_t t = 0; t < T; t++) {
                    const float m = mask ? (float)mask[b * T + t] : 1.f;
                    if (m != 0.f) acc = fmaf(m, h[t * d + c], acc);
                }
                v = acc / cnt;
            }
            srow[c] = v;
            ss = fmaf(v, v, ss);
        }
    }
    ss = warp_sum(ss);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    float tot = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) tot += red[w];
    const float scale = normalize ? 1.f / fmaxf(sqrtf(tot), 1e-12f) : 1.f;
    for (int c = threadIdx.x; c < d; c += blockDim.x) out_f32[b * d + c] = srow[c] * scale;
}

int launch_pool(const float* hidden, const int64_t* mask, int64_t B, int64_t T, int d, int pool, int normalize,
                float* out_f32, cudaStream_t st) {
    if (B <= 0) return B2F_OK;
    if (T <= 0 || (pool != B2F_POOL_CLS && pool != B2F_POOL_MEAN)) {
        set_error("pool: bad T=%lld or pool mode %d", (long long)T, pool);
        return B2F_EINVAL;
    }
    if ((size_t)d * 4 > 48 * 1024) {
        set_error("pool: d=%d too large", d);
        return B2F_EINVAL;
    }
    // srow [d] + the mean path's partial sums [256 / (d/4)][d]
    const int nth = (d % 4 == 0 && d / 4 <= 256) ? 256 / (d / 4) : 0;
    const size_t smem = (size_t)d * 4 * (1 + (pool == B2F_POOL_MEAN ? nth : 0));
    if (smem > 48 * 1024) {
        static size_t configured[kMaxDevices] = {};
        const int dev = current_device_slot();
        std::lock_guard<std::mutex> lk(launch_cache_mutex());
        if (smem > configured[dev]) {
            B2F_CUDA(cudaFuncSetAttribute(pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
            configured[dev] = 160 * 1024;
        }
    }
    pool_kernel<<<(unsigned)B, 256, smem, st>>>(hidden, mask, T, d, pool, normalize, out_f32);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

// ---- synthetic rows: bit-identical twin of oracle/flat_oracle.c orc_synth_rows ---------------------
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z ^= z >> 30; z *= 0xbf58476d1ce4e5b9ULL;
    z ^= z >> 27; z *= 0x94d049bb133111ebULL;
    z ^= z >> 31; return z;
}
__device__ __forceinline__ int32_t synth_int(uint64_t seed, uint64_t idx) {
    const uint64_t a = mix64(seed + 0x9E3779B97F4A7C15ULL * (2 * idx + 1));
    const uint64_t b = mix64(a ^ 0xD1B54A32D192ED03ULL);
    const uint64_t c = mix64(b + idx);
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        s += (uint32_t)((a >> (16 * i)) & 0xffff);
        s += (uint32_t)((b >> (16 * i)) & 0xffff);
        s += (uint32_t)((c >> (16 * i)) & 0xffff);
    }
    return (int32_t)s - 393210;
}

__global__ void __launch_bounds__(256)
synth_kernel(uint64_t seed, int64_t row0, int64_t nrows, int d, int normalize, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t wpg = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < nrows; r += wpg) {
        const uint64_t base = (uint64_t)(row0 + r) * (uint64_t)d;
        if (!normalize) {
            for (int c = lane; c < d; c += 32) out[r * d + c] = (float)synth_int(seed, base + c) * (1.0f / 65536.0f);
        } else {
            long long ss = 0;
            for (int c = lane; c < d; c += 32) {
                const long long v = synth_int(seed, base + c);
                ss += v * v;
            }
#pragma unroll
            for (int s = 16; s >= 1; s >>= 1) ss += __shfl_xor_sync(kFull, ss, s);
            const double nrm = sqrt((double)ss);
            for (int c = lane; c < d; c += 32) {
                const double v = (double)synth_int(seed, base + c);
                out[r * d + c] = ss > 0 ? (float)(v / nrm) : 0.f;
            }
        }
    }
}

int launch_synth(uint64_t seed, int64_t row0, int64_t nrows, int d, int normalize, float* out, cudaStream_t st) {
    if (nrows <= 0) return B2F_OK;
    int64_t blocks = (nrows + 7) / 8;
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    synth_kernel<<<(unsigned)blocks, 256, 0, st>>>(seed, row0, nrows, d, normalize, out);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

// ---- query preparation for the tensor path -------------------------------------------------------
// q' = q - mu (mu may be null); qb: [nq_pad, dpad] bf16(q') (zero padded), qnorm[r] = |bf16(q'_r)|^2,
// qerr[r] = |q'_r - bf16(q'_r)|, qconst[r] = q_r.mu - mu.mu (turns centred inner products back into true ones)
__global__ void __launch_bounds__(256)
prep_queries_kernel(const float* __restrict__ q, int nq, int nq_pad, int d, __nv_bfloat16* __restrict__ qb, int64_t dpad,
                    float* __restrict__ qnorm, float* __restrict__ qerr, float* __restrict__ qconst, const float* __restrict__ mu,
                    uint32_t* __restrict__ zero, int zero_words, uint32_t* __restrict__ fill, int64_t fill_words) {
    {
        const int64_t gt = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, gn = (int64_t)gridDim.x * blockDim.x;
        for (int64_t i = gt; i < zero_words; i += gn) zero[i] = 0u;
        for (int64_t i = gt; i < fill_words; i += gn) fill[i] = 0x7f7f7f7fu;
    }
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= nq_pad) return;
    float nn = 0.f, ee = 0.f;
    double qc = 0.0;
    for (int c = lane; c < dpad; c += 32) {
        const bool in = r < nq && c < d;
        const float m = (mu && in) ? mu[c] : 0.f;
        const float x0 = in ? q[(int64_t)r * d + c] : 0.f;
        const float x = x0 - m;
        const __nv_bfloat16 b = __float2bfloat16_rn(x);
        const float xb = __bfloat162float(b);
        qb[(int64_t)r * dpad + c] = b;
        nn = fmaf(xb, xb, nn);
        ee = fmaf(x - xb, x - xb, ee);
        qc += (double)m * ((double)x0 - (double)m);   // (q - mu).mu = q.mu - mu.mu, in double
    }
    nn = warp_sum(nn);
    ee = warp_sum(ee);
    qc = warp_sum(qc);
    if (lane == 0 && r < nq) {
        qnorm[r] = nn;
        qerr[r] = sqrtf(ee);
        qconst[r] = (float)qc;
    }
}

int launch_prep_queries(const float* q, int nq, int nq_pad, int d, __nv_bfloat16* qb, int64_t dpad, float* qnorm,
                        float* qerr, float* qconst, const float* mu, uint32_t* zero, int zero_words, uint32_t* fill,
                        int64_t fill_words, cudaStream_t st) {
    if (nq_pad <= 0) return B2F_OK;
    prep_queries_kernel<<<(nq_pad + 7) / 8, 256, 0, st>>>(q, nq, nq_pad, d, qb, dpad, qnorm, qerr, qconst, mu, zero, zero_words,
                                                          fill, fill_words);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

// the authoritative rows of a bf16-storage index: r = fl32(mu + x~') (mu null: the rounded rows themselves)
// ---- range pass (second tensor pass over the queries the first could not certify) ------------------------------------
// gather: failed query i (fail_list[i], i < *nfail) with a usable exact k-th key tau goes to slot s of the compact batch
// (its fp32 vector to qf[s], tau to tau2[s], its index in the whole batch to out_map[s]); the others (list overflow, fewer
// than k valid candidates: tau = FLT_MAX) go straight to the exact scan's list.  out_map is pre-filled with -1, qf with 0.
__global__ void __launch_bounds__(256)
gather_failed_kernel(const float* __restrict__ q, int d, const int32_t* __restrict__ fail_list, const float* __restrict__ fail_tau,
                     const int32_t* __restrict__ nfail, int cap, float* __restrict__ qf, float* __restrict__ tau2,
                     int32_t* __restrict__ out_map, int32_t* __restrict__ range_count, int32_t* __restrict__ fail_list2,
                     int32_t* __restrict__ fail_count2) {
    const int lane = threadIdx.x & 31;
    const int n = *nfail;
    for (int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += gridDim.x * (blockDim.x >> 5)) {
        const int32_t orig = fail_list[i];
        const float tau = fail_tau[i];
        int slot = -1;
        if (lane == 0) {
            if (tau < 1.0e37f) {
                slot = atomicAdd(range_count, 1);
                if (slot >= cap) slot = -1;   // more failures than the range pass holds: exact scan
            }
            if (slot < 0) fail_list2[atomicAdd(fail_count2, 1)] = orig;
            else { tau2[slot] = tau; out_map[slot] = orig; }
        }
        slot = __shfl_sync(kFull, slot, 0);
        if (slot >= 0)
            for (int c = lane; c < d; c += 32) qf[(int64_t)slot * d + c] = q[(int64_t)orig * d + c];
    }
}

int launch_gather_failed(const float* q, int d, const int32_t* fail_list, const float* fail_tau, const int32_t* nfail, int nfail_host,
                         int cap, float* qf, float* tau2, int32_t* out_map, int32_t* range_count, int32_t* fail_list2,
                         int32_t* fail_count2, cudaStream_t st) {
    if (nfail_host <= 0) return B2F_OK;
    int blocks = (nfail_host + 7) / 8;
    if (blocks > kNumSMs * 4) blocks = kNumSMs * 4;
    gather_failed_kernel<<<blocks, 256, 0, st>>>(q, d, fail_list, fail_tau, nfail, cap, qf, tau2, out_map, range_count, fail_list2, fail_count2);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

// The fixed threshold of a range query: every row whose exact key is <= tau (the k-th key already found, so: every true
// top-k row) has a coarse key <= thr.  Inverse of the certification test (rerank_certified) with a 1e-6 margin on tau, so
// that re-ranking everything at or below thr certifies by construction.
__global__ void range_thresholds_kernel(const float* __restrict__ tau2, float tau_all, const int32_t* __restrict__ out_map, int n, int d, int l2,
                                        const float* __restrict__ qnorm, const float* __restrict__ qerr,
                                        const float* __restrict__ qconst, float max_row_norm, float max_row_err, float mu_norm,
                                        float* __restrict__ thr) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (out_map && out_map[i] < 0) {
        thr[i] = -__int_as_float(0x7f800000);   // unused slot: nothing is listed
        return;
    }
    const float tau = tau2 ? tau2[i] : tau_all;
    const float qn2 = qnorm[i], qn = sqrtf(qn2), eq = qerr[i];
    const float gam = 4.f * (float)(d + 16) * 5.9604645e-8f;
    if (l2) {
        const float nu = gam * (2.f * qn * max_row_norm + qn2 + max_row_norm * max_row_norm);
        const float t = fmaxf(tau, 0.f) * (1.f + 2e-6f) + 1e-30f;
        const float L = sqrtf(t) * (1.f + 1e-6f) + eq + max_row_err;   // certified <=> (sqrt(c + qn2 - nu) - eq - E)^2 (1 - 4e-7) > tau
        // thr is a difference of numbers as large as |q~|^2 while L^2 can be thousands of times smaller (near-duplicates):
        // the margin covers the fp32 rounding of this difference and of the one the test undoes it with, in units of the
        // LARGE terms (16 ulp), not of the result
        thr[i] = L * L - qn2 + nu + (L * L + qn2 + nu) * 1e-6f + 1e-30f;
    } else {
        const float cq = qconst ? qconst[i] : 0.f;
        const float xmax = max_row_norm + max_row_err + mu_norm;
        const float nu = gam * qn * max_row_norm + 2.4e-7f * (mu_norm * (xmax + qn + eq + mu_norm) + qn * max_row_norm);
        const float slack = nu + (qn + eq) * max_row_err + max_row_norm * eq;
        // certified <=> -thr + cq + slack < -tau  <=>  thr > tau + cq + slack
        const float base = tau + cq + slack;
        thr[i] = base + (fabsf(tau) + fabsf(cq) + slack) * 1e-6f + 1e-30f;   // margin in units of the terms (they may cancel)
    }
}

int launch_range_thresholds(const float* tau2, float tau_all, const int32_t* out_map, int n, int d, int metric, const float* qnorm,
                            const float* qerr, const float* qconst, float max_row_norm, float max_row_err, float mu_norm, float* thr,
                            cudaStream_t st) {
    if (n <= 0) return B2F_OK;
    range_thresholds_kernel<<<(n + 255) / 256, 256, 0, st>>>(tau2, tau_all, out_map, n, d, metric == B2F_METRIC_L2 ? 1 : 0, qnorm, qerr, qconst,
                                                            max_row_norm, max_row_err, mu_norm, thr);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

__global__ void bf16_to_f32_kernel(const __nv_bfloat16* __restrict__ src, int64_t pitch, int64_t n, int d,
                                   const float* __restrict__ mu, float* __restrict__ dst) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * d) return;
    const int64_t r = t / d;
    const int c = (int)(t - r * d);
    const float v = __bfloat162float(src[r * pitch + c]);
    dst[t] = mu ? mu[c] + v : v;
}

int launch_bf16_to_f32(const __nv_bfloat16* src, int64_t pitch, int64_t n, int d, const float* mu, float* dst, cudaStream_t st) {
    const int64_t total = n * d;
    if (total <= 0) return B2F_OK;
    bf16_to_f32_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(src, pitch, n, d, mu, dst);
    B2F_CUDA(cudaGetLastError());
    return B2F_OK;
}

}  // namespace b2f
