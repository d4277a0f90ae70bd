// GroupNorm(32)(+SiLU) and LayerNorm, forward and backward, over channels-last bf16 activations (sm_100a).
//
// Replaces the ATen group_norm / silu / layer_norm calls inside diffusers' ResnetBlock2D, Transformer2DModel
// and BasicTransformerBlock that the reference reaches through train.py:2760 (SURVEY.md 2.1 rows K6, K7).
// Numerics contract (SURVEY.md 8a): statistics and the normalise(+SiLU) math in fp32, ONE rounding to bf16
// on store -- what CUDA autocast does (fp32 norm output rounded when the next conv/linear casts its input).
// All kernels are HBM-streaming: 16-byte vector accesses along the contiguous channel dimension, fp32
// partial sums reduced with warp shuffles, deterministic two-level reductions (no atomics).
//   GroupNorm fwd: 4 B/element (stats pass re-read is served from L2 for SDXL sizes, <= 84 MB per tensor)
//   LayerNorm fwd: 4 B/element; bwd 6 B/element.
#include "common.cuh"

namespace aoz {

constexpr int GN_GROUPS = 32;
constexpr int GN_THREADS = 512;            // upper bound; blocks are launched with cols * row_lanes threads (gn_block_threads)
constexpr int GN_MAX_CHUNKS = 160;         // pixel chunks per image of the backward statistics (per-channel partial rows)
constexpr int GN_FWD_MAX_CHUNKS = 256;     // forward statistics: a partial row is only [32 groups][2]
__device__ unsigned int g_gn_tickets[1024];     // zero at module load; atomicInc wraps back to zero after every use

__device__ __forceinline__ void unpack8(const uint4& a, float* f) {
    f[0] = bf16lo(a.x); f[1] = bf16hi(a.x); f[2] = bf16lo(a.y); f[3] = bf16hi(a.y);
    f[4] = bf16lo(a.z); f[5] = bf16hi(a.z); f[6] = bf16lo(a.w); f[7] = bf16hi(a.w);
}
__device__ __forceinline__ uint4 pack8(const float* f) {
    return make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }
// eight bf16 -> four float2 (elements 2e, 2e+1) for the packed fp32x2 instructions of sm_100 (FADD2 / FMUL2 / FFMA2: two IEEE
// operations per issue slot)
__device__ __forceinline__ void unpack8v(const uint4& a, float2* f) {
    f[0] = make_float2(bf16lo(a.x), bf16hi(a.x)); f[1] = make_float2(bf16lo(a.y), bf16hi(a.y));
    f[2] = make_float2(bf16lo(a.z), bf16hi(a.z)); f[3] = make_float2(bf16lo(a.w), bf16hi(a.w));
}

// ---------------------------------------------------------------------------------------------
// GroupNorm statistics: x [NB, HW, C] -> partial [NB][chunks][GROUPS][2] (sum, sumsq of x - pivot) -> mean / rstd [NB][GROUPS]
// The sums are taken of x - pivot with pivot = x[n, 0, g * cpg] (the group's first element), so var = E[d^2] - E[d]^2 subtracts two
// numbers of the size of the variance: E[x^2] - mean^2 cancels catastrophically once |mean| >> std (offset activations), and
// Welford's update would cost a division per element.  Still one pass, same order, deterministic.
// grid (chunks, NB) ~ one block per SM; block = `cols` vector columns x `row_lanes` row lanes (<= 1024 threads, rounded up to
// whole warps).  A thread owns one 8-channel vector column and walks its row lane of the chunk with four rows in flight.
// No float atomics anywhere (they would make the low bits of every statistic and gradient differ run to run): the row-lane
// partials go to shared memory [row_lanes][2][C], ONE barrier, then 16 threads per (group, sum|sumsq) add the group's
// row_lanes * C/32 entries in a fixed order.  The last block of an image (self-resetting ticket) reduces the chunk partials
// the same way and writes mean / rstd, so the apply kernel starts streaming immediately.
__device__ __forceinline__ float half_warp_sum_fixed(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v;
}

__global__ void __launch_bounds__(1024)
gn_stats_kernel(const __nv_bfloat16* __restrict__ x, int HW, int C, float eps, int cols, int row_lanes, float* __restrict__ partial,
                float* __restrict__ mean_out, float* __restrict__ rstd_out) {
    pdl_enter();
    extern __shared__ float sm[];          // [row_lanes][2][C]
    __shared__ float s_fin[2][GN_GROUPS];
    __shared__ unsigned int s_last;
    const int n = blockIdx.y, chunk = blockIdx.x, chunks = gridDim.x;
    const int vec_per_row = C / 8;
    const int rows_per_chunk = (HW + chunks - 1) / chunks;
    const int r0 = chunk * rows_per_chunk, r1 = min(HW, r0 + rows_per_chunk);
    const __nv_bfloat16* xb = x + (size_t)n * HW * C;
    const int tc = threadIdx.x % cols, tr = threadIdx.x / cols;
    const int cpg = C / GN_GROUPS;
    if (tr < row_lanes) {
        for (int v = tc; v < vec_per_row; v += cols) {             // one trip unless C/8 exceeds the block (then row_lanes == 1)
            float s[8], q[8], pv[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) { s[e] = 0.f; q[e] = 0.f; pv[e] = __bfloat162float(xb[((v * 8 + e) / cpg) * cpg]); }
            int r = r0 + tr;
            for (; r + 3 * row_lanes < r1; r += 4 * row_lanes) {           // four rows in flight
                uint4 px[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) px[u] = ld_stream(xb + (size_t)(r + u * row_lanes) * C + v * 8);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    float f[8];
                    unpack8(px[u], f);
#pragma unroll
                    for (int e = 0; e < 8; ++e) { const float d = f[e] - pv[e]; s[e] += d; q[e] = fmaf(d, d, q[e]); }
                }
            }
            for (; r < r1; r += row_lanes) {
                float f[8];
                unpack8(ld_stream(xb + (size_t)r * C + v * 8), f);
#pragma unroll
                for (int e = 0; e < 8; ++e) { const float d = f[e] - pv[e]; s[e] += d; q[e] = fmaf(d, d, q[e]); }
            }
            float* d = sm + (size_t)tr * 2 * C + v * 8;
#pragma unroll
            for (int e = 0; e < 8; ++e) { d[e] = s[e]; d[C + e] = q[e]; }
        }
    }
    __syncthreads();
    // (group, which) pairs: 16 threads each, fixed summation order
    const int sub = threadIdx.x & 15;
    const int count = row_lanes * cpg;
    for (int p = threadIdx.x >> 4; p < 2 * GN_GROUPS; p += blockDim.x >> 4) {
        const int g = p & (GN_GROUPS - 1), which = p >> 5;
        float a = 0.f;
        for (int idx = sub; idx < count; idx += 16) {
            const int l = idx / cpg, c = idx - l * cpg;
            a += sm[(size_t)(l * 2 + which) * C + g * cpg + c];
        }
        a = half_warp_sum_fixed(a);
        if (sub == 0) partial[(((size_t)n * chunks + chunk) * GN_GROUPS + g) * 2 + which] = a;
    }
    // the LAST block of this image turns the chunk partials into mean / rstd
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicInc(&g_gn_tickets[n & 1023], (unsigned int)chunks - 1);
        s_last = (t == (unsigned int)chunks - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int p = threadIdx.x >> 4; p < 2 * GN_GROUPS; p += blockDim.x >> 4) {
        const int g = p & (GN_GROUPS - 1), which = p >> 5;
        float a = 0.f;
        for (int k = sub; k < chunks; k += 16) a += __ldcg(partial + (((size_t)n * chunks + k) * GN_GROUPS + g) * 2 + which);
        a = half_warp_sum_fixed(a);
        if (sub == 0) s_fin[which][g] = a;
    }
    __syncthreads();
    if (threadIdx.x < GN_GROUPS) {
        const int g = threadIdx.x;
        const float cnt = (float)HW * (float)cpg;
        const float dm = s_fin[0][g] / cnt;                      // mean of x - pivot
        const float var = fmaxf(s_fin[1][g] / cnt - dm * dm, 0.f);
        const float mean = __bfloat162float(xb[g * cpg]) + dm;
        mean_out[n * GN_GROUPS + g] = mean;
        rstd_out[n * GN_GROUPS + g] = rsqrtf(var + eps);
    }
}

// GroupNorm apply: y = silu?((x - mean) * rstd * gamma + beta); also writes mean/rstd [NB][GROUPS] (chunk 0 block)
__global__ void __launch_bounds__(GN_THREADS)
gn_apply_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ gamma,
                const __nv_bfloat16* __restrict__ beta, const float* __restrict__ mean, const float* __restrict__ rstd,
                int HW, int C, int silu, __nv_bfloat16* __restrict__ y) {
    pdl_enter();
    __shared__ float s_mean[GN_GROUPS], s_rstd[GN_GROUPS];
    const int n = blockIdx.y;
    const int cpg = C / GN_GROUPS;
    if (threadIdx.x < GN_GROUPS) {
        s_mean[threadIdx.x] = mean[n * GN_GROUPS + threadIdx.x];
        s_rstd[threadIdx.x] = rstd[n * GN_GROUPS + threadIdx.x];
    }
    __syncthreads();
    // A thread owns one 8-channel vector column (its gamma / beta / mean / rstd stay in registers: no per-element group
    // division or shared-memory lookup in the loop) and walks its row lane of this block's pixel chunk, four rows in flight.
    const int vec_per_row = C / 8;
    const int cols = min(vec_per_row, (int)blockDim.x);
    const int row_lanes = (int)blockDim.x / cols;
    const int tc = threadIdx.x % cols, tr = threadIdx.x / cols;
    const int rows_per_chunk = (HW + gridDim.x - 1) / gridDim.x;
    const int r0 = blockIdx.x * rows_per_chunk, r1 = min(HW, r0 + rows_per_chunk);
    const __nv_bfloat16* xb = x + (size_t)n * HW * C;
    __nv_bfloat16* yb = y + (size_t)n * HW * C;
    if (tr >= row_lanes) return;
    for (int v = tc; v < vec_per_row; v += cols) {
        float gm[8], bt[8], sc[8], sh[8];
        unpack8(*reinterpret_cast<const uint4*>(gamma + v * 8), gm);
        unpack8(*reinterpret_cast<const uint4*>(beta + v * 8), bt);
#pragma unroll
        for (int e = 0; e < 8; ++e) {                          // z = x * sc + sh
            const int g = (v * 8 + e) / cpg;
            sc[e] = s_rstd[g] * gm[e];
            sh[e] = bt[e] - s_mean[g] * sc[e];
        }
        auto one = [&](const uint4& px, int r) {
            float f[8];
            unpack8(px, f);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float z = fmaf(f[e], sc[e], sh[e]);
                if (silu) z = z * sigmoidf_(z);
                f[e] = z;
            }
            st_stream(yb + (size_t)r * C + v * 8, pack8(f));
        };
        int r = r0 + tr;
        for (; r + 3 * row_lanes < r1; r += 4 * row_lanes) {
            uint4 px[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) px[u] = ld_stream(xb + (size_t)(r + u * row_lanes) * C + v * 8);
#pragma unroll
            for (int u = 0; u < 4; ++u) one(px[u], r + u * row_lanes);
        }
        for (; r < r1; r += row_lanes) one(ld_stream(xb + (size_t)r * C + v * 8), r);
    }
}

// GroupNorm backward pass 1: per-channel sums of dz and dz*xhat over a pixel chunk.
// partial [NB][chunks][2][C]
__global__ void __launch_bounds__(GN_THREADS, 1)
gn_bwd_stats_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x,
                    const __nv_bfloat16* __restrict__ gamma, const __nv_bfloat16* __restrict__ beta,
                    const float* __restrict__ mean, const float* __restrict__ rstd, int HW, int C, int silu, int cols,
                    int row_lanes, float* __restrict__ partial) {
    pdl_enter();
    extern __shared__ float sm[];          // [row_lanes][2][C]
    __shared__ float s_mean[GN_GROUPS], s_rstd[GN_GROUPS];
    const int n = blockIdx.y, chunk = blockIdx.x, chunks = gridDim.x;
    const int cpg = C / GN_GROUPS;
    if (threadIdx.x < GN_GROUPS) { s_mean[threadIdx.x] = mean[n * GN_GROUPS + threadIdx.x]; s_rstd[threadIdx.x] = rstd[n * GN_GROUPS + threadIdx.x]; }
    __syncthreads();
    const int vec_per_row = C / 8;
    const int rows_per_chunk = (HW + chunks - 1) / chunks;
    const int r0 = chunk * rows_per_chunk, r1 = min(HW, r0 + rows_per_chunk);
    const size_t base = (size_t)n * HW * C;
    const int tc = threadIdx.x % cols, tr = threadIdx.x / cols;
    float a[8], b[8];
    if (tr < row_lanes) {
        for (int v = tc; v < vec_per_row; v += cols) {
            float gm[8], bt[8], mu[8], rs[8];
            unpack8(*reinterpret_cast<const uint4*>(gamma + v * 8), gm);
            unpack8(*reinterpret_cast<const uint4*>(beta + v * 8), bt);
#pragma unroll
            for (int e = 0; e < 8; ++e) { a[e] = 0.f; b[e] = 0.f; const int g = (v * 8 + e) / cpg; mu[e] = s_mean[g]; rs[e] = s_rstd[g]; }
            auto acc_row = [&](const uint4& px, const uint4& pd) {
                float fx[8], fd[8];
                unpack8(px, fx);
                unpack8(pd, fd);
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const float xh = (fx[e] - mu[e]) * rs[e];
                    float dz = fd[e];
                    if (silu) {
                        const float z = xh * gm[e] + bt[e];
                        const float sg = sigmoidf_(z);
                        dz *= sg * (1.0f + z * (1.0f - sg));
                    }
                    a[e] += dz; b[e] = fmaf(dz, xh, b[e]);
                }
            };
            int r = r0 + tr;
            for (; r + 3 * row_lanes < r1; r += 4 * row_lanes) {           // four rows (eight 16-byte loads) in flight
                uint4 px[4], pd[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const size_t o = base + (size_t)(r + u * row_lanes) * C + v * 8;
                    px[u] = ld_stream(x + o);
                    pd[u] = ld_stream(dy + o);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) acc_row(px[u], pd[u]);
            }
            for (; r < r1; r += row_lanes) acc_row(ld_stream(x + base + (size_t)r * C + v * 8), ld_stream(dy + base + (size_t)r * C + v * 8));
            float* d = sm + (size_t)tr * 2 * C + v * 8;
#pragma unroll
            for (int e = 0; e < 8; ++e) { d[e] = a[e]; d[C + e] = b[e]; }
        }
    }
    __syncthreads();
    float* out = partial + ((size_t)n * chunks + chunk) * 2 * C;
    for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) {        // fixed-order sum over the row lanes
        float t = 0.f;
        for (int l = 0; l < row_lanes; ++l) t += sm[(size_t)l * 2 * C + i];
        out[i] = t;
    }
}

// pass 2a: one block per (group, image): reduce the chunk partials of the group's channels, write the per-channel
// sums chansum[n][2][C] and the group terms db = sum_c gamma*A, ds = sum_c gamma*B  -> group_terms[n][g][2]
__global__ void __launch_bounds__(128)
gn_bwd_group_kernel(const float* __restrict__ partial, const __nv_bfloat16* __restrict__ gamma, int chunks, int C,
                    float* __restrict__ chansum, float* __restrict__ group_terms) {
    pdl_enter();
    __shared__ float s_db[128], s_ds[128], s_a[128], s_b[128];
    const int g = blockIdx.x, n = blockIdx.y;
    const int cpg = C / GN_GROUPS;
    float db = 0.f, ds = 0.f;
    // thread t handles channel (t % cpg) of the group and chunk lanes (t / cpg) when cpg < 128
    const int lanes = max(1, 128 / cpg);
    const int cl = threadIdx.x % cpg, kl = threadIdx.x / cpg;
    if (kl < lanes) {
        for (int c0 = cl; c0 < cpg; c0 += (lanes > 1 ? cpg : 128)) {
            const int c = g * cpg + c0;
            float a = 0.f, b = 0.f;
            for (int k = kl; k < chunks; k += lanes) {
                const float* p = partial + ((size_t)n * chunks + k) * 2 * C;
                a += p[c]; b += p[C + c];
            }
            if (lanes == 1) {
                chansum[((size_t)n * 2 + 0) * C + c] = a;
                chansum[((size_t)n * 2 + 1) * C + c] = b;
                const float gm = __bfloat162float(gamma[c]);
                db = fmaf(gm, a, db); ds = fmaf(gm, b, ds);
            } else {                                   // cpg < 128: one channel per (cl), chunk lanes combined in fixed order below
                s_a[kl * cpg + cl] = a;
                s_b[kl * cpg + cl] = b;
            }
        }
    }
    if (lanes > 1) {
        __syncthreads();
        if (threadIdx.x < cpg) {
            const int c = g * cpg + threadIdx.x;
            float a = 0.f, b = 0.f;
            for (int k = 0; k < lanes; ++k) { a += s_a[k * cpg + threadIdx.x]; b += s_b[k * cpg + threadIdx.x]; }
            chansum[((size_t)n * 2 + 0) * C + c] = a;
            chansum[((size_t)n * 2 + 1) * C + c] = b;
            const float gm = __bfloat162float(gamma[c]);
            db = gm * a; ds = gm * b;
        }
    }
    s_db[threadIdx.x] = db; s_ds[threadIdx.x] = ds;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if (threadIdx.x < o) { s_db[threadIdx.x] += s_db[threadIdx.x + o]; s_ds[threadIdx.x] += s_ds[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        group_terms[((size_t)n * GN_GROUPS + g) * 2 + 0] = s_db[0];
        group_terms[((size_t)n * GN_GROUPS + g) * 2 + 1] = s_ds[0];
    }
}
// pass 2b: dgamma / dbeta = sum over images of the per-channel sums
__global__ void gn_bwd_param_kernel(const float* __restrict__ chansum, int NB, int C, __nv_bfloat16* __restrict__ dgamma,
                                    __nv_bfloat16* __restrict__ dbeta, int accumulate) {
    pdl_enter();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    float a = 0.f, b = 0.f;
    for (int n = 0; n < NB; ++n) { a += chansum[((size_t)n * 2 + 0) * C + c]; b += chansum[((size_t)n * 2 + 1) * C + c]; }
    if (accumulate) { a = round_bf16(a) + __bfloat162float(dbeta[c]); b = round_bf16(b) + __bfloat162float(dgamma[c]); }
    dbeta[c] = __float2bfloat16_rn(a);
    dgamma[c] = __float2bfloat16_rn(b);
}

// pass 3: dx = rstd * (dz*gamma - db/cnt - xhat * ds/cnt)
__global__ void __launch_bounds__(GN_THREADS)
gn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x,
                    const __nv_bfloat16* __restrict__ gamma, const __nv_bfloat16* __restrict__ beta,
                    const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ group_terms,
                    int HW, int C, int silu, const __nv_bfloat16* __restrict__ dres, __nv_bfloat16* __restrict__ dx) {
    pdl_enter();
    __shared__ float s_mean[GN_GROUPS], s_rstd[GN_GROUPS], s_db[GN_GROUPS], s_ds[GN_GROUPS];
    const int n = blockIdx.y;
    const int cpg = C / GN_GROUPS;
    if (threadIdx.x < GN_GROUPS) {
        const float inv = 1.0f / ((float)HW * (float)cpg);
        s_mean[threadIdx.x] = mean[n * GN_GROUPS + threadIdx.x];
        s_rstd[threadIdx.x] = rstd[n * GN_GROUPS + threadIdx.x];
        s_db[threadIdx.x] = group_terms[(n * GN_GROUPS + threadIdx.x) * 2 + 0] * inv;
        s_ds[threadIdx.x] = group_terms[(n * GN_GROUPS + threadIdx.x) * 2 + 1] * inv;
    }
    __syncthreads();
    const int vec_per_row = C / 8;
    const int cols = min(vec_per_row, (int)blockDim.x);
    const int row_lanes = (int)blockDim.x / cols;
    const int tc = threadIdx.x % cols, tr = threadIdx.x / cols;
    const int rows_per_chunk = (HW + gridDim.x - 1) / gridDim.x;
    const int r0 = blockIdx.x * rows_per_chunk, r1 = min(HW, r0 + rows_per_chunk);
    const size_t base = (size_t)n * HW * C;
    if (tr >= row_lanes) return;
    for (int v = tc; v < vec_per_row; v += cols) {             // column-owner loop, see gn_apply_kernel
        float gm[8], bt[8], mu[8], rs[8], gdb[8], gds[8];
        unpack8(*reinterpret_cast<const uint4*>(gamma + v * 8), gm);
        unpack8(*reinterpret_cast<const uint4*>(beta + v * 8), bt);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int g = (v * 8 + e) / cpg;
            mu[e] = s_mean[g]; rs[e] = s_rstd[g]; gdb[e] = s_db[g]; gds[e] = s_ds[g];
        }
        auto one = [&](const uint4& px, const uint4& pd, const uint4& pr, int r) {
            float fx[8], fd[8];
            unpack8(px, fx);
            unpack8(pd, fd);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float xh = (fx[e] - mu[e]) * rs[e];
                float dz = fd[e];
                if (silu) {
                    const float z = xh * gm[e] + bt[e];
                    const float sg = sigmoidf_(z);
                    dz *= sg * (1.0f + z * (1.0f - sg));
                }
                fx[e] = rs[e] * (dz * gm[e] - gdb[e] - xh * gds[e]);
            }
            if (dres) {
                float fr[8];
                unpack8(pr, fr);
#pragma unroll
                for (int e = 0; e < 8; e += 2) { round2_bf16(fx[e], fx[e + 1]); fx[e] += fr[e]; fx[e + 1] += fr[e + 1]; }
            }
            st_stream(dx + base + (size_t)r * C + v * 8, pack8(fx));
        };
        const uint4 zero4 = make_uint4(0, 0, 0, 0);
        int r = r0 + tr;
        for (; r + row_lanes < r1; r += 2 * row_lanes) {        // two rows (up to six 16-byte loads) in flight
            uint4 px[2], pd[2], pr[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const size_t off = base + (size_t)(r + u * row_lanes) * C + v * 8;
                px[u] = ld_stream(x + off);
                pd[u] = ld_stream(dy + off);
                pr[u] = dres ? ld_stream(dres + off) : zero4;
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) one(px[u], pd[u], pr[u], r + u * row_lanes);
        }
        for (; r < r1; r += row_lanes) {
            const size_t off = base + (size_t)r * C + v * 8;
            one(ld_stream(x + off), ld_stream(dy + off), dres ? ld_stream(dres + off) : zero4, r);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// GroupNorm, slab kernels: ONE launch, every element read from HBM once.
// When a (image, group) slab -- HW pixels x C/32 channels, 80 KB for 1280 channels at 32x32 -- fits in shared memory and the
// group's channel run is 16-byte aligned (C/32 a multiple of 8), one CTA per (group, image) pulls its slab in with cp.async
// (no registers held while ~10 copies per thread are in flight), computes the statistics and normalises out of shared memory.
// The two-kernel path above pays two dependent launches and an L2 re-read: 22 us against ~8 for 1280 channels at 32x32, where
// the tensor is 10 MB and everything is latency.  Backward keeps x and dy (two slabs) and adds the residual gradient on the way
// out.  Each thread only ever touches the vectors it copied itself, so cp.async.wait_all is the only ordering the slab needs.
// Deterministic: fixed thread -> element mapping, warp shuffles + fixed-order shared-memory sums.
__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void* g) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(smem_addr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// sum of (a, b) over the block, result in every thread; s_red: [32][2] floats
__device__ __forceinline__ void block_sum2(float& a, float& b, float (*s_red)[2]) {
    a = warp_sum(a); b = warp_sum(b);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    __syncthreads();                                   // s_red may still be read from a previous call
    if (lane == 0) { s_red[warp][0] = a; s_red[warp][1] = b; }
    __syncthreads();
    float ta = 0.f, tb = 0.f;
    for (int w = 0; w < nw; ++w) { ta += s_red[w][0]; tb += s_red[w][1]; }
    a = ta; b = tb;
}

__global__ void __launch_bounds__(GN_THREADS)
gn_slab_fwd_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ gamma,
                   const __nv_bfloat16* __restrict__ beta, int HW, int C, float eps, int silu, __nv_bfloat16* __restrict__ y,
                   float* __restrict__ mean_out, float* __restrict__ rstd_out) {
    pdl_enter();
    extern __shared__ __align__(16) uint8_t gn_slab[];          // [HW][vpg] 16-byte vectors
    __shared__ float s_red[32][2];
    const int g = blockIdx.x, n = blockIdx.y;
    const int cpg = C / GN_GROUPS, vpg = cpg >> 3;
    const int T = blockDim.x, L = T / vpg;                      // blockDim is a multiple of vpg: a thread's channel vector is fixed
    const int tc = threadIdx.x % vpg, r0 = threadIdx.x / vpg;
    const int nvec = HW * vpg;
    const __nv_bfloat16* xb = x + (size_t)n * HW * C + g * cpg + tc * 8;
    __nv_bfloat16* yb = y + (size_t)n * HW * C + g * cpg + tc * 8;
    const uint32_t sl = smem_u32(gn_slab);
    for (int idx = threadIdx.x, r = r0; idx < nvec; idx += T, r += L) cp_async16(sl + (uint32_t)idx * 16u, xb + (size_t)r * C);
    float gm[8], bt[8];
    unpack8(*reinterpret_cast<const uint4*>(gamma + g * cpg + tc * 8), gm);
    unpack8(*reinterpret_cast<const uint4*>(beta + g * cpg + tc * 8), bt);
    const float pivot = __bfloat162float(x[(size_t)n * HW * C + g * cpg]);     // sums of x - pivot: see gn_stats_kernel
    cp_async_wait_all();
    float s = 0.f, q = 0.f;
    for (int idx = threadIdx.x; idx < nvec; idx += T) {
        float f[8];
        unpack8(*reinterpret_cast<const uint4*>(gn_slab + (size_t)idx * 16), f);
#pragma unroll
        for (int e = 0; e < 8; ++e) { const float d = f[e] - pivot; s += d; q = fmaf(d, d, q); }
    }
    block_sum2(s, q, s_red);
    const float cnt = (float)HW * (float)cpg;
    const float dm = s / cnt;
    const float mean = pivot + dm;
    const float rstd = rsqrtf(fmaxf(q / cnt - dm * dm, 0.f) + eps);
    if (threadIdx.x == 0) { mean_out[n * GN_GROUPS + g] = mean; rstd_out[n * GN_GROUPS + g] = rstd; }
    float sc[8], sh[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { sc[e] = rstd * gm[e]; sh[e] = bt[e] - mean * sc[e]; }
    for (int idx = threadIdx.x, r = r0; idx < nvec; idx += T, r += L) {
        float f[8];
        unpack8(*reinterpret_cast<const uint4*>(gn_slab + (size_t)idx * 16), f);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            float z = fmaf(f[e], sc[e], sh[e]);
            if (silu) z = z * sigmoidf_(z);
            f[e] = z;
        }
        st_stream(yb + (size_t)r * C, pack8(f));
    }
}

// chansum [NB][2][C]: per-image, per-channel sums of dz and dz*xhat (dgamma / dbeta = their sum over images: gn_bwd_param_kernel)
__global__ void __launch_bounds__(GN_THREADS)
gn_slab_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x,
                   const __nv_bfloat16* __restrict__ gamma, const __nv_bfloat16* __restrict__ beta,
                   const float* __restrict__ mean, const float* __restrict__ rstd, int HW, int C, int silu,
                   const __nv_bfloat16* __restrict__ dres, __nv_bfloat16* __restrict__ dx, float* __restrict__ chansum) {
    pdl_enter();
    extern __shared__ __align__(16) uint8_t gn_slab[];          // x slab | dy slab | channel table [L][vpg][16] floats
    __shared__ float s_red[32][2];
    const int g = blockIdx.x, n = blockIdx.y;
    const int cpg = C / GN_GROUPS, vpg = cpg >> 3;
    const int T = blockDim.x, L = T / vpg;
    const int tc = threadIdx.x % vpg, r0 = threadIdx.x / vpg;
    const int nvec = HW * vpg;
    const size_t goff = (size_t)n * HW * C + g * cpg + tc * 8;
    const uint8_t* sx = gn_slab;
    const uint8_t* sd = gn_slab + (size_t)nvec * 16;
    float* table = reinterpret_cast<float*>(gn_slab + (size_t)nvec * 32);
    {
        const uint32_t ax = smem_u32(sx), ad = smem_u32(sd);
        for (int idx = threadIdx.x, r = r0; idx < nvec; idx += T, r += L) {
            cp_async16(ax + (uint32_t)idx * 16u, x + goff + (size_t)r * C);
            cp_async16(ad + (uint32_t)idx * 16u, dy + goff + (size_t)r * C);
        }
    }
    float gm[8], bt[8];
    unpack8(*reinterpret_cast<const uint4*>(gamma + g * cpg + tc * 8), gm);
    unpack8(*reinterpret_cast<const uint4*>(beta + g * cpg + tc * 8), bt);
    const float mu = mean[n * GN_GROUPS + g], rs = rstd[n * GN_GROUPS + g];
    cp_async_wait_all();
    float a[8], b[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { a[e] = 0.f; b[e] = 0.f; }
    for (int idx = threadIdx.x; idx < nvec; idx += T) {
        float fx[8], fd[8];
        unpack8(*reinterpret_cast<const uint4*>(sx + (size_t)idx * 16), fx);
        unpack8(*reinterpret_cast<const uint4*>(sd + (size_t)idx * 16), fd);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float xh = (fx[e] - mu) * rs;
            float dz = fd[e];
            if (silu) {
                const float z = xh * gm[e] + bt[e];
                const float sg = sigmoidf_(z);
                dz *= sg * (1.0f + z * (1.0f - sg));
            }
            a[e] += dz; b[e] = fmaf(dz, xh, b[e]);
        }
    }
    float db = 0.f, ds = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) { db = fmaf(gm[e], a[e], db); ds = fmaf(gm[e], b[e], ds); }
    if (threadIdx.x < L * vpg) {
        float* t = table + (size_t)threadIdx.x * 16;            // [row lane][channel vector][dz x 8 | dz*xhat x 8]
#pragma unroll
        for (int e = 0; e < 8; ++e) { t[e] = a[e]; t[8 + e] = b[e]; }
    }
    block_sum2(db, ds, s_red);                                   // its barriers also publish the table
    if (threadIdx.x < 2 * cpg) {                                 // per-channel sums over the row lanes, fixed order
        const int which = threadIdx.x / cpg, c = threadIdx.x - which * cpg;
        float t = 0.f;
        for (int l = 0; l < L; ++l) t += table[((size_t)l * vpg + (c >> 3)) * 16 + which * 8 + (c & 7)];
        chansum[((size_t)n * 2 + which) * C + g * cpg + c] = t;
    }
    const float inv = 1.0f / ((float)HW * (float)cpg);
    const float gdb = db * inv, gds = ds * inv;
    for (int idx = threadIdx.x, r = r0; idx < nvec; idx += T, r += L) {
        float fx[8], fd[8];
        unpack8(*reinterpret_cast<const uint4*>(sx + (size_t)idx * 16), fx);
        unpack8(*reinterpret_cast<const uint4*>(sd + (size_t)idx * 16), fd);
        uint4 pr = make_uint4(0, 0, 0, 0);
        if (dres) pr = ld_stream(dres + goff + (size_t)r * C);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float xh = (fx[e] - mu) * rs;
            float dz = fd[e];
            if (silu) {
                const float z = xh * gm[e] + bt[e];
                const float sg = sigmoidf_(z);
                dz *= sg * (1.0f + z * (1.0f - sg));
            }
            fx[e] = rs * (dz * gm[e] - gdb - xh * gds);
        }
        if (dres) {
            float fr[8];
            unpack8(pr, fr);
#pragma unroll
            for (int e = 0; e < 8; e += 2) { round2_bf16(fx[e], fx[e + 1]); fx[e] += fr[e]; fx[e + 1] += fr[e + 1]; }
        }
        st_stream(dx + goff + (size_t)r * C, pack8(fx));
    }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm, C % 8 == 0, C <= 2048
// ---------------------------------------------------------------------------------------------
// forward : one warp per R consecutive rows.  Every 16-byte load of the R rows is issued before the first reduction, so a
//           warp's whole life is ONE memory round trip (the old one-row-at-a-time loop was a chain of 2..7 of them and
//           ran at ~2.4 TB/s); x stays packed in registers between the mean, variance and output passes.
// backward: "column owner" layout.  A thread owns ONE 8-channel vector column and T rows of a tile, so the dgamma / dbeta
//           accumulators are 16 registers per thread (the warp-per-row kernel needed 2*C/32 = 80 and fit one row in flight per
//           warp); the two per-row sums cross the block through warp shuffles + a small shared-memory table.
constexpr int LN_MAXV = 8;     // vectors of 8 per lane -> C <= 2048
constexpr int LN_FWD_WARPS = 4;

template <int VPL, int R>
__global__ void __launch_bounds__(LN_FWD_WARPS * 32, (VPL <= 5 ? 4 : 2))       // <= 128 registers for the SDXL widths (640, 1280)
ln_fwd_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ gamma,
              const __nv_bfloat16* __restrict__ beta, long long rows, int C, float eps, __nv_bfloat16* __restrict__ y,
              float* __restrict__ mean_out, float* __restrict__ rstd_out) {
    pdl_enter();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nv = C / 8;
    const float inv_c = 1.0f / (float)C;
    const long long stride = (long long)gridDim.x * LN_FWD_WARPS * R;
    for (long long r0 = ((long long)blockIdx.x * LN_FWD_WARPS + warp) * R; r0 < rows; r0 += stride) {
        float f[R][VPL][8];
        {
            uint4 xp[R][VPL];
#pragma unroll
            for (int j = 0; j < R; ++j)
#pragma unroll
                for (int i = 0; i < VPL; ++i) {
                    const int v = lane + 32 * i;
                    xp[j][i] = (v < nv && r0 + j < rows) ? ld_stream(x + (r0 + j) * C + v * 8) : make_uint4(0, 0, 0, 0);
                }
#pragma unroll
            for (int j = 0; j < R; ++j)
#pragma unroll
                for (int i = 0; i < VPL; ++i) unpack8(xp[j][i], f[j][i]);
        }
        float mean[R], rstd[R];
#pragma unroll
        for (int j = 0; j < R; ++j) {
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < VPL; ++i)
#pragma unroll
                for (int e = 0; e < 8; ++e) s += f[j][i][e];
            mean[j] = s;
        }
#pragma unroll
        for (int j = 0; j < R; ++j) mean[j] = warp_sum(mean[j]) * inv_c;
#pragma unroll
        for (int j = 0; j < R; ++j) {
            float q = 0.f;
#pragma unroll
            for (int i = 0; i < VPL; ++i) {
                if (lane + 32 * i < nv) {                       // padding lanes hold zeros, not (0 - mean)
#pragma unroll
                    for (int e = 0; e < 8; ++e) { const float d = f[j][i][e] - mean[j]; q = fmaf(d, d, q); }
                }
            }
            rstd[j] = q;
        }
#pragma unroll
        for (int j = 0; j < R; ++j) rstd[j] = rsqrtf(warp_sum(rstd[j]) * inv_c + eps);
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
            const int v = lane + 32 * i;
            if (v < nv) {
                float gm[8], bt[8];                              // L1-resident after the first warp touched them
                unpack8(__ldg(reinterpret_cast<const uint4*>(gamma + v * 8)), gm);
                unpack8(__ldg(reinterpret_cast<const uint4*>(beta + v * 8)), bt);
#pragma unroll
                for (int j = 0; j < R; ++j) {
                    if (r0 + j < rows) {
                        float o[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) o[e] = (f[j][i][e] - mean[j]) * rstd[j] * gm[e] + bt[e];
                        st_stream(y + (r0 + j) * C + v * 8, pack8(o));
                    }
                }
            }
        }
        if (lane < R && r0 + lane < rows) {
            float m = mean[0], rsd = rstd[0];
#pragma unroll
            for (int j = 1; j < R; ++j) if (lane == j) { m = mean[j]; rsd = rstd[j]; }
            mean_out[r0 + lane] = m; rstd_out[r0 + lane] = rsd;
        }
    }
}

// backward.  blockDim = cols_pad * RL: cols_pad = vector columns rounded up to a warp multiple (a warp never straddles two
// row lanes), RL row lanes.  A tile is RL*T consecutive rows = ONE contiguous range of x, dy and the residual gradient, so a
// tile is fetched by three 1-D TMA bulk copies (cp.async.bulk, <= 32 KB each) into a two-deep shared-memory ring, completion
// on an mbarrier: the next tile streams in while this one is reduced, and no fetched row is held in registers.
// Thread (tc, rl) takes rows base + t*RL + rl.  Per tile: per-row partial sums of the thread's 8 channels -> warp_sum ->
// red[row][warp-in-lane][2] -> barrier -> every thread adds the cols_pad/32 entries of its rows in fixed order
// (deterministic) -> dx.  dgamma / dbeta: 16 accumulators per thread, combined over the row lanes through shared memory at
// the end -> partial [gridDim.x][2][C].
constexpr int LNB_T = 4;                   // the reduce-scatter below is written for exactly 2 x 4 values
constexpr int LNB_MAX_THREADS = 512;

__global__ void __launch_bounds__(LNB_MAX_THREADS, 1)
ln_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x,
              const __nv_bfloat16* __restrict__ gamma, const float* __restrict__ mean, const float* __restrict__ rstd,
              long long rows, int C, const __nv_bfloat16* __restrict__ dres, __nv_bfloat16* __restrict__ dx,
              float* __restrict__ partial, int cols_pad, int RL, long long rows_per_block, int want_col) {
    // want_col: also the column sums of dx (as stored, bf16-rounded) -> third row of the partials.  dx of a pre-LN transformer
    // sublayer is the gradient of the PREVIOUS Linear's output (to_out / ff.net.2 / proj_in), so this is that layer's bias
    // gradient, free of the separate column-sum launch that re-read dx (210 launches per step).
    pdl_enter();
    extern __shared__ __align__(128) uint8_t lnb_smem[];
    const int ncomp = want_col ? 3 : 2;
    const int tc = threadIdx.x % cols_pad, rl = threadIdx.x / cols_pad;
    const int lane = threadIdx.x & 31, wcol = tc >> 5, W = cols_pad >> 5;
    const int nv = C / 8;
    const bool active = tc < nv;
    const float inv_c = 1.0f / (float)C;
    const int tile_rows = RL * LNB_T;
    const uint32_t tensor_bytes = (uint32_t)tile_rows * (uint32_t)C * 2u;      // one tensor's rows of a tile
    uint8_t* ring = lnb_smem;                                                  // [2 slots][x | dy | dres][tensor_bytes]
    float* red = reinterpret_cast<float*>(lnb_smem + 6 * (size_t)tensor_bytes);   // [tile_rows][W][2]
    uint64_t* bars = reinterpret_cast<uint64_t*>(red + (size_t)tile_rows * W * 2);
    // The kernel is issue-bound, not HBM-bound (15 warps, ~1000 issued instructions per thread and 12-row tile before this form):
    // all per-element arithmetic runs as packed fp32x2 instructions on element pairs (2e, 2e+1).
    float2 gm[4], ag[4], ab[4], ac[4];
    {
        const uint4 g4 = active ? *reinterpret_cast<const uint4*>(gamma + tc * 8) : make_uint4(0, 0, 0, 0);
        unpack8v(g4, gm);
#pragma unroll
        for (int e = 0; e < 4; ++e) { ag[e] = make_float2(0.f, 0.f); ab[e] = ag[e]; ac[e] = ag[e]; }
    }
    const long long rb0 = (long long)blockIdx.x * rows_per_block;
    const long long rb1 = rb0 + rows_per_block < rows ? rb0 + rows_per_block : rows;
    const int ntiles = rb1 > rb0 ? (int)((rb1 - rb0 + tile_rows - 1) / tile_rows) : 0;
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1); mbar_init(&bars[1], 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto issue = [&](int i) {                                   // one thread: arm the slot's barrier, start the three copies
        const long long base = rb0 + (long long)i * tile_rows;
        const long long left = rb1 - base;
        const uint32_t bytes = (uint32_t)(left < tile_rows ? left : tile_rows) * (uint32_t)C * 2u;
        uint8_t* slot = ring + (size_t)(i & 1) * 3 * tensor_bytes;
        mbar_arrive_expect_tx(&bars[i & 1], bytes * (dres ? 3u : 2u));
        bulk_load_1d(slot, x + base * C, bytes, &bars[i & 1]);
        bulk_load_1d(slot + tensor_bytes, dy + base * C, bytes, &bars[i & 1]);
        if (dres) bulk_load_1d(slot + 2 * (size_t)tensor_bytes, dres + base * C, bytes, &bars[i & 1]);
    };
    if (threadIdx.x == 0) {
        if (ntiles > 0) issue(0);
        if (ntiles > 1) issue(1);
    }
    for (int i = 0; i < ntiles; ++i) {
        const long long base = rb0 + (long long)i * tile_rows;
        const uint8_t* slot = ring + (size_t)(i & 1) * 3 * tensor_bytes;
        float mu[LNB_T], rs[LNB_T], p1[LNB_T], p2[LNB_T];
        bool ok[LNB_T];
#pragma unroll
        for (int t = 0; t < LNB_T; ++t) {
            const long long row = base + (long long)t * RL + rl;
            ok[t] = active && row < rb1;
            mu[t] = ok[t] ? __ldg(mean + row) : 0.f;
            rs[t] = ok[t] ? __ldg(rstd + row) : 0.f;
        }
        mbar_wait(&bars[i & 1], (uint32_t)((i >> 1) & 1));
#pragma unroll
        for (int t = 0; t < LNB_T; ++t) {
            float2 a = make_float2(0.f, 0.f), b = a;
            if (ok[t]) {
                const size_t off = ((size_t)(t * RL + rl) * C + (size_t)tc * 8) * 2;
                float2 fx[4], fd[4];
                unpack8v(*reinterpret_cast<const uint4*>(slot + off), fx);
                unpack8v(*reinterpret_cast<const uint4*>(slot + tensor_bytes + off), fd);
                const float2 nmu = make_float2(-mu[t], -mu[t]), rs2 = make_float2(rs[t], rs[t]);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float2 xh = __fmul2_rn(__fadd2_rn(fx[e], nmu), rs2);
                    const float2 dg = __fmul2_rn(fd[e], gm[e]);
                    a = __fadd2_rn(a, dg);
                    b = __ffma2_rn(dg, xh, b);
                    ag[e] = __ffma2_rn(fd[e], xh, ag[e]);
                    ab[e] = __fadd2_rn(ab[e], fd[e]);
                }
            }
            p1[t] = a.x + a.y; p2[t] = b.x + b.y;
        }
        // eight warp sums as a reduce-scatter (9 shuffles instead of 8 x 5): after the xor-16 / 8 / 4 steps every lane owns ONE
        // of the eight values, two plain butterfly steps finish it.  Value v = which * 4 + t ends up in the lanes whose bits
        // 4..2 spell v; fixed exchange pattern = fixed summation order.
        {
            const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
            float w4[4], w2[2];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float lo = p1[k], hi = p2[k];
                w4[k] = (b4 ? hi : lo) + __shfl_xor_sync(0xffffffffu, b4 ? lo : hi, 16);
            }
#pragma unroll
            for (int k = 0; k < 2; ++k) w2[k] = (b3 ? w4[k + 2] : w4[k]) + __shfl_xor_sync(0xffffffffu, b3 ? w4[k] : w4[k + 2], 8);
            float z = (b2 ? w2[1] : w2[0]) + __shfl_xor_sync(0xffffffffu, b2 ? w2[0] : w2[1], 4);
            z += __shfl_xor_sync(0xffffffffu, z, 2);
            z += __shfl_xor_sync(0xffffffffu, z, 1);
            if ((lane & 3) == 0) {
                const int v = lane >> 2, which = v >> 2, t = v & 3;
                red[((size_t)(rl * LNB_T + t) * W + wcol) * 2 + which] = z;
            }
        }
        __syncthreads();
#pragma unroll
        for (int t = 0; t < LNB_T; ++t) {
            if (!ok[t]) continue;
            const float2* srow = reinterpret_cast<const float2*>(red + (size_t)(rl * LNB_T + t) * W * 2);
            float s1 = 0.f, s2 = 0.f;
            for (int w = 0; w < W; ++w) { const float2 v = srow[w]; s1 += v.x; s2 += v.y; }
            s1 *= inv_c; s2 *= inv_c;
            const size_t off = ((size_t)(t * RL + rl) * C + (size_t)tc * 8) * 2;
            float2 fx[4], fd[4], o[4];
            unpack8v(*reinterpret_cast<const uint4*>(slot + off), fx);
            unpack8v(*reinterpret_cast<const uint4*>(slot + tensor_bytes + off), fd);
            const float2 nmu = make_float2(-mu[t], -mu[t]), rs2 = make_float2(rs[t], rs[t]);
            const float2 ns1 = make_float2(-s1, -s1), ns2 = make_float2(-s2, -s2);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 xh = __fmul2_rn(__fadd2_rn(fx[e], nmu), rs2);
                // rstd * (dy*gamma - s1 - xhat*s2)
                o[e] = __fmul2_rn(rs2, __ffma2_rn(xh, ns2, __fadd2_rn(__fmul2_rn(fd[e], gm[e]), ns1)));
            }
            if (dres) {
                float2 fr[4];
                unpack8v(*reinterpret_cast<const uint4*>(slot + 2 * (size_t)tensor_bytes + off), fr);
#pragma unroll
                for (int e = 0; e < 4; ++e) { round2_bf16(o[e].x, o[e].y); o[e] = __fadd2_rn(o[e], fr[e]); }
            }
            // the stored (bf16-rounded) dx: one packed conversion serves the store and the column sums
            const uint4 o4 = make_uint4(pack_bf16(o[0].x, o[0].y), pack_bf16(o[1].x, o[1].y), pack_bf16(o[2].x, o[2].y), pack_bf16(o[3].x, o[3].y));
            if (want_col) {
                float2 orr[4];
                unpack8v(o4, orr);
#pragma unroll
                for (int e = 0; e < 4; ++e) ac[e] = __fadd2_rn(ac[e], orr[e]);
            }
            const long long row = base + (long long)t * RL + rl;
            st_stream(dx + row * C + tc * 8, o4);
        }
        __syncthreads();               // slot and table are free: refill the slot with the tile after next
        if (threadIdx.x == 0 && i + 2 < ntiles) issue(i + 2);
    }
    // accumulators -> [RL][ncomp][C] (over the idle ring) -> fixed-order sum over the row lanes -> this block's partial row
    float* fin = reinterpret_cast<float*>(lnb_smem);
    if (active) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            *reinterpret_cast<float2*>(&fin[(size_t)(rl * ncomp + 0) * C + tc * 8 + 2 * e]) = ag[e];
            *reinterpret_cast<float2*>(&fin[(size_t)(rl * ncomp + 1) * C + tc * 8 + 2 * e]) = ab[e];
            if (want_col) *reinterpret_cast<float2*>(&fin[(size_t)(rl * ncomp + 2) * C + tc * 8 + 2 * e]) = ac[e];
        }
    }
    __syncthreads();
    float* out = partial + (size_t)blockIdx.x * ncomp * C;
    for (int i = threadIdx.x; i < ncomp * C; i += blockDim.x) {
        float a = 0.f;
        for (int l = 0; l < RL; ++l) a += fin[(size_t)l * ncomp * C + i];
        out[i] = a;
    }
}

// reduce [blocks][ncomp][C] -> dgamma (first C), dbeta (second C) and, with ncomp == 3, the column sums of dx (third C)
// block = 32 columns x 32 row lanes: lane (cx, ry) sums partial rows ry, ry+32, ... of its column (a warp reads 128
// contiguous bytes per row), then the 32 row lanes are combined through shared memory in fixed order
__global__ void __launch_bounds__(1024)
ln_bwd_finalize_kernel(const float* __restrict__ partial, int blocks, int C, __nv_bfloat16* __restrict__ dgamma,
                       __nv_bfloat16* __restrict__ dbeta, int accumulate, __nv_bfloat16* __restrict__ dcol, int ncomp, int skip_params) {
    pdl_enter();
    __shared__ float sm[32][33];
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + cx;
    float s = 0.f;
    if (i < ncomp * C)
        for (int b = ry; b < blocks; b += 32) s += partial[(size_t)b * ncomp * C + i];
    sm[ry][cx] = s;
    __syncthreads();
    if (ry == 0 && i < ncomp * C) {
        if (skip_params && i < 2 * C) return;                 // frozen LayerNorm: only the column sums are wanted
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 32; ++k) t += sm[k][cx];
        __nv_bfloat16* dst = i < C ? dgamma + i : (i < 2 * C ? dbeta + (i - C) : dcol + (i - 2 * C));
        if (accumulate && i < 2 * C) t = round_bf16(t) + __bfloat162float(*dst);
        *dst = __float2bfloat16_rn(t);
    }
}

}  // namespace aoz

using namespace aoz;

template <int VPL, int R>
static int launch_ln_fwd(const void* x, const void* gamma, const void* beta, long long rows, int C, float eps, void* y, void* mean,
                         void* rstd, cudaStream_t s) {
    const long long warps = (rows + R - 1) / R;
    long long blocks = (warps + LN_FWD_WARPS - 1) / LN_FWD_WARPS;
    if (blocks > sm_count() * 12) blocks = sm_count() * 12;
    launch_k(ln_fwd_kernel<VPL, R>, dim3((int)blocks), dim3(LN_FWD_WARPS * 32), (size_t)(0), s, (const __nv_bfloat16*)x,
             (const __nv_bfloat16*)gamma, (const __nv_bfloat16*)beta, rows, C, eps, (__nv_bfloat16*)y, (float*)mean, (float*)rstd);
    AOZ_CHECK_LAUNCH("ln_fwd_kernel");
    return AOZ_OK;
}

extern "C" {

static int g_gn_slab = 1;                                      // 0: always the multi-kernel path (A/B runs, aoz_groupnorm_set_slab)
constexpr size_t GN_SLAB_MAX_BYTES = 200 * 1024;

// block shape: one thread per 16-byte vector column (C/8 of them) times as many row lanes as fit `max_threads`
static int gn_block_threads(int C, int* row_lanes_out = nullptr, int* cols_out = nullptr, int max_threads = GN_THREADS) {
    const int vec = C / 8;
    const int cols = vec < max_threads ? vec : max_threads;
    const int row_lanes = max_threads / cols;
    if (row_lanes_out) *row_lanes_out = row_lanes;
    if (cols_out) *cols_out = cols;
    return cols * row_lanes;
}

// pixel chunks (grid.x) of the statistics kernels: one block per SM over the whole batch (fewer partials to combine, every
// load of the tensor in flight at once), at least four rows per thread
static int gn_chunks(int NB, int HW, int row_lanes, int max_chunks) {
    int chunks = sm_count() / NB;
    const int by_rows = HW / (row_lanes * 4);
    if (chunks > by_rows) chunks = by_rows;
    if (chunks > max_chunks) chunks = max_chunks;
    if (chunks < 1) chunks = 1;
    return chunks;
}

// pixel chunks (grid.x) of the apply kernels: enough blocks to fill the GPU a few times over, at least 8 rows per thread
static int gn_apply_chunks(int NB, int HW, int C) {
    int row_lanes = 1;
    gn_block_threads(C, &row_lanes);
    int chunks = (HW + row_lanes * 8 - 1) / (row_lanes * 8);
    const int cap = (sm_count() * 6 + NB - 1) / NB;
    if (chunks > cap) chunks = cap;
    if (chunks < 1) chunks = 1;
    return chunks;
}

// experiment switch: 1 = slab kernels where they apply (default), 0 = always the multi-kernel path
int aoz_groupnorm_set_slab(int on) { g_gn_slab = on ? 1 : 0; return AOZ_OK; }

// workspace floats needed by the GroupNorm forward / backward (upper bound)
long long aoz_groupnorm_workspace_floats(int NB, int HW, int C) {
    const long long chunks = GN_MAX_CHUNKS;
    const long long bwd = (long long)NB * chunks * 2 * C + (long long)NB * GN_GROUPS * 2 + 64 + (long long)NB * 2 * C + 64;
    const long long fwd = (long long)NB * GN_FWD_MAX_CHUNKS * GN_GROUPS * 2;
    return bwd > fwd ? bwd : fwd;
}

// y = silu?(GroupNorm32(x)); x, y: [NB, HW, C] bf16 channels-last; mean/rstd out: [NB, 32] fp32
int aoz_groupnorm_fwd(const void* x, const void* gamma, const void* beta, int NB, int HW, int C, float eps, int silu,
                      void* y, void* mean, void* rstd, void* workspace, void* stream) {
    AOZ_CHECK_ARG(x && gamma && beta && y && mean && rstd && workspace, "aoz_groupnorm_fwd: null pointer");
    AOZ_CHECK_ARG(C % GN_GROUPS == 0 && C % 8 == 0, "aoz_groupnorm_fwd: C=%d must be a multiple of 32", C);
    AOZ_CHECK_ARG(NB > 0 && HW > 0, "aoz_groupnorm_fwd: empty input");
    AOZ_CHECK_ARG(C <= 16384, "aoz_groupnorm_fwd: C=%d too large", C);
    cudaStream_t s = (cudaStream_t)stream;
    {   // slab path: one launch, one HBM read (see gn_slab_fwd_kernel)
        const int cpg = C / GN_GROUPS;
        const size_t slab = (size_t)HW * cpg * 2;
        if (g_gn_slab && (cpg % 8) == 0 && slab <= GN_SLAB_MAX_BYTES && (cpg >> 3) <= GN_THREADS) {
            const int vpg = cpg >> 3, threads = (GN_THREADS / vpg) * vpg;
            static size_t attr = 48 * 1024;
            if (slab > attr) { cudaFuncSetAttribute(gn_slab_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)slab); attr = slab; }
            launch_k(gn_slab_fwd_kernel, dim3(GN_GROUPS, NB), dim3(threads), slab, s, (const __nv_bfloat16*)x, (const __nv_bfloat16*)gamma,
                     (const __nv_bfloat16*)beta, HW, C, eps, silu, (__nv_bfloat16*)y, (float*)mean, (float*)rstd);
            AOZ_CHECK_LAUNCH("gn_slab_fwd_kernel");
            return AOZ_OK;
        }
    }
    int cols = 1, row_lanes = 1;
    const int st_threads = (gn_block_threads(C, &row_lanes, &cols, 1024) + 31) & ~31;
    const int chunks = gn_chunks(NB, HW, row_lanes, GN_FWD_MAX_CHUNKS);
    const int threads = gn_block_threads(C);
    AOZ_CHECK_ARG(NB <= 1024, "aoz_groupnorm_fwd: NB=%d > 1024", NB);
    const size_t st_smem = (size_t)row_lanes * 2 * C * sizeof(float);
    static size_t st_attr = 48 * 1024;
    if (st_smem > st_attr) {
        cudaFuncSetAttribute(gn_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)st_smem);
        st_attr = st_smem;
    }
    launch_k(gn_stats_kernel, dim3(chunks, NB), dim3(st_threads), st_smem, s, (const __nv_bfloat16*)x, HW, C, eps, cols, row_lanes,
             (float*)workspace, (float*)mean, (float*)rstd);
    AOZ_CHECK_LAUNCH("gn_stats_kernel");
    int gx = gn_apply_chunks(NB, HW, C);
    launch_k(gn_apply_kernel, dim3(gx, NB), dim3(threads), (size_t)(0), s, (const __nv_bfloat16*)x, (const __nv_bfloat16*)gamma,
             (const __nv_bfloat16*)beta, (const float*)mean, (const float*)rstd, HW, C, silu, (__nv_bfloat16*)y);
    AOZ_CHECK_LAUNCH("gn_apply_kernel");
    return AOZ_OK;
}

int aoz_groupnorm_bwd(const void* dy, const void* x, const void* gamma, const void* beta, const void* mean, const void* rstd,
                      int NB, int HW, int C, int silu, const void* dres, void* dx, void* dgamma, void* dbeta, int accumulate,
                      void* workspace, void* stream) {
    AOZ_CHECK_ARG(dy && x && gamma && beta && mean && rstd && dx && workspace, "aoz_groupnorm_bwd: null pointer");
    AOZ_CHECK_ARG(C % GN_GROUPS == 0 && C % 8 == 0, "aoz_groupnorm_bwd: C=%d must be a multiple of 32", C);
    cudaStream_t s = (cudaStream_t)stream;
    {   // slab path: x and dy slabs + the per-channel table in shared memory, one launch (+ the tiny dgamma / dbeta kernel)
        const int cpg = C / GN_GROUPS;
        if (g_gn_slab && (cpg % 8) == 0 && (cpg >> 3) <= GN_THREADS && 2 * cpg <= (GN_THREADS / (cpg >> 3)) * (cpg >> 3)) {
            const int vpg = cpg >> 3, threads = (GN_THREADS / vpg) * vpg;
            const size_t smem = (size_t)HW * cpg * 4 + (size_t)threads * 16 * sizeof(float);
            if (smem <= GN_SLAB_MAX_BYTES) {
                static size_t attr = 48 * 1024;
                if (smem > attr) { cudaFuncSetAttribute(gn_slab_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr = smem; }
                float* chansum = (float*)workspace;
                launch_k(gn_slab_bwd_kernel, dim3(GN_GROUPS, NB), dim3(threads), smem, s, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x,
                         (const __nv_bfloat16*)gamma, (const __nv_bfloat16*)beta, (const float*)mean, (const float*)rstd, HW, C, silu,
                         (const __nv_bfloat16*)dres, (__nv_bfloat16*)dx, chansum);
                AOZ_CHECK_LAUNCH("gn_slab_bwd_kernel");
                if (dgamma) {
                    launch_k(gn_bwd_param_kernel, dim3((C + 255) / 256), dim3(256), (size_t)(0), s, (const float*)chansum, NB, C,
                             (__nv_bfloat16*)dgamma, (__nv_bfloat16*)dbeta, accumulate);
                    AOZ_CHECK_LAUNCH("gn_bwd_param_kernel");
                }
                return AOZ_OK;
            }
        }
    }
    int cols = 1, row_lanes = 1;
    const int threads = gn_block_threads(C, &row_lanes, &cols);
    const int st_threads = (threads + 31) & ~31;
    const int chunks = gn_chunks(NB, HW, row_lanes, GN_MAX_CHUNKS);
    float* partial = (float*)workspace;
    float* group_terms = partial + (size_t)NB * GN_MAX_CHUNKS * 2 * C;
    const size_t st_smem = (size_t)row_lanes * 2 * C * sizeof(float);
    static size_t st_attr = 48 * 1024;
    if (st_smem > st_attr) {
        cudaFuncSetAttribute(gn_bwd_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)st_smem);
        st_attr = st_smem;
    }
    launch_k(gn_bwd_stats_kernel, dim3(chunks, NB), dim3(st_threads), st_smem, s,
        (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, (const __nv_bfloat16*)gamma, (const __nv_bfloat16*)beta,
        (const float*)mean, (const float*)rstd, HW, C, silu, cols, row_lanes, partial);
    AOZ_CHECK_LAUNCH("gn_bwd_stats_kernel");
    float* chansum = group_terms + (size_t)NB * GN_GROUPS * 2 + 64;
    launch_k(gn_bwd_group_kernel, dim3(GN_GROUPS, NB), dim3(128), (size_t)(0), s, partial, (const __nv_bfloat16*)gamma, chunks, C, chansum, group_terms);
    AOZ_CHECK_LAUNCH("gn_bwd_group_kernel");
    if (dgamma) {
        launch_k(gn_bwd_param_kernel, dim3((C + 255) / 256), dim3(256), (size_t)(0), s, chansum, NB, C, (__nv_bfloat16*)dgamma, (__nv_bfloat16*)dbeta, accumulate);
        AOZ_CHECK_LAUNCH("gn_bwd_param_kernel");
    }
    int gx = gn_apply_chunks(NB, HW, C);
    launch_k(gn_bwd_apply_kernel, dim3(gx, NB), dim3(threads), (size_t)(0), s, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, (const __nv_bfloat16*)gamma,
                                                           (const __nv_bfloat16*)beta, (const float*)mean, (const float*)rstd,
                                                           group_terms, HW, C, silu, (const __nv_bfloat16*)dres, (__nv_bfloat16*)dx);
    AOZ_CHECK_LAUNCH("gn_bwd_apply_kernel");
    return AOZ_OK;
}

int aoz_layernorm_fwd(const void* x, const void* gamma, const void* beta, long long rows, int C, float eps, void* y, void* mean,
                      void* rstd, void* stream) {
    AOZ_CHECK_ARG(x && gamma && beta && y && mean && rstd, "aoz_layernorm_fwd: null pointer");
    AOZ_CHECK_ARG(C % 8 == 0 && C <= LN_MAXV * 256, "aoz_layernorm_fwd: C=%d unsupported (multiple of 8, <= 2048)", C);
    if (rows <= 0) return AOZ_OK;
    cudaStream_t s = (cudaStream_t)stream;
    switch ((C / 8 + 31) / 32) {            // 16-byte vectors per lane; fewer vectors -> more rows in flight per warp
        case 1: return launch_ln_fwd<1, 4>(x, gamma, beta, rows, C, eps, y, mean, rstd, s);
        case 2: return launch_ln_fwd<2, 4>(x, gamma, beta, rows, C, eps, y, mean, rstd, s);
        case 3: return launch_ln_fwd<3, 3>(x, gamma, beta, rows, C, eps, y, mean, rstd, s);
        case 4: return launch_ln_fwd<4, 2>(x, gamma, beta, rows, C, eps, y, mean, rstd, s);
        case 5: return launch_ln_fwd<5, 2>(x, gamma, beta, rows, C, eps, y, mean, rstd, s);
        case 6: return launch_ln_fwd<6, 1>(x, gamma, beta, rows, C, eps, y, mean, rstd, s);
        case 7: return launch_ln_fwd<7, 1>(x, gamma, beta, rows, C, eps, y, mean, rstd, s);
        default: return launch_ln_fwd<8, 1>(x, gamma, beta, rows, C, eps, y, mean, rstd, s);
    }
}

long long aoz_layernorm_bwd_workspace_floats(int C) { return (long long)sm_count() * 2 * 2 * C; }

int aoz_layernorm_bwd_colsum(const void* dy, const void* x, const void* gamma, const void* mean, const void* rstd, long long rows, int C,
                             const void* dres, void* dx, void* dgamma, void* dbeta, int accumulate, void* dcolsum, void* workspace,
                             void* stream);

int aoz_layernorm_bwd(const void* dy, const void* x, const void* gamma, const void* mean, const void* rstd, long long rows, int C,
                      const void* dres, void* dx, void* dgamma, void* dbeta, int accumulate, void* workspace, void* stream) {
    return aoz_layernorm_bwd_colsum(dy, x, gamma, mean, rstd, rows, C, dres, dx, dgamma, dbeta, accumulate, nullptr, workspace, stream);
}

// The same with dcolsum != null: additionally dcolsum[c] = sum over rows of dx[r, c] (the stored, bf16-rounded dx), i.e. the bias
// gradient of the Linear whose output this LayerNorm's input is (to_out / ff.net.2 / proj_in of a pre-LN transformer block).
int aoz_layernorm_bwd_colsum(const void* dy, const void* x, const void* gamma, const void* mean, const void* rstd, long long rows, int C,
                             const void* dres, void* dx, void* dgamma, void* dbeta, int accumulate, void* dcolsum, void* workspace,
                             void* stream) {
    AOZ_CHECK_ARG(dy && x && gamma && mean && rstd && dx && dgamma && dbeta && workspace, "aoz_layernorm_bwd: null pointer");
    AOZ_CHECK_ARG(C % 8 == 0 && C <= LN_MAXV * 256, "aoz_layernorm_bwd: C=%d unsupported", C);
    AOZ_CHECK_ARG(((((uintptr_t)dy) | ((uintptr_t)x) | ((uintptr_t)dres) | ((uintptr_t)dx)) & 15) == 0,
                  "aoz_layernorm_bwd: dy / x / dres / dx must be 16-byte aligned (TMA bulk copies, 16-byte stores)");
    if (rows <= 0) return AOZ_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const int cols_pad = ((C / 8 + 31) / 32) * 32;
    int RL = LNB_MAX_THREADS / cols_pad;
    if (RL > 16) RL = 16;
    const int tile = RL * LNB_T;
    long long blocks = (rows + tile - 1) / tile;
    if (blocks > sm_count()) blocks = sm_count();
    const long long rows_per_block = (rows + blocks - 1) / blocks;
    blocks = (rows + rows_per_block - 1) / rows_per_block;
    // ring: 2 slots x (x, dy, dres) x tile rows; + the row-sum table + 2 mbarriers.  The final [RL][2][C] fp32 staging reuses the ring
    // (RL*2*C*4 = tile bytes of two tensors).
    const size_t smem = 6 * (size_t)tile * C * 2 + (size_t)tile * (cols_pad / 32) * 2 * sizeof(float) + 16;
    static size_t attr = 48 * 1024;
    if (smem > attr) {
        cudaFuncSetAttribute(ln_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr = smem;
    }
    launch_k(ln_bwd_kernel, dim3((int)blocks), dim3(cols_pad * RL), smem, s, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x,
             (const __nv_bfloat16*)gamma, (const float*)mean, (const float*)rstd, rows, C, (const __nv_bfloat16*)dres,
             (__nv_bfloat16*)dx, (float*)workspace, cols_pad, RL, rows_per_block, dcolsum != nullptr ? 1 : 0);
    AOZ_CHECK_LAUNCH("ln_bwd_kernel");
    const int ncomp = dcolsum != nullptr ? 3 : 2;
    launch_k(ln_bwd_finalize_kernel, dim3((ncomp * C + 31) / 32), dim3(1024), (size_t)(0), s, (const float*)workspace, (int)blocks, C,
             (__nv_bfloat16*)dgamma, (__nv_bfloat16*)dbeta, accumulate, (__nv_bfloat16*)dcolsum, ncomp, 0);
    AOZ_CHECK_LAUNCH("ln_bwd_finalize_kernel");
    return AOZ_OK;
}

}  // extern "C"
