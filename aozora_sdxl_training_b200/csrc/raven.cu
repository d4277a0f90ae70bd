// Multi-tensor Raven/Titan AdamW update, gradient sum-of-squares and clip coefficient (sm_100a).
//
// Replaces the per-tensor loop of RavenAdamW.step (reference training_utils/optimizers/raven.py:89-149;
// TitanAdamW titan.py:237-296 has identical math) and torch.nn.utils.clip_grad_norm_ as train.py:2772-2781
// calls it.  The reference streams CPU-resident moments through a 3 x max_numel fp32 scratch with ~15 ATen
// launches + 5 copies per tensor; here the moments live in HBM and ONE launch updates every tensor:
// read p, g, m, v once, write p, m, v once (14 B/param with bf16 state, 28 B/param all-fp32).
//
// Work is cut into fixed chunks of CHUNK elements; chunk c belongs to tensor chunk_tensor[c] and the chunks
// of one tensor are consecutive (chunk_start[t] .. chunk_start[t+1]).  Pure HBM streaming: the update moves its
// operands by bulk copies through shared memory, the gradient norm by 128-bit L1-bypassing loads.
#include "common.cuh"
#include <cuda_fp16.h>

namespace aoz {

constexpr int MT_CHUNK = 16384;     // elements per chunk (kept in sync with host: aoz_mt_chunk_elems)
constexpr int MT_THREADS = 256;

struct alignas(16) RavenHyper {     // per tensor, fp32 images of the float64 host scalars (raven.py:101-137)
    float beta1, one_minus_beta1, beta2, one_minus_beta2;
    float eps, step_size, inv_sqrt_bc2, wd_factor;
};

enum DType : int { DT_F32 = 0, DT_BF16 = 1, DT_F16 = 2 };

template <int DT> struct Elem;
template <> struct Elem<DT_F32> {
    using T = float;
    static __device__ __forceinline__ float ld(const T* p) { return *p; }
    static __device__ __forceinline__ void st(T* p, float v) { *p = v; }
};
template <> struct Elem<DT_BF16> {
    using T = __nv_bfloat16;
    static __device__ __forceinline__ float ld(const T* p) { return __bfloat162float(*p); }
    static __device__ __forceinline__ void st(T* p, float v) { *p = __float2bfloat16_rn(v); }
};
template <> struct Elem<DT_F16> {
    using T = __half;
    static __device__ __forceinline__ float ld(const T* p) { return __half2float(*p); }
    static __device__ __forceinline__ void st(T* p, float v) { *p = __float2half_rn(v); }
};

// load 8 consecutive elements as fp32
template <int DT> __device__ __forceinline__ void ld8(const void* base, size_t i, float* f);

template <> __device__ __forceinline__ void ld8<DT_F32>(const void* base, size_t i, float* f) {
    const float* p = (const float*)base + i;
    uint4 a = ld_stream(p), b = ld_stream(p + 4);
    f[0] = __uint_as_float(a.x); f[1] = __uint_as_float(a.y); f[2] = __uint_as_float(a.z); f[3] = __uint_as_float(a.w);
    f[4] = __uint_as_float(b.x); f[5] = __uint_as_float(b.y); f[6] = __uint_as_float(b.z); f[7] = __uint_as_float(b.w);
}
template <> __device__ __forceinline__ void ld8<DT_BF16>(const void* base, size_t i, float* f) {
    uint4 a = ld_stream((const __nv_bfloat16*)base + i);
    f[0] = bf16lo(a.x); f[1] = bf16hi(a.x); f[2] = bf16lo(a.y); f[3] = bf16hi(a.y);
    f[4] = bf16lo(a.z); f[5] = bf16hi(a.z); f[6] = bf16lo(a.w); f[7] = bf16hi(a.w);
}
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
template <> __device__ __forceinline__ void ld8<DT_F16>(const void* base, size_t i, float* f) {
    uint4 a = ld_stream((const __half*)base + i);
    const __half2* h = reinterpret_cast<const __half2*>(&a);
#pragma unroll
    for (int k = 0; k < 4; ++k) { float2 t = __half22float2(h[k]); f[2 * k] = t.x; f[2 * k + 1] = t.y; }
}

// 8 consecutive elements <-> fp32 in SHARED memory (the bulk-copy ring of raven_step_bulk_kernel)
template <int DT> __device__ __forceinline__ void lds8(const uint8_t* base, int i, float* f);
template <int DT> __device__ __forceinline__ void sts8(uint8_t* base, int i, const float* f);
template <> __device__ __forceinline__ void lds8<DT_F32>(const uint8_t* base, int i, float* f) {
    const float4* p = reinterpret_cast<const float4*>(base) + (i >> 2);
    const float4 a = p[0], b = p[1];
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
template <> __device__ __forceinline__ void sts8<DT_F32>(uint8_t* base, int i, const float* f) {
    float4* p = reinterpret_cast<float4*>(base) + (i >> 2);
    p[0] = make_float4(f[0], f[1], f[2], f[3]); p[1] = make_float4(f[4], f[5], f[6], f[7]);
}
template <> __device__ __forceinline__ void lds8<DT_BF16>(const uint8_t* base, int i, float* f) {
    const uint4 a = reinterpret_cast<const uint4*>(base)[i >> 3];
    f[0] = bf16lo(a.x); f[1] = bf16hi(a.x); f[2] = bf16lo(a.y); f[3] = bf16hi(a.y);
    f[4] = bf16lo(a.z); f[5] = bf16hi(a.z); f[6] = bf16lo(a.w); f[7] = bf16hi(a.w);
}
template <> __device__ __forceinline__ void sts8<DT_BF16>(uint8_t* base, int i, const float* f) {
    reinterpret_cast<uint4*>(base)[i >> 3] = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
}
template <> __device__ __forceinline__ void lds8<DT_F16>(const uint8_t* base, int i, float* f) {
    const uint4 a = reinterpret_cast<const uint4*>(base)[i >> 3];
    const __half2* h = reinterpret_cast<const __half2*>(&a);
#pragma unroll
    for (int k = 0; k < 4; ++k) { float2 t = __half22float2(h[k]); f[2 * k] = t.x; f[2 * k + 1] = t.y; }
}
template <> __device__ __forceinline__ void sts8<DT_F16>(uint8_t* base, int i, const float* f) {
    reinterpret_cast<uint4*>(base)[i >> 3] = make_uint4(pack_f16(f[0], f[1]), pack_f16(f[2], f[3]), pack_f16(f[4], f[5]), pack_f16(f[6], f[7]));
}

// One element of the update, in the reference's operation order (raven.py:126-143); fp32 throughout.
// __fmul_rn/__fadd_rn keep nvcc from contracting across the reference's separate ATen kernels.
template <int GDT>
__device__ __forceinline__ void raven_elem(float& p, float g, float& m, float& v, const RavenHyper& h, float clip,
                                           bool use_clip) {
    if (use_clip) {
        g = g * clip;                                   // torch._foreach_mul_(grads, coef): rounds to grad dtype
        if (GDT == DT_BF16) g = round_bf16(g);
        if (GDT == DT_F16) g = __half2float(__float2half_rn(g));
    }
    m = __fmaf_rn(h.one_minus_beta1, g, __fmul_rn(m, h.beta1));                     // mul_(b1).add_(g, alpha=1-b1)
    v = __fmaf_rn(__fmul_rn(h.one_minus_beta2, g), g, __fmul_rn(v, h.beta2));       // mul_(b2).addcmul_(g, g, 1-b2)
    p = __fmul_rn(p, h.wd_factor);                                                  // p.mul_(1 - lr*wd)
    float denom = __fadd_rn(__fmul_rn(sqrtf(v), h.inv_sqrt_bc2), h.eps);            // sqrt().div_(sqrt_bc2).add_(eps)
    p = __fmaf_rn(-h.step_size, __fdiv_rn(m, denom), p);                            // addcdiv_(m, denom, -step_size)
}

// ---- the update, streamed through shared memory by the TMA engine ---------------------------------------------
// One thread per CTA runs BULK_STAGES - 1 items ahead of the math: an item is BULK_SUB elements of one chunk, fetched as four
// cp.async.bulk copies (p, g, m, v) into a ring in shared memory; 256 threads update 8 elements each in place (one 16-byte
// shared-memory access per stream); three bulk copies write p, m, v back.  No register ever waits on HBM, and the dependent loads
// of a chunk's metadata are hidden behind the items in flight.  (Streaming through registers -- 2 x 4 16-byte requests per thread,
// load and compute / store phases alternating, ~1 us stalls at every chunk start -- reached 0.73-0.79 of the measured HBM
// bandwidth over the real 1680-tensor table; this kernel took the step's update from 7.4 to 6.9 ms.)
// Pieces that cannot be moved in 16-byte granules (pointers off alignment, the last < 8 elements of a tensor) take the direct path.
constexpr int BULK_SUB = 2048;                  // elements per item = 8 per thread
constexpr int BULK_STAGES = 4;

struct BulkMeta {                               // written by the producer thread when it issues an item's loads
    int cnt;                                    // elements moved by bulk copies (multiple of 8); the math covers exactly these
    int tail;                                   // following elements handled directly in global memory (0..BULK_SUB: unaligned items)
    int tensor;
    int pad;
    long long first;                            // element index of the item inside its tensor
};

__device__ __forceinline__ void bulk_store_1d(void* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}

template <int PDT, int GDT, int MDT>
__global__ void __launch_bounds__(MT_THREADS)
raven_step_bulk_kernel(int n_chunks, const uint64_t* __restrict__ p_ptrs, const uint64_t* __restrict__ g_ptrs,
                       const uint64_t* __restrict__ m_ptrs, const uint64_t* __restrict__ v_ptrs,
                       const int64_t* __restrict__ numel, const int32_t* __restrict__ chunk_start,
                       const int32_t* __restrict__ chunk_tensor, const RavenHyper* __restrict__ hyper,
                       const float* __restrict__ clip_coef) {
    using PE = Elem<PDT>;
    using GE = Elem<GDT>;
    using ME = Elem<MDT>;
    constexpr int SP = sizeof(typename PE::T), SG = sizeof(typename GE::T), SM_ = sizeof(typename ME::T);
    constexpr int STAGE_BYTES = BULK_SUB * (SP + SG + 2 * SM_);
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t full[BULK_STAGES];
    __shared__ BulkMeta meta[BULK_STAGES];
    const bool use_clip = clip_coef != nullptr;
    const float clip = use_clip ? __ldg(clip_coef) : 1.0f;
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int i = 0; i < BULK_STAGES; ++i) mbar_init(&full[i], 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto stage_ptr = [&](int s, int which) -> uint8_t* {       // which: 0 p, 1 g, 2 m, 3 v
        uint8_t* b = smem + (size_t)s * STAGE_BYTES;
        return which == 0 ? b : which == 1 ? b + BULK_SUB * SP : which == 2 ? b + BULK_SUB * (SP + SG) : b + BULK_SUB * (SP + SG + SM_);
    };
    // the item sequence of this CTA: chunks blockIdx.x, + gridDim.x, ...; inside a chunk BULK_SUB elements at a time
    struct Cursor { int c; int k; };
    auto next_item = [&](Cursor& cur) -> bool {                // advance to the next existing item; false when the CTA is done
        for (;;) {
            if (cur.c >= n_chunks) return false;
            const int t = chunk_tensor[cur.c];
            const int64_t begin = (int64_t)(cur.c - chunk_start[t]) * MT_CHUNK + (int64_t)cur.k * BULK_SUB;
            const int64_t end = min((int64_t)(cur.c - chunk_start[t] + 1) * MT_CHUNK, numel[t]);
            if (begin < end) return true;
            cur.c += gridDim.x; cur.k = 0;
        }
    };
    auto issue = [&](const Cursor& cur, int slot) {            // producer thread only
        const int t = chunk_tensor[cur.c];
        const int64_t first = (int64_t)(cur.c - chunk_start[t]) * MT_CHUNK + (int64_t)cur.k * BULK_SUB;
        const int64_t end = min((int64_t)(cur.c - chunk_start[t] + 1) * MT_CHUNK, numel[t]);
        const int n = (int)min((int64_t)BULK_SUB, end - first);
        uint8_t* p = (uint8_t*)p_ptrs[t] + first * SP;
        uint8_t* g = (uint8_t*)g_ptrs[t] + first * SG;
        uint8_t* m = (uint8_t*)m_ptrs[t] + first * SM_;
        uint8_t* v = (uint8_t*)v_ptrs[t] + first * SM_;
        const bool aligned = ((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0);
        const int cnt = aligned ? (n & ~7) : 0;
        meta[slot].cnt = cnt; meta[slot].tail = n - cnt; meta[slot].tensor = t; meta[slot].first = first;
        if (cnt > 0) {
            mbar_arrive_expect_tx(&full[slot], (uint32_t)cnt * (SP + SG + 2 * SM_));
            bulk_load_1d(stage_ptr(slot, 0), p, cnt * SP, &full[slot]);
            bulk_load_1d(stage_ptr(slot, 1), g, cnt * SG, &full[slot]);
            bulk_load_1d(stage_ptr(slot, 2), m, cnt * SM_, &full[slot]);
            bulk_load_1d(stage_ptr(slot, 3), v, cnt * SM_, &full[slot]);
        } else {
            mbar_arrive(&full[slot]);
        }
    };
    Cursor prod{(int)blockIdx.x, 0};
    int produced = 0;
    bool more = true;
    if (tid == 0) {
        for (; produced < BULK_STAGES - 1; ++produced) {
            more = next_item(prod);
            if (!more) break;
            issue(prod, produced % BULK_STAGES);
            ++prod.k;
        }
    }
    Cursor cons{(int)blockIdx.x, 0};
    for (int n = 0; next_item(cons); ++n, ++cons.k) {
        const int slot = n % BULK_STAGES;
        mbar_wait(&full[slot], (n / BULK_STAGES) & 1);
        const BulkMeta mt = meta[slot];
        const RavenHyper h = hyper[mt.tensor];
        // ---- math on the staged elements (shared memory, 8 per thread) ----
        if (8 * tid < mt.cnt) {
            float pf[8], gf[8], mf[8], vf[8];
            lds8<PDT>(stage_ptr(slot, 0), 8 * tid, pf); lds8<GDT>(stage_ptr(slot, 1), 8 * tid, gf);
            lds8<MDT>(stage_ptr(slot, 2), 8 * tid, mf); lds8<MDT>(stage_ptr(slot, 3), 8 * tid, vf);
#pragma unroll
            for (int k = 0; k < 8; ++k) raven_elem<GDT>(pf[k], gf[k], mf[k], vf[k], h, clip, use_clip);
            sts8<PDT>(stage_ptr(slot, 0), 8 * tid, pf); sts8<MDT>(stage_ptr(slot, 2), 8 * tid, mf); sts8<MDT>(stage_ptr(slot, 3), 8 * tid, vf);
        }
        // ---- the part that bulk copies cannot move: straight through global memory ----
        if (mt.tail > 0) {
            typename PE::T* p = (typename PE::T*)p_ptrs[mt.tensor];
            const typename GE::T* g = (const typename GE::T*)g_ptrs[mt.tensor];
            typename ME::T* m = (typename ME::T*)m_ptrs[mt.tensor];
            typename ME::T* v = (typename ME::T*)v_ptrs[mt.tensor];
            for (int64_t i = mt.first + mt.cnt + tid; i < mt.first + mt.cnt + mt.tail; i += MT_THREADS) {
                float pf = PE::ld(p + i), gf = GE::ld(g + i), mf = ME::ld(m + i), vf = ME::ld(v + i);
                raven_elem<GDT>(pf, gf, mf, vf, h, clip, use_clip);
                PE::st(p + i, pf); ME::st(m + i, mf); ME::st(v + i, vf);
            }
        }
        fence_proxy_async_smem();
        __syncthreads();
        if (tid == 0) {
            if (mt.cnt > 0) {
                bulk_store_1d((uint8_t*)p_ptrs[mt.tensor] + mt.first * SP, stage_ptr(slot, 0), mt.cnt * SP);
                bulk_store_1d((uint8_t*)m_ptrs[mt.tensor] + mt.first * SM_, stage_ptr(slot, 2), mt.cnt * SM_);
                bulk_store_1d((uint8_t*)v_ptrs[mt.tensor] + mt.first * SM_, stage_ptr(slot, 3), mt.cnt * SM_);
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            // the ring slot that the next load overwrites was stored from one iteration ago: all but the newest group must have
            // finished READING shared memory
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            if (more) {
                more = next_item(prod);
                if (more) { issue(prod, produced % BULK_STAGES); ++produced; ++prod.k; }
            }
        }
    }
    if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---- gradient norm: per-chunk partial sum of squares (deterministic, no atomics) ------------------------
template <int GDT>
__global__ void __launch_bounds__(MT_THREADS)
sumsq_mt_kernel(int n_chunks, const uint64_t* __restrict__ g_ptrs, const int64_t* __restrict__ numel,
                const int32_t* __restrict__ chunk_start, const int32_t* __restrict__ chunk_tensor,
                float* __restrict__ partial) {
    using GE = Elem<GDT>;
    __shared__ float wsum[MT_THREADS / 32];
    for (int c = blockIdx.x; c < n_chunks; c += gridDim.x) {
        const int t = chunk_tensor[c];
        const typename GE::T* g = (const typename GE::T*)g_ptrs[t];
        const int64_t n = numel[t];
        const int64_t begin = (int64_t)(c - chunk_start[t]) * MT_CHUNK;
        const int64_t end = min(begin + (int64_t)MT_CHUNK, n);
        const bool aligned = (((uintptr_t)g) & (GDT == DT_F32 ? 31 : 15)) == 0;
        int64_t vec_end = aligned ? begin + ((end - begin) & ~(int64_t)7) : begin;
        float acc = 0.f;
        for (int64_t i = begin + (int64_t)threadIdx.x * 8; i < vec_end; i += (int64_t)MT_THREADS * 8) {
            float f[8];
            ld8<GDT>(g, i, f);
#pragma unroll
            for (int k = 0; k < 8; ++k) acc = fmaf(f[k], f[k], acc);
        }
        for (int64_t i = vec_end + threadIdx.x; i < end; i += MT_THREADS) {
            float f = GE::ld(g + i);
            acc = fmaf(f, f, acc);
        }
        acc = warp_sum(acc);
        if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x < 32) {
            float s = threadIdx.x < MT_THREADS / 32 ? wsum[threadIdx.x] : 0.f;
            s = warp_sum(s);
            if (threadIdx.x == 0) partial[c] = s;
        }
        __syncthreads();
    }
}

// Final reduction + clip coefficient, one block.  out[0] = total norm, out[1] = clip coefficient
// clamp(max_norm / (norm + 1e-6), max=1), out[2] = total sum of squares (fp32, unrounded; used by the
// data-parallel path which all-reduces it before forming the norm).
// emulate_bf16 != 0 reproduces torch's dtype behaviour for bf16 grads (SURVEY.md a7): every per-tensor norm,
// the total norm and the coefficient are rounded to bf16, exactly what clip_grad_norm_ does on bf16 tensors.
__global__ void __launch_bounds__(1024)
gradnorm_finalize_kernel(int n_tensors, const int32_t* __restrict__ chunk_start, const float* __restrict__ partial,
                         float max_norm, int emulate_bf16, float* __restrict__ out) {
    __shared__ float wsum[32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float acc = 0.f;   // sum over this warp's tensors of (per-tensor norm)^2 (lane 0 holds it)
    for (int t = warp; t < n_tensors; t += 32) {
        float s = 0.f;
        for (int c = chunk_start[t] + lane; c < chunk_start[t + 1]; c += 32) s += partial[c];
        s = warp_sum(s);
        if (emulate_bf16) {
            float nrm = round_bf16(sqrtf(s));
            s = nrm * nrm;
        }
        acc += s;
    }
    if (lane == 0) wsum[warp] = acc;
    __syncthreads();
    if (warp == 0) {
        float s = warp_sum(wsum[lane]);
        if (lane == 0) {
            float nrm = sqrtf(s);
            float coef;
            if (emulate_bf16) {
                nrm = round_bf16(nrm);
                float d = round_bf16(nrm + 1e-6f);
                coef = round_bf16(max_norm / d);
            } else {
                coef = max_norm / (nrm + 1e-6f);
            }
            coef = fminf(coef, 1.0f);
            out[0] = nrm;
            out[1] = coef;
            out[2] = s;
        }
    }
}

// coefficient from an externally reduced sum of squares (data-parallel: after the all-reduce of out[2])
__global__ void clip_coef_from_sumsq_kernel(const float* __restrict__ sumsq, float max_norm, int emulate_bf16,
                                            float* __restrict__ out) {
    float nrm = sqrtf(sumsq[0]);
    float coef;
    if (emulate_bf16) {
        nrm = round_bf16(nrm);
        coef = round_bf16(max_norm / round_bf16(nrm + 1e-6f));
    } else {
        coef = max_norm / (nrm + 1e-6f);
    }
    out[0] = nrm;
    out[1] = fminf(coef, 1.0f);
}

// ---- gradient accumulation: y[t] = copy ? b[t] : a[t] + b[t], bf16, every tensor in one launch -----------------------
// The arithmetic is add_kernel's (elementwise.cu): fp32 add, one round-to-nearest-even to bf16, so each tensor is bit-identical to
// aoz_add on it.  y may alias a or b: every element is read and then written by the same thread and never read again, which is why
// the loads are the coherent ones and no pointer is __restrict__.  Each CTA owns a contiguous run of chunks, so consecutive chunks
// mostly share a tensor and its table entries stay in registers.  A chunk whose pointers are not all 16-byte aligned, and the last
// (< 8) elements of a tensor, go element by element.
constexpr int ACC_UNROLL = 4;                   // 16-byte vectors per operand in flight per thread

__device__ __forceinline__ uint4 ld_once(const void* p) {
    uint4 r;
    asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
    return r;
}

template <bool COPY>
__global__ void __launch_bounds__(MT_THREADS)
grad_accum_mt_kernel(int n_chunks, int chunks_per_cta, const uint64_t* __restrict__ a_ptrs, const uint64_t* __restrict__ b_ptrs,
                     const uint64_t* __restrict__ y_ptrs, const int64_t* __restrict__ numel,
                     const int32_t* __restrict__ chunk_start, const int32_t* __restrict__ chunk_tensor) {
    const int c0 = blockIdx.x * chunks_per_cta;
    const int c1 = min(c0 + chunks_per_cta, n_chunks);
    if (c0 >= c1) return;
    int t = chunk_tensor[c0];
    int t_first = chunk_start[t], t_next = chunk_start[t + 1];
    const __nv_bfloat16* a = COPY ? nullptr : (const __nv_bfloat16*)a_ptrs[t];
    const __nv_bfloat16* b = (const __nv_bfloat16*)b_ptrs[t];
    __nv_bfloat16* y = (__nv_bfloat16*)y_ptrs[t];
    int64_t n = numel[t];
    for (int c = c0; c < c1; ++c) {
        if (c >= t_next) {                      // tensors without elements own no chunk: skip past them
            do { ++t; t_first = t_next; t_next = chunk_start[t + 1]; } while (c >= t_next);
            if (!COPY) a = (const __nv_bfloat16*)a_ptrs[t];
            b = (const __nv_bfloat16*)b_ptrs[t];
            y = (__nv_bfloat16*)y_ptrs[t];
            n = numel[t];
        }
        const int64_t begin = (int64_t)(c - t_first) * MT_CHUNK;
        const int64_t end = min(begin + (int64_t)MT_CHUNK, n);
        const bool aligned = ((((uintptr_t)a | (uintptr_t)b | (uintptr_t)y) & 15) == 0);
        const int64_t vec_end = aligned ? begin + ((end - begin) & ~(int64_t)7) : begin;
        for (int64_t i = begin + (int64_t)threadIdx.x * 8; i < vec_end; i += (int64_t)MT_THREADS * 8 * ACC_UNROLL) {
            uint4 va[ACC_UNROLL], vb[ACC_UNROLL];
#pragma unroll
            for (int u = 0; u < ACC_UNROLL; ++u) {
                const int64_t j = i + (int64_t)u * MT_THREADS * 8;
                if (j < vec_end) {
                    vb[u] = ld_once(b + j);
                    if (!COPY) va[u] = ld_once(a + j);
                }
            }
#pragma unroll
            for (int u = 0; u < ACC_UNROLL; ++u) {
                const int64_t j = i + (int64_t)u * MT_THREADS * 8;
                if (j < vec_end) {
                    if (COPY) {
                        st_stream(y + j, vb[u]);
                    } else {
                        const uint4 ra = va[u], rb = vb[u];
                        st_stream(y + j, make_uint4(pack_bf16(bf16lo(ra.x) + bf16lo(rb.x), bf16hi(ra.x) + bf16hi(rb.x)),
                                                    pack_bf16(bf16lo(ra.y) + bf16lo(rb.y), bf16hi(ra.y) + bf16hi(rb.y)),
                                                    pack_bf16(bf16lo(ra.z) + bf16lo(rb.z), bf16hi(ra.z) + bf16hi(rb.z)),
                                                    pack_bf16(bf16lo(ra.w) + bf16lo(rb.w), bf16hi(ra.w) + bf16hi(rb.w))));
                    }
                }
            }
        }
        for (int64_t i = vec_end + threadIdx.x; i < end; i += MT_THREADS)
            y[i] = COPY ? b[i] : __float2bfloat16_rn(__bfloat162float(a[i]) + __bfloat162float(b[i]));
    }
}

}  // namespace aoz

using namespace aoz;

extern "C" {

int aoz_mt_chunk_elems(void) { return MT_CHUNK; }

int aoz_raven_step_mt(int n_tensors, int n_chunks, const void* p_ptrs, const void* g_ptrs, const void* m_ptrs,
                      const void* v_ptrs, const void* numel, const void* chunk_start, const void* chunk_tensor,
                      const void* hyper, const void* clip_coef, int p_dtype, int g_dtype, int m_dtype, void* stream) {
    AOZ_CHECK_ARG(n_tensors >= 0 && n_chunks >= 0, "aoz_raven_step_mt: negative sizes");
    if (n_tensors == 0 || n_chunks == 0) return AOZ_OK;
    AOZ_CHECK_ARG(p_ptrs && g_ptrs && m_ptrs && v_ptrs && numel && chunk_start && chunk_tensor && hyper,
                  "aoz_raven_step_mt: null table pointer");
    cudaStream_t s = (cudaStream_t)stream;
#define AOZ_RAVEN_LAUNCH(P, G, M)                                                                                  \
    do {                                                                                                           \
        constexpr int esz = (P == DT_F32 ? 4 : 2) + (G == DT_F32 ? 4 : 2) + 2 * (M == DT_F32 ? 4 : 2);             \
        constexpr int smem = BULK_STAGES * BULK_SUB * esz;                                                         \
        static bool attr = false;                                                                                  \
        if (!attr) { cudaFuncSetAttribute(raven_step_bulk_kernel<P, G, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); attr = true; } \
        const int per_sm = (200 * 1024) / (smem + 1024) > 0 ? (200 * 1024) / (smem + 1024) : 1;                    \
        const int grid = n_chunks < sm_count() * per_sm ? n_chunks : sm_count() * per_sm;                          \
        raven_step_bulk_kernel<P, G, M><<<grid, MT_THREADS, smem, s>>>(                                            \
            n_chunks, (const uint64_t*)p_ptrs, (const uint64_t*)g_ptrs, (const uint64_t*)m_ptrs, (const uint64_t*)v_ptrs, \
            (const int64_t*)numel, (const int32_t*)chunk_start, (const int32_t*)chunk_tensor, (const RavenHyper*)hyper,  \
            (const float*)clip_coef);                                                                              \
    } while (0)
#define AOZ_RAVEN_M(P, G)                                                          \
    if (m_dtype == DT_BF16) AOZ_RAVEN_LAUNCH(P, G, DT_BF16);                        \
    else if (m_dtype == DT_F32) AOZ_RAVEN_LAUNCH(P, G, DT_F32);                     \
    else AOZ_RAVEN_LAUNCH(P, G, DT_F16)
    if (m_dtype < 0 || m_dtype > 2) { set_error("aoz_raven_step_mt: bad m_dtype %d", m_dtype); return AOZ_ERR_UNSUPPORTED; }
    if (p_dtype == DT_BF16 && g_dtype == DT_BF16) { AOZ_RAVEN_M(DT_BF16, DT_BF16); }
    else if (p_dtype == DT_BF16 && g_dtype == DT_F32) { AOZ_RAVEN_M(DT_BF16, DT_F32); }
    else if (p_dtype == DT_F32 && g_dtype == DT_F32) { AOZ_RAVEN_M(DT_F32, DT_F32); }
    else { set_error("aoz_raven_step_mt: unsupported dtypes p=%d g=%d m=%d", p_dtype, g_dtype, m_dtype); return AOZ_ERR_UNSUPPORTED; }
#undef AOZ_RAVEN_M
#undef AOZ_RAVEN_LAUNCH
    AOZ_CHECK_LAUNCH("raven_step_bulk_kernel");
    return AOZ_OK;
}

int aoz_gradnorm_mt(int n_tensors, int n_chunks, const void* g_ptrs, const void* numel, const void* chunk_start,
                    const void* chunk_tensor, void* partial, float max_norm, int emulate_bf16, void* out3,
                    int g_dtype, void* stream) {
    AOZ_CHECK_ARG(n_tensors >= 0 && n_chunks >= 0, "aoz_gradnorm_mt: negative sizes");
    AOZ_CHECK_ARG(out3 != nullptr, "aoz_gradnorm_mt: out is null");
    cudaStream_t s = (cudaStream_t)stream;
    if (n_chunks > 0) {
        AOZ_CHECK_ARG(g_ptrs && numel && chunk_start && chunk_tensor && partial, "aoz_gradnorm_mt: null table pointer");
        int grid = n_chunks < sm_count() * 8 ? n_chunks : sm_count() * 8;
        if (g_dtype == DT_BF16)
            sumsq_mt_kernel<DT_BF16><<<grid, MT_THREADS, 0, s>>>(n_chunks, (const uint64_t*)g_ptrs, (const int64_t*)numel,
                                                                  (const int32_t*)chunk_start, (const int32_t*)chunk_tensor, (float*)partial);
        else if (g_dtype == DT_F32)
            sumsq_mt_kernel<DT_F32><<<grid, MT_THREADS, 0, s>>>(n_chunks, (const uint64_t*)g_ptrs, (const int64_t*)numel,
                                                                 (const int32_t*)chunk_start, (const int32_t*)chunk_tensor, (float*)partial);
        else if (g_dtype == DT_F16)
            sumsq_mt_kernel<DT_F16><<<grid, MT_THREADS, 0, s>>>(n_chunks, (const uint64_t*)g_ptrs, (const int64_t*)numel,
                                                                 (const int32_t*)chunk_start, (const int32_t*)chunk_tensor, (float*)partial);
        else { set_error("aoz_gradnorm_mt: unsupported dtype %d", g_dtype); return AOZ_ERR_UNSUPPORTED; }
        AOZ_CHECK_LAUNCH("sumsq_mt_kernel");
    }
    gradnorm_finalize_kernel<<<1, 1024, 0, s>>>(n_tensors, (const int32_t*)chunk_start, (const float*)partial, max_norm,
                                                emulate_bf16, (float*)out3);
    AOZ_CHECK_LAUNCH("gradnorm_finalize_kernel");
    return AOZ_OK;
}

int aoz_clip_coef_from_sumsq(const void* sumsq, float max_norm, int emulate_bf16, void* out2, void* stream) {
    AOZ_CHECK_ARG(sumsq && out2, "aoz_clip_coef_from_sumsq: null pointer");
    clip_coef_from_sumsq_kernel<<<1, 1, 0, (cudaStream_t)stream>>>((const float*)sumsq, max_norm, emulate_bf16, (float*)out2);
    AOZ_CHECK_LAUNCH("clip_coef_from_sumsq_kernel");
    return AOZ_OK;
}

int aoz_grad_accum_mt(int n_tensors, int n_chunks, const void* a_ptrs, const void* b_ptrs, const void* y_ptrs,
                      const void* numel, const void* chunk_start, const void* chunk_tensor, int copy, void* stream) {
    AOZ_CHECK_ARG(n_tensors > 0 && n_chunks >= 0, "aoz_grad_accum_mt: n_tensors must be positive, n_chunks non-negative");
    AOZ_CHECK_ARG(b_ptrs && y_ptrs && numel && chunk_start && chunk_tensor && (copy || a_ptrs),
                  "aoz_grad_accum_mt: null table pointer");
    AOZ_CHECK_ARG(((((uintptr_t)a_ptrs | (uintptr_t)b_ptrs | (uintptr_t)y_ptrs | (uintptr_t)numel) & 7) == 0) &&
                  ((((uintptr_t)chunk_start | (uintptr_t)chunk_tensor) & 3) == 0),
                  "aoz_grad_accum_mt: misaligned table pointer");
    if (n_chunks == 0) return AOZ_OK;
    static int per_sm = 0;
    if (per_sm == 0) {
        int k = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&k, grad_accum_mt_kernel<false>, MT_THREADS, 0);
        per_sm = k > 0 ? k : 1;
    }
    const int ctas = n_chunks < sm_count() * per_sm ? n_chunks : sm_count() * per_sm;
    const int per_cta = (n_chunks + ctas - 1) / ctas;
    const int grid = (n_chunks + per_cta - 1) / per_cta;
    cudaStream_t s = (cudaStream_t)stream;
    if (copy)
        grad_accum_mt_kernel<true><<<grid, MT_THREADS, 0, s>>>(n_chunks, per_cta, (const uint64_t*)a_ptrs, (const uint64_t*)b_ptrs,
                                                               (const uint64_t*)y_ptrs, (const int64_t*)numel,
                                                               (const int32_t*)chunk_start, (const int32_t*)chunk_tensor);
    else
        grad_accum_mt_kernel<false><<<grid, MT_THREADS, 0, s>>>(n_chunks, per_cta, (const uint64_t*)a_ptrs, (const uint64_t*)b_ptrs,
                                                                (const uint64_t*)y_ptrs, (const int64_t*)numel,
                                                                (const int32_t*)chunk_start, (const int32_t*)chunk_tensor);
    AOZ_CHECK_LAUNCH("grad_accum_mt_kernel");
    return AOZ_OK;
}

}  // extern "C"
