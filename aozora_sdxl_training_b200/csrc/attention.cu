// Flash-style attention forward and backward on tcgen05 / TMEM / TMA for head_dim 64 (sm_100a).
//
// Replaces F.scaled_dot_product_attention as called by diffusers' AttnProcessor2_0 for Attention.attn1
// (self, Tk = Tq) and Attention.attn2 (cross, Tk = 77*n) inside the UNet (reference: train.py:213-229 selects the
// processor, train.py:2760 runs it; no mask, no dropout, scale 1/sqrt(64)).  The reference's backward is autograd
// through SDPA; here the backward recomputes P from the saved log-sum-exp, after attn_bwd_prep_kernel has formed
// D = rowsum(dO * O), in one of two forms:
//   attn_bwd_fused_kernel (default)          ONE kernel: dK, dV and each KV tile's share of dQ, the shares summed in fp32
//                                            (not bit-reproducible); attn_dq_tiles_convert_kernel scales and rounds them
//   attn_bwd_dkv_kernel + attn_bwd_dq_kernel bit-reproducible: the reference the fused kernel is tested against, and the
//                                            path taken when Tq % 4 != 0 (aoz_attn_set_bwd_mode(0) selects it everywhere)
//
// Common structure (per CTA): compute warps, one thread per tile row, do the softmax / dS math on the TMEM accumulators
// (tcgen05.ld); one warp is the TMA producer (4-D tensor maps over [B, T, H, 64]; rows past T are zero-filled by the TMA
// unit), one the MMA issuer (tcgen05.mma, completion through tcgen05.commit -> mbarrier).  S / dP / O / dK / dV / dQ
// accumulators live in TMEM.  Tiles: 128 query rows x 128 key rows (forward: 64 key rows).
//
// forward : per Q tile, loop over KV tiles:  S = Q K^T -> online softmax (log2 domain, lazy rescale of O) -> O += P V ;
//           stores O (bf16), LSE (fp32)
// fused   : per KV tile, loop over Q tiles:  S^T = K Q^T, dP^T = V dO^T, P^T = exp(S^T - LSE), dS^T = P^T (dP^T - D),
//           dV += P^T dO, dK += dS^T Q, dQ share += dS K
// dK/dV   : per KV tile, loop over Q tiles:  S = Q K^T, dP = dO V^T, P = exp(S - LSE), dS = P (dP - D),
//           dV += P^T dO, dK += dS^T Q
// dQ      : per Q tile, loop over KV tiles:  S = Q K^T, dP = dO V^T, dS = P (dP - D), dQ += dS K
// A [rows, 64] tile loaded once by TMA serves both as a K-major operand (contraction over d) and as an
// MN-major operand (contraction over its rows): only the UMMA descriptor changes.
#include "common.cuh"
#include <cstring>

namespace aoz {

constexpr int BWD_CW = 16;                 // backward: 16 compute warps = four per TMEM lane quarter, 32 of a tile's 128 columns each
constexpr int BWD_CT = BWD_CW * 32;        // (the math is latency-bound: 8 warps left the issue slots 73 % idle, ncu r01)
constexpr int ATT_BWD_THREADS = BWD_CT + 64;   // + TMA producer warp + MMA issuer warp
constexpr int TILE = 128;
constexpr int HD = 64;
constexpr int TILE_BYTES = TILE * HD * 2;     // 16 KB: one [128, 64] bf16 tile
constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;

struct AttnParams {
    CUtensorMap tmQ, tmK, tmV, tmDO;
    int B, H, Tq, Tk;
    float scale;
    __nv_bfloat16* O; long long ldo;
    float* lse;                 // [B, H, Tq]
    const float* Dvec;          // [B, H, Tq]  rowsum(dO * O)
    __nv_bfloat16* dQ; long long lddq;
    __nv_bfloat16* dK; long long lddk;
    __nv_bfloat16* dV; long long lddv;
    float* dQacc;               // one-kernel backward: the KV tiles' dQ shares, summed into swizzled fp32 tiles
    int q_split;                // one-kernel backward: the Q tiles of a KV tile are cut over q_split CTAs (cross-attention: one KV tile,
    float* dKacc;               //   B * H CTAs would leave most SMs idle); with q_split > 1 the CTAs' dK / dV shares are summed into
    float* dVacc;               //   these fp32 tile buffers by bulk reduce-add, like dQ
};

__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ float4 ld_shared_f4(uint32_t addr) {       // explicit shared-space load (a generic LD costs ~2x the latency)
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" :: "r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// descriptors for the three operand shapes used below
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t tile_addr, int k16) {            // [rows,64] tile, contraction over d
    return make_sdesc_sw128(tile_addr + k16 * 32, 16, 1024);
}
__device__ __forceinline__ uint64_t desc_rows_as_k(uint32_t tile_addr, int k16) {         // [rows,64] tile, contraction over rows
    return make_sdesc_sw128(tile_addr + k16 * 2048, 8192, 1024);
}
__device__ __forceinline__ uint64_t desc_ptile(uint32_t p_addr, int k16) {                 // [128, 128] as two [128,64] blocks
    return make_sdesc_sw128(p_addr + (k16 >> 2) * TILE_BYTES + (k16 & 3) * 32, 16, 1024);
}
// write 16 consecutive bf16 values (8 words) of row `r`, columns [c0, c0+16) of a [128,128] P tile
__device__ __forceinline__ void store_p_16(uint32_t p_addr, int r, int c0, const uint32_t* w) {
    const uint32_t blk = p_addr + (c0 >> 6) * TILE_BYTES;
    const int chunk0 = (c0 & 63) >> 3;
    st_shared_v4(blk + sw128_offset(r, chunk0), w[0], w[1], w[2], w[3]);
    st_shared_v4(blk + sw128_offset(r, chunk0 + 1), w[4], w[5], w[6], w[7]);
}

// ================================================================================================
// forward: S = Q K^T -> online softmax -> O += P V, P kept in tensor memory
// ================================================================================================
// Measured on B200 (tools/tmem_probe.cu, profiles/r02_tmem_probe.txt): tcgen05.ld sustains ~930 B/clk/SM and ex2 exactly 16 /clk/SM,
// so a 128 x 128 score tile costs 1024 MUFU cycles against 512 MMA cycles and ~70 cycles of TMEM reads: the exponentials are the
// bound.  The round-1 forward (split statistics, P through shared memory) ran at 1966 cycles per tile (ncu r01) for two reasons
// that ncu's source view showed in round 2: its single issuing THREAD was the critical path (see elect_one_sync), and with ~9
// instructions per score element the softmax warps were issue-bound.  This kernel is built to keep the MUFU pipe fed:
//   * one thread per query row and 64-key tiles; per score element 1 FFMA + 1 MUFU + 1 FADD + 0.5 F2FP + 0.17 integer max;
//   * P never leaves tensor memory: a thread overwrites the front of ITS OWN score row with 32 packed bf16x2 words (tcgen05.st) and
//     P V is a tcgen05.mma whose A operand is read from TMEM (layout verified by tools/tmem_probe.cu) -- no shared-memory P tile,
//     no proxy fence, 48 KB of shared memory and 128 TMEM columns (S | O) per CTA, so FOUR CTAs are resident per SM and the
//     hardware interleaves their softmax / MMA phases (16 softmax warps per SM; measured 3 CTAs: 697, 4 CTAs: 724 TFLOP/s);
//   * the running maximum is only a REFERENCE (any value that keeps 2^(s - ref) finite works: LSE = ref + log2 l exactly), so the
//     common path does not track the maximum of S at all -- it takes an integer max over the packed bf16 P words and falls back
//     to an exact max + rescale of O and l only when some P exceeded 2^8.
constexpr int KT = 64;                         // keys per score tile
constexpr int KT_BYTES = KT * HD * 2;          // 8 KB: one [64, 64] bf16 tile
constexpr int TM_STAGES = 2;                   // K / V ring
constexpr int ATT_TM_THREADS = 192;            // 4 softmax warps + producer + issuer
constexpr int TM_CTAS = 4;                     // resident CTAs per SM (TMEM: 4 x 128 columns; 80 registers per thread)

struct TmSmem {
    static constexpr int Q = 0;
    static constexpr int K = Q + TILE_BYTES;
    static constexpr int V = K + TM_STAGES * KT_BYTES;
    static constexpr int BAR = V + TM_STAGES * KT_BYTES;    // 256 B of mbarriers
    static constexpr int TOTAL = BAR + 256;
};
static_assert(TM_CTAS * (TmSmem::TOTAL + 1024) <= 228 * 1024, "attention forward must keep TM_CTAS CTAs per SM");

__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ uint32_t max_u16x2(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("max.u16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}

__global__ void __launch_bounds__(ATT_TM_THREADS, TM_CTAS)
attn_fwd_tm_kernel(const __grid_constant__ AttnParams P) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = (uint64_t*)(smem + TmSmem::BAR);
    uint64_t* q_full = bars;                    // 1
    uint64_t* kv_full = bars + 1;               // TM_STAGES
    uint64_t* kv_empty = bars + 1 + TM_STAGES;  // TM_STAGES
    uint64_t* s_ready = bars + 1 + 2 * TM_STAGES;      // S(j) has landed (and with it every earlier MMA of the issuer: P V(j-1) has retired)
    uint64_t* p_ready = s_ready + 1;                   // P(j) is in tensor memory (128 arrivals)
    uint64_t* o_ready = p_ready + 1;
    uint32_t* tmem_slot = (uint32_t*)(o_ready + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q_tiles = (P.Tq + TILE - 1) / TILE;
    const int qt = blockIdx.x % q_tiles;
    const int bh = blockIdx.x / q_tiles;
    const int h = bh % P.H, b = bh / P.H;
    const int q0 = qt * TILE;
    const int nkv = (P.Tk + KT - 1) / KT;

    if (threadIdx.x == 0) {
        mbar_init(q_full, 1);
        for (int i = 0; i < TM_STAGES; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 1); }
        mbar_init(s_ready, 1); mbar_init(p_ready, 4); mbar_init(o_ready, 1);      // p_ready: ONE arrival per softmax warp
        fence_mbar_init();
    }
    if (warp == 5) tmem_alloc(tmem_slot, 128);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tS = tmem, tO = tmem + 64;
    pdl_enter();          // prologue done: wait for the previous kernel's results before the first global access

    if (warp == 4) {
        if (lane == 0) {
            tma_prefetch_desc(&P.tmQ); tma_prefetch_desc(&P.tmK); tma_prefetch_desc(&P.tmV);
            mbar_arrive_expect_tx(q_full, TILE_BYTES);
            tma_load_4d(smem + TmSmem::Q, &P.tmQ, q_full, 0, h, q0, b);
            for (int j = 0; j < nkv; ++j) {
                const int s = j % TM_STAGES;
                mbar_wait_relaxed(&kv_empty[s], ((j / TM_STAGES) & 1) ^ 1);
                mbar_arrive_expect_tx(&kv_full[s], 2 * KT_BYTES);
                tma_load_4d(smem + TmSmem::K + s * KT_BYTES, &P.tmK, &kv_full[s], 0, h, j * KT, b);
                tma_load_4d(smem + TmSmem::V + s * KT_BYTES, &P.tmV, &kv_full[s], 0, h, j * KT, b);
            }
        }
    } else if (warp == 5) {
        // MMA issuer: the WHOLE warp runs this loop converged (waits included) and one elected lane issues -- see elect_one_sync().
        // Every descriptor is the stage-0 descriptor plus an integer offset on its low word (address field, 16-byte units).
        const uint32_t idesc_qk = make_idesc_bf16(128, KT, 0, 0);
        const uint32_t idesc_pv = make_idesc_bf16(128, 64, 0, 1);           // A = P from tensor memory (K-major), B = V rows as K
        const uint64_t dQ = desc_kmajor(smem_u32(smem + TmSmem::Q), 0);     // + 2 per 16-wide k block (32 bytes)
        const uint64_t dK = desc_kmajor(smem_u32(smem + TmSmem::K), 0);     // + 2 per k block, + KT_BYTES / 16 per stage
        const uint64_t dV = desc_rows_as_k(smem_u32(smem + TmSmem::V), 0);  // + 128 per 16 keys (2048 bytes), + KT_BYTES / 16 per stage
        auto issue_s = [&](int j) {
            const int s = j % TM_STAGES;
            mbar_wait(&kv_full[s], (j / TM_STAGES) & 1);
            tc_fence_after();
            if (elect_one_sync()) {
                const uint64_t dk = dK + (uint64_t)(s * (KT_BYTES >> 4));
                umma_bf16(tS, dQ, dk, idesc_qk, 0u);
#pragma unroll
                for (int k = 1; k < 4; ++k) umma_bf16(tS, dQ + 2 * k, dk + 2 * k, idesc_qk, 1u);
                umma_commit(s_ready);
            }
            __syncwarp();
        };
        mbar_wait(q_full, 0);
        issue_s(0);
        for (int j = 0; j < nkv; ++j) {
            const int s = j % TM_STAGES;
            mbar_wait(p_ready, j & 1);
            tc_fence_after();
            if (elect_one_sync()) {
                const uint64_t dv = dV + (uint64_t)(s * (KT_BYTES >> 4));       // P(j): 32 packed words over the front of the score tile
                umma_bf16_ts(tO, tS, dv, idesc_pv, j > 0 ? 1u : 0u);
#pragma unroll
                for (int k = 1; k < 4; ++k) umma_bf16_ts(tO, tS + 8 * k, dv + 128 * k, idesc_pv, 1u);
                umma_commit(&kv_empty[s]);
                if (j + 1 == nkv) umma_commit(o_ready);
            }
            __syncwarp();
            if (j + 1 < nkv) issue_s(j + 1);                       // overwrites S / P(j): ordered behind P V(j) inside the tensor pipe
        }
    } else {
        // ---- softmax warps 0..3: one thread per query row, all 64 key columns of a tile ----
        const int r = warp * 32 + lane;
        const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
        const float sl2 = P.scale * LOG2E;
        float m_ref = -INFINITY, l = 0.f;
        // P(j) = 2^(s * sl2 - m_ref) for the 64 score columns -> 32 packed words in w; adds the row sum to lsum and returns the u16x2 max
        // over the words (bf16 bit patterns of non-negative numbers order like the numbers).  Four 16-column chunks, the tcgen05.ld of
        // chunk c + 1 in flight during the math of chunk c.
        auto exp_pass = [&](uint32_t* w, float& lsum) -> uint32_t {
            uint32_t v[2][16];
            uint32_t mw = 0;
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
            tmem_ld16(tS + lane_off, v[0]);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                tc_wait_ld();
                if (c + 1 < 4) tmem_ld16(tS + lane_off + (c + 1) * 16, v[(c + 1) & 1]);
                const uint32_t* cv = v[c & 1];
#pragma unroll
                for (int e = 0; e < 16; e += 4) {
                    float p[4];
#pragma unroll
                    for (int t = 0; t < 4; ++t) p[t] = fast_exp2(fmaf(__uint_as_float(cv[e + t]), sl2, -m_ref));
                    a0 += p[0]; a1 += p[1]; a2 += p[2]; a3 += p[3];
                    const uint32_t w0 = pack_bf16(p[0], p[1]), w1 = pack_bf16(p[2], p[3]);
                    w[c * 8 + (e >> 1)] = w0; w[c * 8 + (e >> 1) + 1] = w1;
                    mw = max_u16x2(mw, max_u16x2(w0, w1));
                }
            }
            lsum = (a0 + a1) + (a2 + a3);
            return mw;
        };
        // exact maximum of the valid columns of S (first tile, and the rare rescale)
        auto max_pass = [&](int kvalid) -> float {
            float mx = -3.0e38f;
#pragma unroll 1
            for (int c = 0; c < 2; ++c) {
                uint32_t v[32];
                tmem_ld32(tS + lane_off + c * 32, v);
                tc_wait_ld();
#pragma unroll
                for (int e = 0; e < 32; ++e)
                    if (c * 32 + e < kvalid) mx = fmaxf(mx, __uint_as_float(v[e]));
            }
            return mx;
        };
        // masked variant of exp_pass for the last, partial tile (keys >= kvalid are padding: P = 0)
        auto exp_pass_masked = [&](int kvalid, uint32_t* w, float& lsum) {
            float acc = 0.f;
#pragma unroll 1
            for (int c = 0; c < 2; ++c) {
                uint32_t v[32];
                tmem_ld32(tS + lane_off + c * 32, v);
                tc_wait_ld();
#pragma unroll
                for (int e = 0; e < 32; e += 2) {
                    const int ka = c * 32 + e;
                    const float p0 = ka < kvalid ? fast_exp2(fmaf(__uint_as_float(v[e]), sl2, -m_ref)) : 0.f;
                    const float p1 = ka + 1 < kvalid ? fast_exp2(fmaf(__uint_as_float(v[e + 1]), sl2, -m_ref)) : 0.f;
                    acc += p0 + p1;
                    const uint32_t pk = pack_bf16(p0, p1);
                    if (c == 0) w[e >> 1] = pk; else w[16 + (e >> 1)] = pk;
                }
            }
            lsum = acc;
        };
        for (int j = 0; j < nkv; ++j) {
            mbar_wait(s_ready, j & 1);                       // also: P V(j-1) has retired, O may be rescaled
            tc_fence_after();
            const int kvalid = P.Tk - j * KT;                // keys >= kvalid are padding
            uint32_t w[32];
            float lsum = 0.f;
            if (j == 0) {
                m_ref = max_pass(kvalid) * sl2;              // the first tile seeds the reference with its exact maximum
                if (kvalid >= KT) exp_pass(w, lsum); else exp_pass_masked(kvalid, w, lsum);
            } else {
                bool need;
                if (kvalid >= KT) {
                    const uint32_t mw = exp_pass(w, lsum);   // optimistic pass against the running reference
                    need = (mw & 0xffffu) > 0x4380u || (mw >> 16) > 0x4380u;          // some P above 2^8 (bf16 256.0 = 0x4380)
                } else {
                    need = max_pass(kvalid) * sl2 - m_ref > 8.0f;
                    if (!__any_sync(0xffffffffu, need)) exp_pass_masked(kvalid, w, lsum);
                }
                if (__any_sync(0xffffffffu, need)) {
                    const float m_new = fmaxf(m_ref, max_pass(kvalid) * sl2);
                    const float alpha = fast_exp2(m_ref - m_new);
#pragma unroll 1
                    for (int c = 0; c < 2; ++c) {
                        uint32_t v[32];
                        tmem_ld32(tO + lane_off + c * 32, v);
                        tc_wait_ld();
#pragma unroll
                        for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * alpha);
                        tmem_st32(tO + lane_off + c * 32, v);
                        tc_wait_st();
                    }
                    l *= alpha;
                    m_ref = m_new;
                    if (kvalid >= KT) exp_pass(w, lsum); else exp_pass_masked(kvalid, w, lsum);     // S is still intact: P again, new reference
                }
            }
            l += lsum;
            // P(j) over the front of this thread's own score row: words [0, 32)
            tmem_st32(tS + lane_off, w);
            tc_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(p_ready);             // one arrival per warp: 32 same-address arrivals serialise in the MIO pipe
        }
        mbar_wait(o_ready, 0);
        tc_fence_after();
        const int q = q0 + r;
        const float inv_l = 1.0f / l;
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
            uint32_t v[32];
            tmem_ld32(tO + lane_off + c * 32, v);
            tc_wait_ld();
            if (q < P.Tq) {
                __nv_bfloat16* dst = P.O + ((long long)b * P.Tq + q) * P.ldo + h * HD + c * 32;
#pragma unroll
                for (int e = 0; e < 32; e += 8) {
                    uint4 o;
                    o.x = pack_bf16(__uint_as_float(v[e]) * inv_l, __uint_as_float(v[e + 1]) * inv_l);
                    o.y = pack_bf16(__uint_as_float(v[e + 2]) * inv_l, __uint_as_float(v[e + 3]) * inv_l);
                    o.z = pack_bf16(__uint_as_float(v[e + 4]) * inv_l, __uint_as_float(v[e + 5]) * inv_l);
                    o.w = pack_bf16(__uint_as_float(v[e + 6]) * inv_l, __uint_as_float(v[e + 7]) * inv_l);
                    *reinterpret_cast<uint4*>(dst + e) = o;
                }
            }
        }
        if (q < P.Tq) P.lse[((long long)b * P.H + h) * P.Tq + q] = (m_ref + log2f(l)) * LN2;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) { tc_fence_after(); tmem_dealloc(tmem, 128); }
}

// ================================================================================================
// backward preprocess: D[b,h,q] = sum_d dO * O
// ================================================================================================
// 8 lanes per (token, head) row: each lane multiplies 8 elements (one 16-byte load of O and of dO), three shuffles sum
// the row; a warp covers 4 rows = 512 contiguous bytes per tensor when the heads are adjacent
__global__ void __launch_bounds__(256)
attn_bwd_prep_kernel(const __nv_bfloat16* __restrict__ O, long long ldo, const __nv_bfloat16* __restrict__ dO,
                     long long lddo, int B, int H, int Tq, float* __restrict__ D, const float* __restrict__ lse = nullptr,
                     float* __restrict__ lse2 = nullptr, float4* __restrict__ zero = nullptr, long long zero_n4 = 0) {
    pdl_enter();
    // the one-kernel backward's fp32 accumulation tiles are cleared here (saves a memset node per attention layer)
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < zero_n4; i += (long long)gridDim.x * blockDim.x)
        zero[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    const long long total = (long long)B * Tq * H * 8;                    // one work item = 8 elements of one row
    const long long bound = (total + 31) & ~31LL;                         // whole warps stay in the loop (full-mask shuffles)
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < bound; i += (long long)gridDim.x * blockDim.x) {
        const long long w = i >> 3;                                       // (token, head) row; whole 8-lane groups stay together
        const int part = (int)(i & 7);
        float s = 0.f;
        int h = 0, t = 0, b = 0;
        if (w < (long long)B * Tq * H) {
            h = (int)(w % H);
            const long long bt = w / H;
            t = (int)(bt % Tq); b = (int)(bt / Tq);
            const uint4 o4 = ld_stream(O + bt * ldo + h * HD + part * 8);
            const uint4 d4 = ld_stream(dO + bt * lddo + h * HD + part * 8);
            const uint32_t ow[4] = {o4.x, o4.y, o4.z, o4.w}, dw[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) s += bf16lo(ow[e]) * bf16lo(dw[e]) + bf16hi(ow[e]) * bf16hi(dw[e]);
        }
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        if (part == 0 && w < (long long)B * Tq * H) {
            const long long idx = ((long long)b * H + h) * Tq + t;
            D[idx] = s;
            if (lse2 != nullptr) lse2[idx] = lse[idx] * LOG2E;              // the one-kernel backward works in the log2 domain
        }
    }
}

// ================================================================================================
// backward: dK, dV  (CTA = one KV tile; loop over Q tiles)
// ================================================================================================
// Ring depth of the streamed operand tiles in the backward kernels.  A slot is refilled only after the accumulating MMAs of
// the tile that used it have retired, and a TMA round trip is ~2000 cycles: with 2 slots the score MMAs of tile i+1
// waited for their operands every iteration (20 % of the dQ kernel's samples at s_ready, ncu r01); 3 slots hide it.
constexpr int BWD_STAGES = 3;

struct KvSmem {
    static constexpr int K = 0;
    static constexpr int V = K + TILE_BYTES;
    static constexpr int Q = V + TILE_BYTES;             // BWD_STAGES stages
    static constexpr int DO = Q + BWD_STAGES * TILE_BYTES;   // BWD_STAGES stages
    static constexpr int PT = DO + BWD_STAGES * TILE_BYTES;  // 32 KB
    static constexpr int DST = PT + 2 * TILE_BYTES;      // 32 KB
    static constexpr int VEC = DST + 2 * TILE_BYTES;     // lse2[2][128], D[2][128] floats
    static constexpr int BAR = VEC + 2048;
    static constexpr int TOTAL = BAR + 256 + 1024;
};

// [128 q, 128 k] bf16 tile (two 64-column blocks, 16 KB apart) read as an MN-major A operand: contraction over its ROWS
// (queries), M = its 128 columns (keys).  k16 selects 16 query rows.
__device__ __forceinline__ uint64_t desc_ptile_rows_as_k(uint32_t p_addr, int k16) {
    return make_sdesc_sw128(p_addr + k16 * 2048, TILE_BYTES, 1024);
}

// Scores are computed query-major here exactly as in the dQ kernel (S = Q K^T, dP = dO V^T: one thread = one query row, its
// LSE and D are two registers), and P / dS are written once as [q, k] tiles; dV += P^T dO and dK += dS^T Q then read those
// tiles as MN-major A operands (contraction over the query rows), so no transposed score tile, no per-column LSE / D
// broadcast loads and no per-tile block barrier are needed.
__global__ void __launch_bounds__(ATT_BWD_THREADS, 1)
attn_bwd_dkv_kernel(const __grid_constant__ AttnParams P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + KvSmem::BAR);
    uint64_t* kv_once = bars;           // 1
    uint64_t* q_full = bars + 1;        // BWD_STAGES
    uint64_t* q_empty = bars + 5;       // BWD_STAGES
    uint64_t* s_ready = bars + 9;
    uint64_t* pds_ready = bars + 10;
    uint64_t* acc_ready = bars + 11;
    uint64_t* st_free = bars + 12;      // compute warps have moved S / dP into registers: next tile's MMAs may overwrite TMEM
    uint64_t* pd_free = bars + 13;      // dV / dK MMAs that read the P / dS smem tiles have completed
    uint32_t* tmem_slot = (uint32_t*)(bars + 14);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kv_tiles = (P.Tk + TILE - 1) / TILE;
    const int kt = blockIdx.x % kv_tiles;
    const int bh = blockIdx.x / kv_tiles;
    const int h = bh % P.H, b = bh / P.H;
    const int k0 = kt * TILE;
    const int nq = (P.Tq + TILE - 1) / TILE;

    if (threadIdx.x == 0) {
        mbar_init(kv_once, 1);
        for (int i = 0; i < BWD_STAGES; ++i) { mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1); }
        mbar_init(s_ready, 1); mbar_init(pds_ready, BWD_CT); mbar_init(acc_ready, 1);
        mbar_init(st_free, BWD_CT); mbar_init(pd_free, 1);
        fence_mbar_init();
    }
    if (warp == BWD_CW + 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tS = tmem, tdP = tmem + 128, tdV = tmem + 256, tdK = tmem + 320;
    pdl_enter();          // prologue done: wait for the previous kernel's results before the first global access

    if (warp == BWD_CW) {
        if (lane == 0) {
            tma_prefetch_desc(&P.tmQ); tma_prefetch_desc(&P.tmK); tma_prefetch_desc(&P.tmV); tma_prefetch_desc(&P.tmDO);
            mbar_arrive_expect_tx(kv_once, 2 * TILE_BYTES);
            tma_load_4d(smem + KvSmem::K, &P.tmK, kv_once, 0, h, k0, b);
            tma_load_4d(smem + KvSmem::V, &P.tmV, kv_once, 0, h, k0, b);
            for (int i = 0; i < nq; ++i) {
                const int s = i % BWD_STAGES;
                mbar_wait(&q_empty[s], ((i / BWD_STAGES) & 1) ^ 1);
                mbar_arrive_expect_tx(&q_full[s], 2 * TILE_BYTES);
                tma_load_4d(smem + KvSmem::Q + s * TILE_BYTES, &P.tmQ, &q_full[s], 0, h, i * TILE, b);
                tma_load_4d(smem + KvSmem::DO + s * TILE_BYTES, &P.tmDO, &q_full[s], 0, h, i * TILE, b);
            }
        }
    } else if (warp == BWD_CW + 1) {
        // Software pipeline: S / dP of Q tile i+1 are issued as soon as the compute warps have pulled tile i's S / dP into
        // registers, so the tensor pipe works on tile i+1 while they do the exp / dS math of tile i.
        // The whole warp runs the loop converged and one elected lane issues (see elect_one_sync in common.cuh); descriptors are the
        // stage-0 descriptors plus integer offsets on the address field (16-byte units).
        const uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);
        const uint32_t idesc_acc = make_idesc_bf16(128, 64, 1, 1);           // A = P / dS read MN-major, B = dO / Q read MN-major
        const uint64_t dK_k = desc_kmajor(smem_u32(smem + KvSmem::K), 0), dV_k = desc_kmajor(smem_u32(smem + KvSmem::V), 0);
        const uint64_t dQ_k = desc_kmajor(smem_u32(smem + KvSmem::Q), 0), dDO_k = desc_kmajor(smem_u32(smem + KvSmem::DO), 0);
        const uint64_t dQ_r = desc_rows_as_k(smem_u32(smem + KvSmem::Q), 0), dDO_r = desc_rows_as_k(smem_u32(smem + KvSmem::DO), 0);
        const uint64_t dP_r = desc_ptile_rows_as_k(smem_u32(smem + KvSmem::PT), 0), dDS_r = desc_ptile_rows_as_k(smem_u32(smem + KvSmem::DST), 0);
        constexpr uint64_t STG = TILE_BYTES >> 4;
        auto issue_scores = [&](int i) {
            const int s = i % BWD_STAGES;
            mbar_wait(&q_full[s], (i / BWD_STAGES) & 1);
            tc_fence_after();
            if (elect_one_sync()) {
                const uint64_t q = dQ_k + s * STG, d = dDO_k + s * STG;
                umma_bf16(tS, q, dK_k, idesc_s, 0u);
#pragma unroll
                for (int k = 1; k < 4; ++k) umma_bf16(tS, q + 2 * k, dK_k + 2 * k, idesc_s, 1u);
                umma_bf16(tdP, d, dV_k, idesc_s, 0u);
#pragma unroll
                for (int k = 1; k < 4; ++k) umma_bf16(tdP, d + 2 * k, dV_k + 2 * k, idesc_s, 1u);
                umma_commit(s_ready);
            }
            __syncwarp();
        };
        mbar_wait(kv_once, 0);
        issue_scores(0);
        for (int i = 0; i < nq; ++i) {
            const int s = i % BWD_STAGES;
            if (i + 1 < nq) {
                mbar_wait(st_free, i & 1);
                tc_fence_after();
                issue_scores(i + 1);
            }
            mbar_wait(pds_ready, i & 1);
            tc_fence_after();
            if (elect_one_sync()) {
                const uint64_t q = dQ_r + s * STG, d = dDO_r + s * STG;
                const uint32_t acc = i > 0 ? 1u : 0u;
                umma_bf16(tdV, dP_r, d, idesc_acc, acc);
#pragma unroll
                for (int k = 1; k < 8; ++k) umma_bf16(tdV, dP_r + 128 * k, d + 128 * k, idesc_acc, 1u);
                umma_bf16(tdK, dDS_r, q, idesc_acc, acc);
#pragma unroll
                for (int k = 1; k < 8; ++k) umma_bf16(tdK, dDS_r + 128 * k, q + 128 * k, idesc_acc, 1u);
                umma_commit(&q_empty[s]);
                umma_commit(pd_free);
                if (i == nq - 1) umma_commit(acc_ready);
            }
            __syncwarp();
        }
    } else {
        // compute warps: quarter = warp & 3 (TMEM lanes = query rows), hf = warp >> 2 selects 32 of the tile's 128 key columns
        const int qtr = warp & 3, hf = warp >> 2;
        const int r = qtr * 32 + lane;                       // query row inside the tile
        const uint32_t lane_off = (uint32_t)(qtr * 32) << 16;
        const uint32_t sP = smem_u32(smem + KvSmem::PT), sDS = smem_u32(smem + KvSmem::DST);
        const float sl2 = P.scale * LOG2E;
        const int kvalid = P.Tk - k0;                        // keys >= kvalid of this tile are padding
        // per-query LSE / D of the NEXT Q tile are fetched one tile ahead (their global-load latency hides behind this tile's math)
        float nx_lse = INFINITY, nx_d = 0.f;
        auto fetch_vec = [&](int i) {
            const int q = i * TILE + r;
            const long long idx = ((long long)b * P.H + h) * P.Tq + q;
            nx_lse = q < P.Tq ? P.lse[idx] : INFINITY;       // +inf -> P = 0 for padded queries
            nx_d = q < P.Tq ? P.Dvec[idx] : 0.f;
        };
        fetch_vec(0);
        for (int i = 0; i < nq; ++i) {
            const float lse2 = nx_lse * LOG2E, dvec = nx_d;
            if (i + 1 < nq) fetch_vec(i + 1);
            mbar_wait(s_ready, i & 1);
            tc_fence_after();
            // two 16-column chunks, software-pipelined: the tcgen05.ld of chunk 1 is in flight during chunk 0's math
            uint32_t vs[2][16], vp[2][16], hp[2][8], hd[2][8];
            tmem_ld16(tS + lane_off + hf * 32, vs[0]);
            tmem_ld16(tdP + lane_off + hf * 32, vp[0]);
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                tc_wait_ld();
                if (c + 1 < 2) {
                    tmem_ld16(tS + lane_off + hf * 32 + (c + 1) * 16, vs[(c + 1) & 1]);
                    tmem_ld16(tdP + lane_off + hf * 32 + (c + 1) * 16, vp[(c + 1) & 1]);
                } else {
                    tc_fence_before();
                    mbar_arrive(st_free);                    // TMEM S / dP may be overwritten by the next tile's MMAs
                }
                uint32_t* wp = hp[c & 1];
                uint32_t* wd = hd[c & 1];
                const uint32_t* cs = vs[c & 1];
                const uint32_t* cp = vp[c & 1];
                if (kvalid >= TILE) {
#pragma unroll
                    for (int e = 0; e < 16; e += 2) {
                        const float p0 = fast_exp2(fmaf(__uint_as_float(cs[e]), sl2, -lse2));
                        const float p1 = fast_exp2(fmaf(__uint_as_float(cs[e + 1]), sl2, -lse2));
                        wp[e >> 1] = pack_bf16(p0, p1);
                        wd[e >> 1] = pack_bf16(p0 * (__uint_as_float(cp[e]) - dvec), p1 * (__uint_as_float(cp[e + 1]) - dvec));
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < 16; e += 2) {
                        const int ka = hf * 32 + c * 16 + e;
                        const float p0 = (ka < kvalid) ? fast_exp2(fmaf(__uint_as_float(cs[e]), sl2, -lse2)) : 0.f;
                        const float p1 = (ka + 1 < kvalid) ? fast_exp2(fmaf(__uint_as_float(cs[e + 1]), sl2, -lse2)) : 0.f;
                        wp[e >> 1] = pack_bf16(p0, p1);
                        wd[e >> 1] = pack_bf16(p0 * (__uint_as_float(cp[e]) - dvec), p1 * (__uint_as_float(cp[e + 1]) - dvec));
                    }
                }
                // chunk 0 waits in registers: the previous tile's dV / dK MMAs (issued when that tile's P / dS were complete)
                // still read these smem tiles for the first few hundred cycles of this tile
                if (c == 1) {
                    if (i > 0) mbar_wait(pd_free, (i - 1) & 1);
                    store_p_16(sP, r, hf * 32, hp[0]);
                    store_p_16(sDS, r, hf * 32, hd[0]);
                    store_p_16(sP, r, hf * 32 + 16, hp[1]);
                    store_p_16(sDS, r, hf * 32 + 16, hd[1]);
                }
            }
            fence_proxy_async_smem();
            tc_fence_before();
            mbar_arrive(pds_ready);
        }
        mbar_wait(acc_ready, 0);
        tc_fence_after();
        const int key = k0 + r;                              // accumulator rows are keys
        {
            const int which = hf >> 1, c = hf & 1;               // warps hf 0,1 store dV chunks 0,1; hf 2,3 store dK chunks 0,1
            const uint32_t tacc = which == 0 ? tdV : tdK;
            const float mul = which == 0 ? 1.0f : P.scale;
            __nv_bfloat16* base = which == 0 ? P.dV : P.dK;
            const long long ld = which == 0 ? P.lddv : P.lddk;
            uint32_t v[32];
            tmem_ld32(tacc + lane_off + c * 32, v);
            tc_wait_ld();
            if (key < P.Tk) {
                __nv_bfloat16* dst = base + ((long long)b * P.Tk + key) * ld + h * HD + c * 32;
#pragma unroll
                for (int e = 0; e < 32; e += 8) {
                    uint4 o;
                    o.x = pack_bf16(__uint_as_float(v[e]) * mul, __uint_as_float(v[e + 1]) * mul);
                    o.y = pack_bf16(__uint_as_float(v[e + 2]) * mul, __uint_as_float(v[e + 3]) * mul);
                    o.z = pack_bf16(__uint_as_float(v[e + 4]) * mul, __uint_as_float(v[e + 5]) * mul);
                    o.w = pack_bf16(__uint_as_float(v[e + 6]) * mul, __uint_as_float(v[e + 7]) * mul);
                    *reinterpret_cast<uint4*>(dst + e) = o;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == BWD_CW + 1) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// ================================================================================================
// backward: dQ  (CTA = one Q tile; loop over KV tiles)
// ================================================================================================
struct DqSmem {
    static constexpr int Q = 0;
    static constexpr int DO = Q + TILE_BYTES;
    static constexpr int K = DO + TILE_BYTES;            // BWD_STAGES stages
    static constexpr int V = K + BWD_STAGES * TILE_BYTES;    // BWD_STAGES stages
    static constexpr int DS = V + BWD_STAGES * TILE_BYTES;   // 32 KB
    static constexpr int BAR = DS + 2 * TILE_BYTES;
    static constexpr int TOTAL = BAR + 256 + 1024;
};

__global__ void __launch_bounds__(ATT_BWD_THREADS, 1)
attn_bwd_dq_kernel(const __grid_constant__ AttnParams P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + DqSmem::BAR);
    uint64_t* q_once = bars;
    uint64_t* kv_full = bars + 1;       // BWD_STAGES
    uint64_t* kv_empty = bars + 5;      // BWD_STAGES
    uint64_t* s_ready = bars + 9;
    uint64_t* ds_ready = bars + 10;
    uint64_t* acc_ready = bars + 11;
    uint64_t* st_free = bars + 12;
    uint64_t* ds_free = bars + 13;
    uint32_t* tmem_slot = (uint32_t*)(bars + 14);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q_tiles = (P.Tq + TILE - 1) / TILE;
    const int qt = blockIdx.x % q_tiles;
    const int bh = blockIdx.x / q_tiles;
    const int h = bh % P.H, b = bh / P.H;
    const int q0 = qt * TILE;
    const int nkv = (P.Tk + TILE - 1) / TILE;

    if (threadIdx.x == 0) {
        mbar_init(q_once, 1);
        for (int i = 0; i < BWD_STAGES; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], 1); }
        mbar_init(s_ready, 1); mbar_init(ds_ready, BWD_CT); mbar_init(acc_ready, 1);
        mbar_init(st_free, BWD_CT); mbar_init(ds_free, 1);
        fence_mbar_init();
    }
    if (warp == BWD_CW + 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tS = tmem, tdP = tmem + 128, tdQ = tmem + 256;
    pdl_enter();          // prologue done: wait for the previous kernel's results before the first global access

    if (warp == BWD_CW) {
        if (lane == 0) {
            tma_prefetch_desc(&P.tmQ); tma_prefetch_desc(&P.tmK); tma_prefetch_desc(&P.tmV); tma_prefetch_desc(&P.tmDO);
            mbar_arrive_expect_tx(q_once, 2 * TILE_BYTES);
            tma_load_4d(smem + DqSmem::Q, &P.tmQ, q_once, 0, h, q0, b);
            tma_load_4d(smem + DqSmem::DO, &P.tmDO, q_once, 0, h, q0, b);
            for (int j = 0; j < nkv; ++j) {
                const int s = j % BWD_STAGES;
                mbar_wait(&kv_empty[s], ((j / BWD_STAGES) & 1) ^ 1);
                mbar_arrive_expect_tx(&kv_full[s], 2 * TILE_BYTES);
                tma_load_4d(smem + DqSmem::K + s * TILE_BYTES, &P.tmK, &kv_full[s], 0, h, j * TILE, b);
                tma_load_4d(smem + DqSmem::V + s * TILE_BYTES, &P.tmV, &kv_full[s], 0, h, j * TILE, b);
            }
        }
    } else if (warp == BWD_CW + 1) {
        // converged warp, one elected lane issues (see elect_one_sync in common.cuh)
        const uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);
        const uint32_t idesc_acc = make_idesc_bf16(128, 64, 0, 1);
        const uint64_t dQ_k = desc_kmajor(smem_u32(smem + DqSmem::Q), 0), dDO_k = desc_kmajor(smem_u32(smem + DqSmem::DO), 0);
        const uint64_t dK_k = desc_kmajor(smem_u32(smem + DqSmem::K), 0), dV_k = desc_kmajor(smem_u32(smem + DqSmem::V), 0);
        const uint64_t dK_r = desc_rows_as_k(smem_u32(smem + DqSmem::K), 0);
        const uint32_t sDS = smem_u32(smem + DqSmem::DS);
        constexpr uint64_t STG = TILE_BYTES >> 4;
        auto issue_scores = [&](int j) {
            const int s = j % BWD_STAGES;
            mbar_wait(&kv_full[s], (j / BWD_STAGES) & 1);
            tc_fence_after();
            if (elect_one_sync()) {
                const uint64_t kk = dK_k + s * STG, vv = dV_k + s * STG;
                umma_bf16(tS, dQ_k, kk, idesc_s, 0u);
#pragma unroll
                for (int k = 1; k < 4; ++k) umma_bf16(tS, dQ_k + 2 * k, kk + 2 * k, idesc_s, 1u);
                umma_bf16(tdP, dDO_k, vv, idesc_s, 0u);
#pragma unroll
                for (int k = 1; k < 4; ++k) umma_bf16(tdP, dDO_k + 2 * k, vv + 2 * k, idesc_s, 1u);
                umma_commit(s_ready);
            }
            __syncwarp();
        };
        mbar_wait(q_once, 0);
        issue_scores(0);
        for (int j = 0; j < nkv; ++j) {
            const int s = j % BWD_STAGES;
            if (j + 1 < nkv) {
                mbar_wait(st_free, j & 1);
                tc_fence_after();
                issue_scores(j + 1);
            }
            mbar_wait(ds_ready, j & 1);
            tc_fence_after();
            if (elect_one_sync()) {
                const uint64_t kr = dK_r + s * STG;
                umma_bf16(tdQ, desc_ptile(sDS, 0), kr, idesc_acc, j > 0 ? 1u : 0u);
#pragma unroll
                for (int k = 1; k < 8; ++k) umma_bf16(tdQ, desc_ptile(sDS, k), kr + 128 * k, idesc_acc, 1u);
                umma_commit(&kv_empty[s]);
                umma_commit(ds_free);
                if (j == nkv - 1) umma_commit(acc_ready);
            }
            __syncwarp();
        }
    } else {
        const int qtr = warp & 3, hf = warp >> 2;            // four warps per TMEM lane quarter, each owns 32 key columns
        const int r = qtr * 32 + lane;
        const uint32_t lane_off = (uint32_t)(qtr * 32) << 16;
        const uint32_t sDS = smem_u32(smem + DqSmem::DS);
        const float sl2 = P.scale * LOG2E;
        const int q = q0 + r;
        const long long idx = ((long long)b * P.H + h) * P.Tq + q;
        const float lse2 = q < P.Tq ? P.lse[idx] * LOG2E : INFINITY;
        const float dvec = q < P.Tq ? P.Dvec[idx] : 0.f;
        for (int j = 0; j < nkv; ++j) {
            mbar_wait(s_ready, j & 1);
            tc_fence_after();
            const int kvalid = P.Tk - j * TILE;
            // four 16-column chunks, software-pipelined like the dK/dV kernel
            uint32_t vs[2][16], vp[2][16], hd[2][8];
            tmem_ld16(tS + lane_off + hf * 32, vs[0]);
            tmem_ld16(tdP + lane_off + hf * 32, vp[0]);
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                tc_wait_ld();
                if (c + 1 < 2) {
                    tmem_ld16(tS + lane_off + hf * 32 + (c + 1) * 16, vs[(c + 1) & 1]);
                    tmem_ld16(tdP + lane_off + hf * 32 + (c + 1) * 16, vp[(c + 1) & 1]);
                } else {
                    tc_fence_before();
                    mbar_arrive(st_free);                    // TMEM S / dP may be overwritten by the next tile's MMAs
                }
                uint32_t* wd = hd[c & 1];
                const uint32_t* cs = vs[c & 1];
                const uint32_t* cp = vp[c & 1];
                if (kvalid >= TILE) {
#pragma unroll
                    for (int e = 0; e < 16; e += 2) {
                        const float p0 = fast_exp2(fmaf(__uint_as_float(cs[e]), sl2, -lse2));
                        const float p1 = fast_exp2(fmaf(__uint_as_float(cs[e + 1]), sl2, -lse2));
                        wd[e >> 1] = pack_bf16(p0 * (__uint_as_float(cp[e]) - dvec), p1 * (__uint_as_float(cp[e + 1]) - dvec));
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < 16; e += 2) {
                        const int ka = hf * 32 + c * 16 + e;
                        float p0 = (ka < kvalid) ? fast_exp2(fmaf(__uint_as_float(cs[e]), sl2, -lse2)) : 0.f;
                        float p1 = (ka + 1 < kvalid) ? fast_exp2(fmaf(__uint_as_float(cs[e + 1]), sl2, -lse2)) : 0.f;
                        wd[e >> 1] = pack_bf16(p0 * (__uint_as_float(cp[e]) - dvec), p1 * (__uint_as_float(cp[e + 1]) - dvec));
                    }
                }
                if (c == 1) {                                // see the dK/dV kernel: the previous tile's dQ MMAs still read sDS
                    if (j > 0) mbar_wait(ds_free, (j - 1) & 1);
                    store_p_16(sDS, r, hf * 32, hd[0]);
                    store_p_16(sDS, r, hf * 32 + 16, hd[1]);
                }
            }
            fence_proxy_async_smem();
            tc_fence_before();
            mbar_arrive(ds_ready);
        }
        mbar_wait(acc_ready, 0);
        tc_fence_after();
        {
            uint32_t v[16];                                      // each of the four warps of a lane quarter stores 16 of the 64 columns
            tmem_ld16(tdQ + lane_off + hf * 16, v);
            tc_wait_ld();
            if (q < P.Tq) {
                __nv_bfloat16* dst = P.dQ + ((long long)b * P.Tq + q) * P.lddq + h * HD + hf * 16;
                const float mul = P.scale;
#pragma unroll
                for (int e = 0; e < 16; e += 8) {
                    uint4 o;
                    o.x = pack_bf16(__uint_as_float(v[e]) * mul, __uint_as_float(v[e + 1]) * mul);
                    o.y = pack_bf16(__uint_as_float(v[e + 2]) * mul, __uint_as_float(v[e + 3]) * mul);
                    o.z = pack_bf16(__uint_as_float(v[e + 4]) * mul, __uint_as_float(v[e + 5]) * mul);
                    o.w = pack_bf16(__uint_as_float(v[e + 6]) * mul, __uint_as_float(v[e + 7]) * mul);
                    *reinterpret_cast<uint4*>(dst + e) = o;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == BWD_CW + 1) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// ================================================================================================
// backward, ONE kernel: dK, dV and dQ  (CTA = one KV tile of 128 keys; loop over Q tiles)
// ================================================================================================
// Five MMAs and ONE exponential pass per (Q tile, KV tile) pair instead of the seven MMAs and two passes of the dK/dV + dQ pair.
// Scores are computed KEY-major (S^T = K Q^T, dP^T = V dO^T: a thread owns one key row), so that P^T and dS^T -- written back over
// the front of the thread's own S^T / dP^T columns as packed bf16 (tcgen05.st) -- are the K-major A operands of dV += P^T dO and
// dK += dS^T Q straight from TENSOR MEMORY: no shared-memory P tile, no proxy fence for it.  dS^T additionally goes to shared
// memory once, as the MN-major A operand of dQ(i) = dS(i) K.  dQ(i) is only this KV tile's share: it is double-buffered in TMEM,
// drained by four dedicated warps into a shared-memory staging tile and added into an fp32 buffer by ONE bulk reduction per tile
// (cp.reduce.async.bulk .add.f32, 32 KB, issued by the TMA engine: no per-thread atomics on the load/store path -- the per-thread
// red.global form measured SLOWER than two kernels, profiles/r02_attn_bwd_notes.txt).  attn_dq_tiles_convert_kernel then scales and
// rounds.  The sum over KV tiles is not bit-reproducible (aoz_attn_set_bwd_mode(0) selects the two-kernel form).
//
// Tensor memory (512 columns): S^T | dP^T | dV | dK | dQ0 | dQ1.  The tensor pipe runs half a tile ahead of the compute warps:
//   issuer:  ... dV(i) S^T(i+1) | dK(i) dQ(i) dP^T(i+1) | dV(i+1) S^T(i+2) | ...
//   compute: ... exp phase (i)  ->  dS phase (i)        ->  exp phase (i+1) ...
// S^T(i+1) overwrites P^T(i) and dP^T(i+1) overwrites dS^T(i): both are queued behind the MMAs that read them (in-order pipe).
constexpr int FB_CW = 16;                                   // compute warps
constexpr int FB_THREADS = (FB_CW + 2 + 4) * 32;            // + producer + issuer + 4 drain warps (one per TMEM lane quarter)
constexpr int FB_STAGES = 3;                                // Q / dO / lse2 / D ring

struct FbSmem {
    static constexpr int K = 0;
    static constexpr int V = K + TILE_BYTES;
    static constexpr int Q = V + TILE_BYTES;                      // FB_STAGES
    static constexpr int DO = Q + FB_STAGES * TILE_BYTES;         // FB_STAGES
    static constexpr int DST = DO + FB_STAGES * TILE_BYTES;       // 32 KB: dS^T [128 keys][128 queries] bf16, two 64-query blocks
    static constexpr int DQS = DST + 2 * TILE_BYTES;              // 32 KB: dQ staging tile [128 queries][64] fp32, 16-byte chunks XOR-swizzled
    static constexpr int VEC = DQS + 2 * TILE_BYTES;              // FB_STAGES x (lse2[128], D[128]) fp32
    static constexpr int BAR = VEC + FB_STAGES * 1024;
    static constexpr int TOTAL = BAR + 256 + 1024;
};
static_assert(FbSmem::TOTAL <= 227 * 1024, "one-kernel attention backward: shared memory");

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void bulk_reduce_add_f32(float* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;"
                 :: "l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__global__ void __launch_bounds__(FB_THREADS, 1)
attn_bwd_fused_kernel(const __grid_constant__ AttnParams P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + FbSmem::BAR);
    uint64_t* kv_once = bars;                 // 1
    uint64_t* q_full = bars + 1;              // FB_STAGES
    uint64_t* q_empty = bars + 4;             // FB_STAGES
    uint64_t* s_ready = bars + 7;             // S^T(i) landed
    uint64_t* dp_ready = bars + 8;            // dP^T(i) landed
    uint64_t* p_ready = bars + 9;             // P^T(i) in tensor memory (512 arrivals)
    uint64_t* ds_ready = bars + 10;           // dS^T(i) in tensor memory and shared memory (512 arrivals)
    uint64_t* ds_free = bars + 11;            // dQ(i) has retired: the shared dS^T tile may be overwritten
    uint64_t* dq_ready = bars + 12;           // 2: dQ(i) landed in buffer i & 1
    uint64_t* dq_free = bars + 14;            // 2: the drain warps have read buffer i & 1 (128 arrivals)
    uint64_t* acc_ready = bars + 16;
    uint32_t* tmem_slot = (uint32_t*)(bars + 17);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kv_tiles = (P.Tk + TILE - 1) / TILE;
    const int qs = blockIdx.x % P.q_split;                  // which share of the Q tiles
    const int kt = (blockIdx.x / P.q_split) % kv_tiles;
    const int bh = blockIdx.x / (P.q_split * kv_tiles);
    const int h = bh % P.H, b = bh / P.H;
    const int k0 = kt * TILE;
    const int q_tiles = (P.Tq + TILE - 1) / TILE;
    const int per = (q_tiles + P.q_split - 1) / P.q_split;
    const int i0 = qs * per;                                // this CTA's Q tiles: i0 .. i0 + nq - 1 (loop index i is LOCAL below)
    const int nq = max(0, min(per, q_tiles - i0));

    if (threadIdx.x == 0) {
        mbar_init(kv_once, 1);
        for (int i = 0; i < FB_STAGES; ++i) { mbar_init(&q_full[i], 1); mbar_init(&q_empty[i], 1); }
        mbar_init(s_ready, 1); mbar_init(dp_ready, 1); mbar_init(p_ready, FB_CW); mbar_init(ds_ready, FB_CW);          // one arrival per compute warp
        mbar_init(ds_free, 1);
        for (int i = 0; i < 2; ++i) { mbar_init(&dq_ready[i], 1); mbar_init(&dq_free[i], 4); }
        mbar_init(acc_ready, 1);
        fence_mbar_init();
    }
    if (warp == FB_CW + 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tS = tmem, tdP = tmem + 128, tdV = tmem + 256, tdK = tmem + 320, tdQ = tmem + 384;     // dQ buffers: +384, +448
    pdl_enter();          // prologue done: wait for the previous kernel's results before the first global access
    const long long vec0 = ((long long)b * P.H + h) * P.Tq;          // first element of this (b, h) in lse2 / D

    if (warp == FB_CW) {
        // ---------------- TMA producer ----------------
        if (lane == 0) {
            tma_prefetch_desc(&P.tmQ); tma_prefetch_desc(&P.tmK); tma_prefetch_desc(&P.tmV); tma_prefetch_desc(&P.tmDO);
            mbar_arrive_expect_tx(kv_once, 2 * TILE_BYTES);
            tma_load_4d(smem + FbSmem::K, &P.tmK, kv_once, 0, h, k0, b);
            tma_load_4d(smem + FbSmem::V, &P.tmV, kv_once, 0, h, k0, b);
            for (int i = 0; i < nq; ++i) {
                const int s = i % FB_STAGES;
                mbar_wait_relaxed(&q_empty[s], ((i / FB_STAGES) & 1) ^ 1);
                const int qrow = (i0 + i) * TILE;
                const int rows = min(TILE, P.Tq - qrow);                       // Tq is a multiple of 4 here: 16-byte granules
                mbar_arrive_expect_tx(&q_full[s], 2 * TILE_BYTES + 2 * rows * 4);
                tma_load_4d(smem + FbSmem::Q + s * TILE_BYTES, &P.tmQ, &q_full[s], 0, h, qrow, b);
                tma_load_4d(smem + FbSmem::DO + s * TILE_BYTES, &P.tmDO, &q_full[s], 0, h, qrow, b);
                bulk_load_1d(smem + FbSmem::VEC + s * 1024, P.lse + vec0 + qrow, rows * 4, &q_full[s]);          // lse * log2(e)
                bulk_load_1d(smem + FbSmem::VEC + s * 1024 + 512, P.Dvec + vec0 + qrow, rows * 4, &q_full[s]);
            }
        }
    } else if (warp == FB_CW + 1) {
        // ---------------- MMA issuer: converged warp, one elected lane issues (see elect_one_sync) ----------------
        const uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);
        const uint32_t idesc_ts = make_idesc_bf16(128, 64, 0, 1);            // A = P^T / dS^T from tensor memory, B = dO / Q rows as K
        const uint32_t idesc_dq = make_idesc_bf16(128, 64, 1, 1);            // A = dS^T tile in smem read MN-major, B = K rows as K
        const uint64_t dK_k = desc_kmajor(smem_u32(smem + FbSmem::K), 0), dV_k = desc_kmajor(smem_u32(smem + FbSmem::V), 0);
        const uint64_t dQ_k = desc_kmajor(smem_u32(smem + FbSmem::Q), 0), dDO_k = desc_kmajor(smem_u32(smem + FbSmem::DO), 0);
        const uint64_t dQ_r = desc_rows_as_k(smem_u32(smem + FbSmem::Q), 0), dDO_r = desc_rows_as_k(smem_u32(smem + FbSmem::DO), 0);
        const uint64_t dK_r = desc_rows_as_k(smem_u32(smem + FbSmem::K), 0);
        const uint64_t dDS_r = desc_ptile_rows_as_k(smem_u32(smem + FbSmem::DST), 0);
        constexpr uint64_t STG = TILE_BYTES >> 4;
        auto issue_st = [&](int i) {                                            // S^T(i) = K Q(i)^T
            const int s = i % FB_STAGES;
            mbar_wait(&q_full[s], (i / FB_STAGES) & 1);
            tc_fence_after();
            if (elect_one_sync()) {
                const uint64_t q = dQ_k + s * STG;
                umma_bf16(tS, dK_k, q, idesc_s, 0u);
#pragma unroll
                for (int k = 1; k < 4; ++k) umma_bf16(tS, dK_k + 2 * k, q + 2 * k, idesc_s, 1u);
                umma_commit(s_ready);
            }
            __syncwarp();
        };
        auto issue_dpt = [&](int i) {                                           // dP^T(i) = V dO(i)^T  (its stage was awaited by issue_st)
            const int s = i % FB_STAGES;
            if (elect_one_sync()) {
                const uint64_t d = dDO_k + s * STG;
                umma_bf16(tdP, dV_k, d, idesc_s, 0u);
#pragma unroll
                for (int k = 1; k < 4; ++k) umma_bf16(tdP, dV_k + 2 * k, d + 2 * k, idesc_s, 1u);
                umma_commit(dp_ready);
            }
            __syncwarp();
        };
        mbar_wait(kv_once, 0);
        if (nq > 0) { issue_st(0); issue_dpt(0); }
        for (int i = 0; i < nq; ++i) {
            const int s = i % FB_STAGES;
            const uint32_t acc = i > 0 ? 1u : 0u;
            mbar_wait(p_ready, i & 1);
            tc_fence_after();
            if (elect_one_sync()) {                                             // dV += P^T(i) dO(i)
                const uint64_t d = dDO_r + s * STG;
                umma_bf16_ts(tdV, tS, d, idesc_ts, acc);
#pragma unroll
                for (int k = 1; k < 8; ++k) umma_bf16_ts(tdV, tS + 32 * (k >> 1) + 8 * (k & 1), d + 128 * k, idesc_ts, 1u);
            }
            __syncwarp();
            if (i + 1 < nq) issue_st(i + 1);                                    // overwrites P^T(i): queued behind dV(i)
            mbar_wait(ds_ready, i & 1);
            tc_fence_after();
            if (i >= 2) { mbar_wait(&dq_free[i & 1], ((i >> 1) - 1) & 1); tc_fence_after(); }
            if (elect_one_sync()) {
                const uint64_t q = dQ_r + s * STG;                              // dK += dS^T(i) Q(i)
                umma_bf16_ts(tdK, tdP, q, idesc_ts, acc);
#pragma unroll
                for (int k = 1; k < 8; ++k) umma_bf16_ts(tdK, tdP + 32 * (k >> 1) + 8 * (k & 1), q + 128 * k, idesc_ts, 1u);
            }
            __syncwarp();
            if (i + 1 < nq) issue_dpt(i + 1);                                   // overwrites dS^T(i) in TMEM: queued behind dK(i); ahead of
                                                                                // dQ(i), which reads dS from shared memory (dP^T is on the
                                                                                // compute warps' critical path, dQ is not)
            if (elect_one_sync()) {
                const uint32_t tq = tdQ + (i & 1) * 64;                         // dQ(i) = dS(i) K   (this KV tile's share)
                umma_bf16(tq, dDS_r, dK_r, idesc_dq, 0u);
#pragma unroll
                for (int k = 1; k < 8; ++k) umma_bf16(tq, dDS_r + 128 * k, dK_r + 128 * k, idesc_dq, 1u);
                umma_commit(&dq_ready[i & 1]);
                umma_commit(ds_free);
                umma_commit(&q_empty[s]);
                if (i == nq - 1) umma_commit(acc_ready);
            }
            __syncwarp();
        }
    } else if (warp >= FB_CW + 2) {
        // ---------------- dQ drain warps: TMEM -> swizzled staging tile -> one bulk reduce-add per Q tile ----------------
        const int qtr = warp & 3;                                               // warps 18..21 -> lane quarters 2, 3, 0, 1
        const int r = qtr * 32 + lane;                                          // query row inside the tile
        const uint32_t lane_off = (uint32_t)(qtr * 32) << 16;
        const bool leader = warp == FB_CW + 2 && lane == 0;
        uint8_t* stage = smem + FbSmem::DQS;
        float* gtile = P.dQacc + ((long long)bh * q_tiles + i0) * (TILE * HD);
        for (int i = 0; i < nq; ++i) {
            mbar_wait(&dq_ready[i & 1], (i >> 1) & 1);
            tc_fence_after();
            uint32_t v[64];
            tmem_ld32(tdQ + (i & 1) * 64 + lane_off, v);
            tmem_ld32(tdQ + (i & 1) * 64 + lane_off + 32, v + 32);
            tc_wait_ld();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&dq_free[i & 1]);
            if (kv_tiles == 1) {
                // one KV tile: this IS dQ(i) -- scaled, rounded and stored directly (no accumulation buffer, no convert pass)
                const int q = (i0 + i) * TILE + r;
                if (q < P.Tq) {
                    __nv_bfloat16* dst = P.dQ + ((long long)b * P.Tq + q) * P.lddq + h * HD;
                    const float mul = P.scale;
#pragma unroll
                    for (int e = 0; e < 64; e += 8) {
                        uint4 o;
                        o.x = pack_bf16(__uint_as_float(v[e]) * mul, __uint_as_float(v[e + 1]) * mul);
                        o.y = pack_bf16(__uint_as_float(v[e + 2]) * mul, __uint_as_float(v[e + 3]) * mul);
                        o.z = pack_bf16(__uint_as_float(v[e + 4]) * mul, __uint_as_float(v[e + 5]) * mul);
                        o.w = pack_bf16(__uint_as_float(v[e + 6]) * mul, __uint_as_float(v[e + 7]) * mul);
                        *reinterpret_cast<uint4*>(dst + e) = o;
                    }
                }
                continue;
            }
            if (leader) bulk_wait_read0();                                      // the previous tile's reduction has read the staging tile
            named_bar_sync(2, 128);
#pragma unroll
            for (int c = 0; c < 16; ++c)                                        // 16-byte chunk c of row r lives at chunk c ^ (r & 15)
                st_shared_v4(smem_u32(stage) + r * 256 + ((c ^ (r & 15)) << 4), v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
            fence_proxy_async_smem();
            named_bar_sync(2, 128);
            if (leader) bulk_reduce_add_f32(gtile + (long long)i * (TILE * HD), stage, TILE * HD * 4);
        }
        if (leader) bulk_wait_read0();         // shared memory must outlive the reads; the global writes complete with the kernel
    } else {
        // ---------------- compute warps: qtr = TMEM lane quarter (key rows), hf = which 32 of the tile's 128 query columns ----------------
        const int qtr = warp & 3, hf = warp >> 2;
        const int r = qtr * 32 + lane;                                          // key row inside the tile
        const uint32_t lane_off = (uint32_t)(qtr * 32) << 16;
        const uint32_t sDS = smem_u32(smem + FbSmem::DST);
        const float sl2 = P.scale * LOG2E;
        const bool key_ok = k0 + r < P.Tk;                                      // padded key rows contribute nothing
        for (int i = 0; i < nq; ++i) {
            const int s = i % FB_STAGES;
            const uint32_t vec = smem_u32(smem + FbSmem::VEC + s * 1024) + hf * 128;         // lse2[hf * 32 ..], D at + 512
            const int qvalid = P.Tq - (i0 + i) * TILE - hf * 32;                 // this thread's columns >= qvalid are padded queries
            // ---- exp phase: P^T = 2^(S^T sl2 - lse2[q]) ----
            // (lse2 / D of this Q tile arrived with Q: the issuer waited for q_full before the MMAs that s_ready reports)
            mbar_wait(s_ready, i & 1);
            tc_fence_after();
            float p[32];
            {
                uint32_t vs[2][16];
                tmem_ld16(tS + lane_off + hf * 32, vs[0]);
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    tc_wait_ld();
                    if (c == 0) tmem_ld16(tS + lane_off + hf * 32 + 16, vs[1]);
#pragma unroll
                    for (int e = 0; e < 16; e += 4) {
                        const float4 l4 = ld_shared_f4(vec + (c * 16 + e) * 4);
                        p[c * 16 + e] = fast_exp2(fmaf(__uint_as_float(vs[c][e]), sl2, -l4.x));
                        p[c * 16 + e + 1] = fast_exp2(fmaf(__uint_as_float(vs[c][e + 1]), sl2, -l4.y));
                        p[c * 16 + e + 2] = fast_exp2(fmaf(__uint_as_float(vs[c][e + 2]), sl2, -l4.z));
                        p[c * 16 + e + 3] = fast_exp2(fmaf(__uint_as_float(vs[c][e + 3]), sl2, -l4.w));
                    }
                }
            }
            if (!key_ok || qvalid < 32) {
#pragma unroll
                for (int e = 0; e < 32; ++e) if (!key_ok || e >= qvalid) p[e] = 0.f;
            }
            {
                uint32_t pw[16];
#pragma unroll
                for (int e = 0; e < 16; ++e) pw[e] = pack_bf16(p[2 * e], p[2 * e + 1]);
                tmem_st16(tS + lane_off + hf * 32, pw);                          // over the front of this thread's own S^T columns
            }
            tc_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(p_ready);                                 // one arrival per warp (32 same-address arrivals serialise)
            // ---- dS phase: dS^T = P^T (dP^T - D[q]) ----
            mbar_wait(dp_ready, i & 1);
            tc_fence_after();
            uint32_t dsw[16];
            {
                uint32_t vp[2][16];
                tmem_ld16(tdP + lane_off + hf * 32, vp[0]);
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    tc_wait_ld();
                    if (c == 0) tmem_ld16(tdP + lane_off + hf * 32 + 16, vp[1]);
#pragma unroll
                    for (int e = 0; e < 16; e += 4) {
                        const float4 d4 = ld_shared_f4(vec + 512 + (c * 16 + e) * 4);
                        const float a0 = p[c * 16 + e] * (__uint_as_float(vp[c][e]) - d4.x);
                        const float a1 = p[c * 16 + e + 1] * (__uint_as_float(vp[c][e + 1]) - d4.y);
                        const float a2 = p[c * 16 + e + 2] * (__uint_as_float(vp[c][e + 2]) - d4.z);
                        const float a3 = p[c * 16 + e + 3] * (__uint_as_float(vp[c][e + 3]) - d4.w);
                        dsw[c * 8 + (e >> 1)] = pack_bf16(a0, a1);
                        dsw[c * 8 + (e >> 1) + 1] = pack_bf16(a2, a3);
                    }
                }
            }
            if (!key_ok || qvalid < 32) {                                        // padded rows / columns: exact zeros (their lse2 / D slots hold
#pragma unroll                                                                   // whatever the ring slot held before: 0 x garbage could be NaN)
                for (int e = 0; e < 16; ++e) if (!key_ok || 2 * e >= qvalid) dsw[e] = 0u;
            }
            tmem_st16(tdP + lane_off + hf * 32, dsw);                            // A operand of dK += dS^T Q
            if (i > 0) mbar_wait(ds_free, (i - 1) & 1);                          // dQ(i-1) has finished reading the shared dS^T tile
            store_p_16(sDS, r, hf * 32, dsw);                                    // A operand (MN-major) of dQ(i) = dS(i) K
            store_p_16(sDS, r, hf * 32 + 16, dsw + 8);
            fence_proxy_async_smem();
            tc_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(ds_ready);
        }
        if (nq > 0) { mbar_wait(acc_ready, 0); tc_fence_after(); }
        const int key = k0 + r;
        if (P.q_split > 1) {
            // this CTA saw only a share of the Q tiles: dV / dK shares (unscaled fp32) go through swizzled staging tiles in the idle
            // Q / dO ring and two bulk reduce-adds; attn_dq_tiles_convert_kernel rounds (and scales dK) afterwards
            if (nq > 0) {
                const int which = hf >> 1, c = hf & 1;
                uint32_t v[32];
                tmem_ld32((which == 0 ? tdV : tdK) + lane_off + c * 32, v);
                tc_wait_ld();
                const uint32_t st = smem_u32(smem + (which == 0 ? FbSmem::Q : FbSmem::DO)) + r * 256;
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    st_shared_v4(st + (((c * 8 + e) ^ (r & 15)) << 4), v[4 * e], v[4 * e + 1], v[4 * e + 2], v[4 * e + 3]);
                fence_proxy_async_smem();
            }
            named_bar_sync(3, FB_CW * 32);
            if (threadIdx.x == 0 && nq > 0) {
                const long long tile = ((long long)bh * kv_tiles + kt) * (TILE * HD);
                bulk_reduce_add_f32(P.dVacc + tile, smem + FbSmem::Q, TILE * HD * 4);
                bulk_reduce_add_f32(P.dKacc + tile, smem + FbSmem::DO, TILE * HD * 4);
                bulk_wait_read0();
            }
        } else {
            const int which = hf >> 1, c = hf & 1;               // warps hf 0,1 store dV chunks 0,1; hf 2,3 store dK chunks 0,1
            const uint32_t tacc = which == 0 ? tdV : tdK;
            const float mul = which == 0 ? 1.0f : P.scale;
            __nv_bfloat16* base = which == 0 ? P.dV : P.dK;
            const long long ld = which == 0 ? P.lddv : P.lddk;
            uint32_t v[32];
            tmem_ld32(tacc + lane_off + c * 32, v);
            tc_wait_ld();
            if (key < P.Tk) {
                __nv_bfloat16* dst = base + ((long long)b * P.Tk + key) * ld + h * HD + c * 32;
#pragma unroll
                for (int e = 0; e < 32; e += 8) {
                    uint4 o;
                    o.x = pack_bf16(__uint_as_float(v[e]) * mul, __uint_as_float(v[e + 1]) * mul);
                    o.y = pack_bf16(__uint_as_float(v[e + 2]) * mul, __uint_as_float(v[e + 3]) * mul);
                    o.z = pack_bf16(__uint_as_float(v[e + 4]) * mul, __uint_as_float(v[e + 5]) * mul);
                    o.w = pack_bf16(__uint_as_float(v[e + 6]) * mul, __uint_as_float(v[e + 7]) * mul);
                    *reinterpret_cast<uint4*>(dst + e) = o;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == FB_CW + 1) { tc_fence_after(); tmem_dealloc(tmem, 512); }
}

// dQ = scale * (sum of the KV tiles' shares): fp32 tiles [B * H][q_tiles][128][64] with XOR-swizzled 16-byte chunks (the staging
// layout of attn_bwd_fused_kernel) -> bf16 [B, Tq, H, 64] with a row stride
__global__ void __launch_bounds__(256)
attn_dq_tiles_convert_kernel(const float* __restrict__ acc, __nv_bfloat16* __restrict__ dq, long long lddq, int B, int H, int Tq, float scale,
                             const float* __restrict__ acc2 = nullptr, __nv_bfloat16* __restrict__ out2 = nullptr, long long ld2 = 0,
                             float scale2 = 1.0f) {
    pdl_enter();
    const int q_tiles = (Tq + TILE - 1) / TILE;
    const long long per_tensor = (long long)B * H * q_tiles * TILE * 8;    // one work item = 8 elements (two 16-byte fp32 chunks)
    const long long total = acc2 != nullptr ? 2 * per_tensor : per_tensor; // second tensor of the same shape (dK and dV in one launch)
    for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < total; i0 += (long long)gridDim.x * blockDim.x) {
        long long i = i0;
        if (i >= per_tensor) { i -= per_tensor; acc = acc2; dq = out2; lddq = ld2; scale = scale2; }
        const int part = (int)(i & 7);
        const long long row = i >> 3;                                     // (bh, tile, r)
        const int r = (int)(row % TILE);
        const long long bt = row / TILE;
        const int tile = (int)(bt % q_tiles);
        const long long bh = bt / q_tiles;
        const int q = tile * TILE + r;
        if (q >= Tq) continue;
        const int h = (int)(bh % H), b = (int)(bh / H);
        const float* src = acc + row * HD;
        const float4 a0 = *reinterpret_cast<const float4*>(src + (((2 * part) ^ (r & 15)) << 2));
        const float4 a1 = *reinterpret_cast<const float4*>(src + (((2 * part + 1) ^ (r & 15)) << 2));
        uint4 o;
        o.x = pack_bf16(a0.x * scale, a0.y * scale); o.y = pack_bf16(a0.z * scale, a0.w * scale);
        o.z = pack_bf16(a1.x * scale, a1.y * scale); o.w = pack_bf16(a1.z * scale, a1.w * scale);
        *reinterpret_cast<uint4*>(dq + ((long long)b * Tq + q) * lddq + h * HD + part * 8) = o;
    }
}

static int make_qkv_map(CUtensorMap* m, const void* base, long long ld, int B, int H, int T, int rows = TILE) {
    uint64_t dims[4] = {(uint64_t)HD, (uint64_t)H, (uint64_t)T, (uint64_t)B};
    uint64_t strides[3] = {(uint64_t)HD * 2, (uint64_t)ld * 2, (uint64_t)T * (uint64_t)ld * 2};
    uint32_t box[4] = {HD, 1, (uint32_t)rows, 1};
    return make_tmap_bf16(m, base, 4, dims, strides, box, nullptr);
}

}  // namespace aoz

using namespace aoz;

extern "C" {

int aoz_attn_fwd(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv, void* o, long long ldo,
                 void* lse, int B, int H, int Tq, int Tk, float scale, void* stream) {
    AOZ_CHECK_ARG(q && k && v && o && lse, "aoz_attn_fwd: null pointer");
    AOZ_CHECK_ARG(B > 0 && H > 0 && Tq > 0 && Tk > 0, "aoz_attn_fwd: empty problem");
    AOZ_CHECK_ARG((ldq % 8) == 0 && (ldk % 8) == 0 && (ldv % 8) == 0 && (ldo % 8) == 0, "aoz_attn_fwd: strides must be multiples of 8");
    AttnParams P;
    memset(&P, 0, sizeof(P));
    int rc;
    if ((rc = make_qkv_map(&P.tmQ, q, ldq, B, H, Tq)) != AOZ_OK) return rc;
    if ((rc = make_qkv_map(&P.tmK, k, ldk, B, H, Tk, KT)) != AOZ_OK) return rc;       // the forward streams 64-key tiles
    if ((rc = make_qkv_map(&P.tmV, v, ldv, B, H, Tk, KT)) != AOZ_OK) return rc;
    P.B = B; P.H = H; P.Tq = Tq; P.Tk = Tk; P.scale = scale;
    P.O = (__nv_bfloat16*)o; P.ldo = ldo; P.lse = (float*)lse;
    static bool attr = false;
    if (!attr) { cudaFuncSetAttribute(attn_fwd_tm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TmSmem::TOTAL); attr = true; }
    launch_k(attn_fwd_tm_kernel, dim3(B * H * ((Tq + TILE - 1) / TILE)), dim3(ATT_TM_THREADS), (size_t)(TmSmem::TOTAL), (cudaStream_t)stream, P);
    AOZ_CHECK_LAUNCH("attn_fwd_tm_kernel");
    return AOZ_OK;
}

// one per-row vector [B, H, Tq] of the backward workspace (D, lse2), padded to 128-byte granules
static long long bwd_vec_floats(int B, int H, int Tq) { return (((long long)B * H * Tq + 31) / 32) * 32; }
long long aoz_attn_bwd_workspace_floats(int B, int H, int Tq) {
    // D and lse2 vectors, the dQ tile buffer, and (one KV tile, Q tiles cut over several CTAs) one dK and one dV tile per (b, h)
    return 2 * bwd_vec_floats(B, H, Tq) + (long long)B * H * ((Tq + TILE - 1) / TILE + 2) * TILE * HD;
}

// 2 = attn_bwd_fused_kernel (key-major scores, P^T / dS^T in tensor memory, bulk-reduced dQ; default), 0 = dK/dV kernel + dQ kernel
// (bit-reproducible).  Any other value is refused rather than mapped onto one of the two.
static int g_bwd_fused = 2;
int aoz_attn_set_bwd_mode(int fused) {
    AOZ_CHECK_ARG(fused == 0 || fused == 2, "aoz_attn_set_bwd_mode: mode must be 2 (one kernel) or 0 (two kernels)");
    g_bwd_fused = fused;
    return AOZ_OK;
}

int aoz_attn_bwd(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv, const void* o,
                 long long ldo, const void* d_o, long long lddo, const void* lse, void* dq, long long lddq, void* dk,
                 long long lddk, void* dv, long long lddv, int B, int H, int Tq, int Tk, float scale, void* workspace,
                 void* stream) {
    AOZ_CHECK_ARG(q && k && v && o && d_o && lse && dq && dk && dv && workspace, "aoz_attn_bwd: null pointer");
    AOZ_CHECK_ARG(B > 0 && H > 0 && Tq > 0 && Tk > 0, "aoz_attn_bwd: empty problem");
    AOZ_CHECK_ARG((ldq % 8) == 0 && (ldk % 8) == 0 && (ldv % 8) == 0 && (ldo % 8) == 0 && (lddo % 8) == 0 && (lddq % 8) == 0 &&
                  (lddk % 8) == 0 && (lddv % 8) == 0, "aoz_attn_bwd: strides must be multiples of 8");
    cudaStream_t s = (cudaStream_t)stream;
    AttnParams P;
    memset(&P, 0, sizeof(P));
    int rc;
    if ((rc = make_qkv_map(&P.tmQ, q, ldq, B, H, Tq)) != AOZ_OK) return rc;
    if ((rc = make_qkv_map(&P.tmK, k, ldk, B, H, Tk)) != AOZ_OK) return rc;
    if ((rc = make_qkv_map(&P.tmV, v, ldv, B, H, Tk)) != AOZ_OK) return rc;
    if ((rc = make_qkv_map(&P.tmDO, d_o, lddo, B, H, Tq)) != AOZ_OK) return rc;
    P.B = B; P.H = H; P.Tq = Tq; P.Tk = Tk; P.scale = scale;
    P.lse = (float*)const_cast<void*>(lse); P.Dvec = (const float*)workspace;
    P.dQ = (__nv_bfloat16*)dq; P.lddq = lddq; P.dK = (__nv_bfloat16*)dk; P.lddk = lddk; P.dV = (__nv_bfloat16*)dv; P.lddv = lddv;
    float* const acc_ws = (float*)workspace + 2 * bwd_vec_floats(B, H, Tq);
    const bool one_kernel = g_bwd_fused == 2 && (Tq % 4) == 0;
    const int q_tiles = (Tq + TILE - 1) / TILE, kv_tiles = (Tk + TILE - 1) / TILE;
    // One KV tile (cross-attention): B * H CTAs would leave most of the 148 SMs idle, so the Q tiles are cut over q_split CTAs
    // (about two waves of CTAs, at least two Q tiles each) whose dK / dV shares are summed like dQ.
    int q_split = 1;
    if (one_kernel && kv_tiles == 1) {
        q_split = (2 * sm_count() + B * H - 1) / (B * H);
        if (q_split > (q_tiles + 1) / 2) q_split = (q_tiles + 1) / 2;
        if (q_split < 1) q_split = 1;
        const int per = (q_tiles + q_split - 1) / q_split;
        q_split = (q_tiles + per - 1) / per;                    // no CTA without a Q tile
    }
    const long long dq_floats = (long long)B * H * q_tiles * TILE * HD, kv_floats = (long long)B * H * kv_tiles * TILE * HD;
    // cleared by the prep kernel: the dQ tile buffer when several KV tiles add into it; the dK / dV tile buffers when several CTAs
    // share a KV tile
    float* const z0 = kv_tiles > 1 ? acc_ws : acc_ws + dq_floats;
    const long long zn = one_kernel ? (kv_tiles > 1 ? dq_floats : 0) + (q_split > 1 ? 2 * kv_floats : 0) : 0;
    {
        const long long items = (long long)B * Tq * H * 8;
        long long blocks = (items + 255) / 256;
        if (blocks > sm_count() * 16) blocks = sm_count() * 16;
        launch_k(attn_bwd_prep_kernel, dim3((int)blocks), dim3(256), (size_t)(0), s, (const __nv_bfloat16*)o, ldo, (const __nv_bfloat16*)d_o, lddo, B, H, Tq, (float*)workspace,
                 (const float*)lse, (float*)workspace + bwd_vec_floats(B, H, Tq), (float4*)z0, zn / 4);
        AOZ_CHECK_LAUNCH("attn_bwd_prep_kernel");
    }
    if (one_kernel) {
        // one kernel: dK, dV and this KV tile's share of dQ; lse is read in the log2 domain from the workspace
        static bool attr_f = false;
        if (!attr_f) { cudaFuncSetAttribute(attn_bwd_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FbSmem::TOTAL); attr_f = true; }
        P.lse = (float*)workspace + bwd_vec_floats(B, H, Tq);
        P.dQacc = acc_ws;
        P.dKacc = acc_ws + dq_floats;
        P.dVacc = acc_ws + dq_floats + kv_floats;
        P.q_split = q_split;
        launch_k(attn_bwd_fused_kernel, dim3(B * H * kv_tiles * q_split), dim3(FB_THREADS), (size_t)(FbSmem::TOTAL), s, P);
        AOZ_CHECK_LAUNCH("attn_bwd_fused_kernel");
        auto blocks_for = [&](long long items) {
            long long blocks = (items + 255) / 256;
            return (int)(blocks > sm_count() * 16 ? sm_count() * 16 : blocks);
        };
        if (kv_tiles > 1) {                                         // (one KV tile: the drain warps stored dQ directly)
            launch_k(attn_dq_tiles_convert_kernel, dim3(blocks_for((long long)B * H * q_tiles * TILE * 8)), dim3(256), (size_t)(0), s,
                     (const float*)P.dQacc, (__nv_bfloat16*)dq, lddq, B, H, Tq, scale, (const float*)nullptr, (__nv_bfloat16*)nullptr, 0LL, 1.0f);
            AOZ_CHECK_LAUNCH("attn_dq_tiles_convert_kernel");
        }
        if (q_split > 1) {                                          // dK (scaled) and dV in one launch
            launch_k(attn_dq_tiles_convert_kernel, dim3(blocks_for(2LL * B * H * kv_tiles * TILE * 8)), dim3(256), (size_t)(0), s,
                     (const float*)P.dKacc, (__nv_bfloat16*)dk, lddk, B, H, Tk, scale, (const float*)P.dVacc, (__nv_bfloat16*)dv, lddv, 1.0f);
            AOZ_CHECK_LAUNCH("attn_dq_tiles_convert_kernel");
        }
        return AOZ_OK;
    }
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(attn_bwd_dkv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, KvSmem::TOTAL);
        cudaFuncSetAttribute(attn_bwd_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DqSmem::TOTAL);
        attr = true;
    }
    launch_k(attn_bwd_dkv_kernel, dim3(B * H * ((Tk + TILE - 1) / TILE)), dim3(ATT_BWD_THREADS), (size_t)(KvSmem::TOTAL), s, P);
    AOZ_CHECK_LAUNCH("attn_bwd_dkv_kernel");
    launch_k(attn_bwd_dq_kernel, dim3(B * H * ((Tq + TILE - 1) / TILE)), dim3(ATT_BWD_THREADS), (size_t)(DqSmem::TOTAL), s, P);
    AOZ_CHECK_LAUNCH("attn_bwd_dq_kernel");
    return AOZ_OK;
}

}  // extern "C"
