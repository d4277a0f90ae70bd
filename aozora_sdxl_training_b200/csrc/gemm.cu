// tcgen05 / TMEM / TMA GEMM core for the SDXL UNet training step (sm_100a).
//
// One persistent, warp-specialised kernel serves every dense contraction of the hot path
// (SURVEY.md 2.1 rows K3, K4, K5): the Linear layers (to_q/k/v, to_out, proj_in/out, GEGLU feed-forward,
// time-embedding MLPs), their dgrad / wgrad, and the 3x3 / 1x1 convolutions as implicit GEMM over NHWC
// activations (forward, dgrad, wgrad).  What the reference reaches through cuBLASLt / cuDNN calls inside
// diffusers' UNet2DConditionModel (train.py:2760) is here:
//
//   warp 0      TMA producer : cp.async.bulk.tensor loads of A / B tiles into a 128B-swizzled smem ring
//   warp 1      MMA issuer   : one elected thread issues tcgen05.mma (128 x BN x 16, bf16 -> fp32 in TMEM)
//   warps 2..5  epilogue     : tcgen05.ld the accumulator (double-buffered in TMEM so the next tile's
//                              main loop overlaps), fused bias / time-embedding / residual / GEGLU, bf16 store
//
// Operands are bf16.  Each operand is either K-major (rows = M or N index, 64 K-elements = 128 bytes per row)
// or MN-major (rows = K index, 64 M/N-elements per row); both are expressed with the same 128B-swizzle
// shared-memory layout and differ only in the UMMA descriptors, so x*W^T (forward), dy*W (dgrad) and
// dy^T*x (wgrad) need no transposed copies.  Convolutions fetch the A operand (and B for wgrad) as shifted
// 4-D TMA boxes of the NHWC tensor; out-of-bounds box elements are zero-filled by the TMA unit, which is
// exactly the conv's zero padding.
#include "common.cuh"
#include <cstring>

namespace aoz {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int GEMM_THREADS = 320;   // 10 warps: TMA, MMA, 8 epilogue
constexpr int MAX_STAGES = 8;
constexpr int SMEM_TILE_BYTES = 196608;                 // 192 KB ring of A/B stages
constexpr int EPI_STAGE_BYTES = 8 * 4096;               // 8 epilogue warps x (32 rows x 32 fp32): register-layout -> row-segment transpose
constexpr int GEMM_SMEM_TOTAL = SMEM_TILE_BYTES + 1024 + EPI_STAGE_BYTES + 1024;   // + barriers + staging + alignment slack (226 KB)

enum GemmMode : int { GM_LINEAR = 0, GM_CONV_FWD = 1, GM_CONV_WGRAD = 2 };
constexpr int MAX_GROUPS = 10;     // 10 x 320 B of descriptors + the base parameters stay under the 4 KB kernel-parameter limit

// one problem of a grouped launch (GM_LINEAR, EPI_STORE, same K / operand majors / tile shape for all problems): the
// weight gradients of one transformer block run as ONE persistent launch, so ~900 tiles fill the 148 SMs in ~6 full
// waves instead of six launches with one or two ragged waves each
struct alignas(64) GroupDesc {
    CUtensorMap tmA, tmB;
    __nv_bfloat16* C; long long ldc;
    int M, N, m_tiles, tile_start;      // m_tiles counts work-unit rows (256-row pair tiles when CTA2)
};
enum GemmEpi : int { EPI_STORE = 0, EPI_GEGLU = 1, EPI_PARTIAL = 2 };

struct GemmParams {
    CUtensorMap tmA, tmB;
    int mode, epi;
    int dbg;                        // experiment flags: 1 = epilogue does not load/store, 2 = MMA ignores full barriers, 4 = producer ignores empty barriers
    int bn, stages;                 // N extent of the accumulator tile (multiple of 32, <= 256; 320 = the wide one-wave plan); smem pipeline depth
    int a_mn, b_mn;                 // 1 = MN-major operand
    int M, N, K;                    // logical extents (CONV_FWD: M = NB*H*W output pixels, K = taps*cin_chunks*64)
    int m_tiles, n_tiles, k_iters;  // tile counts; k_iters = total K iterations (before split)
    int splits;                     // split-K factor (EPI_PARTIAL when > 1)
    // tail split: work items [0, full_work) are whole tiles (x splits); the last `tail_tiles` tiles -- the ones that would
    // run as a mostly empty final wave -- are cut along K into `tail_splits` slices each, written as fp32 partials to
    // `tail_ws` ([slice][128 rows][bn]) and finished (sum + fused epilogue) by tail_fixup_kernel.
    int full_work, tail_tiles, tail_splits;
    float* tail_ws;
    int vec_ok;                     // EPI_STORE: every output / bias / residual row segment is 16-byte aligned
    // conv geometry (NHWC).  H, W = OUTPUT spatial size (CONV_FWD) / dy spatial size (CONV_WGRAD)
    int NB, H, W, TH, TW, tiles_h, tiles_w;
    int taps_s, pad, stride, cin_chunks, flip;   // taps_s = filter width (3 or 1); taps = taps_s*taps_s
    int Cin, n_tiles_per_tap;       // CONV_WGRAD: column = tap*Cin + cin
    int geglu_half;                 // EPI_GEGLU: N/2 (gate rows start here in W)
    // epilogue
    __nv_bfloat16* C; long long ldc;
    const __nv_bfloat16* bias;      // [N] or null
    const __nv_bfloat16* rowgroup_bias; int rows_per_group; long long ld_rgb;   // [groups, N] added per row group (temb)
    const __nv_bfloat16* residual; long long ldr;
    __nv_bfloat16* aux; long long ld_aux;          // GEGLU: pre-activation [M, 2*half]
    float* partial;                 // EPI_PARTIAL: [splits][M][N] fp32
    int accumulate;                 // EPI_STORE: C += result
    int n_groups;                   // > 0: grouped launch, tile indices run over grp[0..n_groups) back to back
    GroupDesc grp[MAX_GROUPS];
};

static_assert(sizeof(GemmParams) <= 4096, "GemmParams must fit the kernel parameter space");

// erf GELU (torch F.gelu default), fp32: x * Phi(x)
__device__ __forceinline__ float gelu_erf(float x) { float e; return x * gelu_cdf(x, e); }

// ---- cluster helpers (CTA-pair mode) ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t local_smem_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" :: "r"(cluster_addr) : "memory");
}
// TMA loads issued by either CTA of a pair, completing on the LEADER's mbarrier (cluster address)
__device__ __forceinline__ void tma2_load_2d(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        :: "r"(smem_u32(smem_dst)), "l"(m), "r"(bar_cluster_addr), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma2_load_4d(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1,
                                             int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        :: "r"(smem_u32(smem_dst)), "l"(m), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on the mbarrier at the same smem offset in BOTH CTAs of the pair once the issued MMAs have completed
__device__ __forceinline__ void umma2_commit_both(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 :: "r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_result, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(smem_result)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" :: "r"(taddr), "r"(ncols) : "memory");
}

__device__ __forceinline__ void st_shared_v4u(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" :: "r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void ld_shared_v4f(uint32_t addr, float* f) {
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(f[0]), "=f"(f[1]), "=f"(f[2]), "=f"(f[3]) : "r"(addr) : "memory");
}
// Epilogue transpose.  tcgen05.ld hands every thread ONE accumulator row (32 consecutive fp32 columns); storing from that
// layout makes each warp store touch 32 different rows with 16 bytes each -- half-used sectors, ~5 cycles per transaction,
// ~21k cycles per 128x256 tile, which made every K <= 1280 GEMM epilogue-bound.  Each warp therefore bounces its 32x32
// chunk through 4 KB of shared memory (XOR-swizzled 16-byte chunks, conflict-free both ways) and continues with 4 lanes
// per row: lane l owns row (l >> 2) + 8*step, columns (l & 3)*8..+8, so loads of the residual and stores of the result
// are 64-byte row segments (full sectors), 8 rows per instruction.
__device__ __forceinline__ void stage_chunk(uint32_t stg, int lane, const uint32_t* r) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
        st_shared_v4u(stg + lane * 128 + ((j ^ (lane & 7)) << 4), r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
}
__device__ __forceinline__ void unstage8(uint32_t stg, int lane, int step, float* f) {
    const int rr = step * 8 + (lane >> 2);
    const int j0 = (lane & 3) * 2;
    ld_shared_v4f(stg + rr * 128 + ((j0 ^ (rr & 7)) << 4), f);
    ld_shared_v4f(stg + rr * 128 + (((j0 + 1) ^ (rr & 7)) << 4), f + 4);
}

struct WorkItem { int tile, split, k_begin, k_end, tail_slot; };      // tail_slot < 0: not a tail slice

__device__ __forceinline__ WorkItem decode_work(const GemmParams& P, int work, int k_per_split) {
    WorkItem w;
    if (work < P.full_work) {
        // (an integer division is ~200 cycles of dependent instructions for the single producer thread before its first TMA issue)
        w.tile = P.splits == 1 ? work : work / P.splits;
        w.split = work - w.tile * P.splits;
        w.k_begin = w.split * k_per_split;
        w.k_end = min(P.k_iters, w.k_begin + k_per_split);
        w.tail_slot = -1;
    } else {
        const int j = work - P.full_work;
        const int t = j / P.tail_splits;
        const int kps = (P.k_iters + P.tail_splits - 1) / P.tail_splits;
        w.tile = (P.splits == 1 ? P.full_work : P.full_work / P.splits) + t;
        w.split = j - t * P.tail_splits;
        w.k_begin = w.split * kps;
        w.k_end = min(P.k_iters, w.k_begin + kps);
        w.tail_slot = j;
    }
    return w;
}

// the problem a tile belongs to (the launch's own operands unless this is a grouped launch)
struct Prob { const CUtensorMap* tmA; const CUtensorMap* tmB; __nv_bfloat16* C; long long ldc; int M, N, m_tiles, ltile; };

__device__ __forceinline__ Prob select_prob(const GemmParams& P, int tile) {
    Prob pr;
    if (P.n_groups == 0) {
        pr.tmA = &P.tmA; pr.tmB = &P.tmB; pr.C = P.C; pr.ldc = P.ldc; pr.M = P.M; pr.N = P.N; pr.m_tiles = P.m_tiles; pr.ltile = tile;
    } else {
        int g = 0;
#pragma unroll 1
        while (g + 1 < P.n_groups && tile >= P.grp[g + 1].tile_start) ++g;
        const GroupDesc& d = P.grp[g];
        pr.tmA = &d.tmA; pr.tmB = &d.tmB; pr.C = d.C; pr.ldc = d.ldc; pr.M = d.M; pr.N = d.N; pr.m_tiles = d.m_tiles;
        pr.ltile = tile - d.tile_start;
    }
    return pr;
}

struct RowMap { long long row; bool ok; int group; };

// output row (and time-embedding row group) of row `row_in_tile` of the 128-row tile `m_blk`
__device__ __forceinline__ RowMap map_row(const GemmParams& P, int M, int m_blk, int row_in_tile) {
    RowMap r;
    if (P.mode == GM_CONV_FWD) {
        int t = m_blk;
        const int tw = t % P.tiles_w; t /= P.tiles_w;
        const int th = t % P.tiles_h; const int img = t / P.tiles_h;
        const int h = th * P.TH + row_in_tile / P.TW, w = tw * P.TW + row_in_tile % P.TW;
        r.ok = (h < P.H) && (w < P.W) && (img < P.NB);
        r.row = ((long long)img * P.H + h) * P.W + w;
        r.group = img;
    } else {
        r.row = (long long)m_blk * BM + row_in_tile;
        r.ok = r.row < M;
        r.group = P.rows_per_group > 0 ? (int)(r.row / P.rows_per_group) : 0;
    }
    return r;
}

// EPI_STORE for 8 consecutive output columns [col, col+8) of output row `row`: bias -> per-image time embedding -> residual
// -> accumulate, each with the bf16 rounding point the op-by-op autocast path has, then one 16-byte store.
// `has_pre` / `pre`: the residual vector of this segment when the caller fetched it ahead of time (vector path only).
__device__ __forceinline__ void epi_store8(const GemmParams& P, __nv_bfloat16* C, long long ldc, long long row, int group, int col,
                                           int col_limit, float* f, bool has_pre = false, uint4 pre = make_uint4(0u, 0u, 0u, 0u)) {
    __nv_bfloat16* dst = C + row * ldc + col;
    const __nv_bfloat16* res = P.residual ? P.residual + row * P.ldr + col : nullptr;
    const __nv_bfloat16* rgb = P.rowgroup_bias ? P.rowgroup_bias + (long long)group * P.ld_rgb + col : nullptr;
    if (P.vec_ok && col + 7 < col_limit) {
        if (P.bias) {
            const uint4 bb = __ldg(reinterpret_cast<const uint4*>(P.bias + col));
            const uint32_t bw[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) { f[2 * e] += bf16lo(bw[e]); f[2 * e + 1] += bf16hi(bw[e]); }
        }
        if (rgb) {
            const uint4 gg = __ldg(reinterpret_cast<const uint4*>(rgb));
            const uint32_t gw[4] = {gg.x, gg.y, gg.z, gg.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const uint32_t pk = pack_bf16(f[2 * e], f[2 * e + 1]);          // both roundings in one packed conversion
                f[2 * e] = bf16lo(pk) + bf16lo(gw[e]);
                f[2 * e + 1] = bf16hi(pk) + bf16hi(gw[e]);
            }
        }
        if (res) {
            const uint4 rr = has_pre ? pre : *reinterpret_cast<const uint4*>(res);
            const uint32_t rw[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const uint32_t pk = pack_bf16(f[2 * e], f[2 * e + 1]);          // both roundings in one packed conversion
                f[2 * e] = bf16lo(pk) + bf16lo(rw[e]);
                f[2 * e + 1] = bf16hi(pk) + bf16hi(rw[e]);
            }
        }
        if (P.accumulate) {
            const uint4 oo = *reinterpret_cast<const uint4*>(dst);
            const uint32_t ow[4] = {oo.x, oo.y, oo.z, oo.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const uint32_t pk = pack_bf16(f[2 * e], f[2 * e + 1]);          // both roundings in one packed conversion
                f[2 * e] = bf16lo(pk) + bf16lo(ow[e]);
                f[2 * e + 1] = bf16hi(pk) + bf16hi(ow[e]);
            }
        }
        *reinterpret_cast<uint4*>(dst) = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
    } else {
        for (int e = 0; e < 8; ++e) {
            if (col + e < col_limit) {
                float x = f[e];
                if (P.bias) x += __bfloat162float(P.bias[col + e]);
                if (rgb) x = round_bf16(x) + __bfloat162float(rgb[e]);
                if (res) x = round_bf16(x) + __bfloat162float(res[e]);
                if (P.accumulate) x = round_bf16(x) + __bfloat162float(dst[e]);
                dst[e] = __float2bfloat16_rn(x);
            }
        }
    }
}

// CTA2 = true: two CTAs of a cluster (one SM pair) compute a 256 x BN tile with tcgen05.mma.cta_group::2.  Each CTA
// stages its own 128 rows of A and HALF of the B tile, so the L2 -> shared-memory traffic per FLOP drops by a third
// (the 1-CTA 128 x 256 tile needs ~26 TB/s of L2 bandwidth at tensor peak -- more than the chip has).  Only the
// leader CTA (cluster rank 0) issues MMAs; completion is multicast to both CTAs' barriers.
template <bool CTA2>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_kernel(const __grid_constant__ GemmParams P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* bar_base = smem + SMEM_TILE_BYTES;
    uint64_t* full_bar = (uint64_t*)bar_base;                 // [MAX_STAGES]
    uint64_t* empty_bar = full_bar + MAX_STAGES;              // [MAX_STAGES]
    uint64_t* tfull_bar = empty_bar + MAX_STAGES;             // [2]
    uint64_t* tempty_bar = tfull_bar + 2;                     // [2]
    uint32_t* tmem_slot = (uint32_t*)(tempty_bar + 2);
    const int BN = P.bn;                                      // accumulator tile width (runtime: picked by the host cost model)
    const int B_ROWS = CTA2 ? BN / 2 : BN;                    // B rows this CTA stages (a pair splits the B tile)
    const int A_BYTES = BM * BK * 2;
    // MN-major B arrives in whole 64-wide chunks (the wide plan's 160 rows = 2.5 chunks: the third is half used)
    const int B_BYTES = P.b_mn ? ((B_ROWS + 63) / 64) * 8192 : B_ROWS * BK * 2;
    const int STAGE_BYTES = A_BYTES + B_BYTES;
    // Wide one-wave plan (CTA pairs, BN = 320): ONE 256 x 320 tile per pair, a single accumulator of 320 TMEM columns written by
    // two MMAs per K step (N = 256 over B rows [0, 128) of each CTA, N = 64 over rows [128, 160)).  4096 x 1280 outputs are
    // 16 x 4 = 64 tiles on 74 SM pairs instead of 80 tiles of 256 x 256 = two rounds with the second one 8 % full.
    const bool WIDE = CTA2 && BN == 320;
    const int STAGES = P.stages;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // dbg 64 (experiments): CTA 0 stamps clock64 at its phase boundaries into the scratch buffer (tools/gemm_timeline.py)
    long long* tl = ((P.dbg & 64) && blockIdx.x == 0 && P.tail_ws != nullptr) ? reinterpret_cast<long long*>(P.tail_ws) : nullptr;
    if (tl && threadIdx.x == 0) tl[0] = clock64();
    const uint32_t rank = CTA2 ? cluster_ctarank() : 0u;
    const bool leader = rank == 0;
    const int unit = CTA2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;          // persistent work unit (CTA or CTA pair)
    const int n_units = CTA2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;

    if (warp == 0 && lane == 0) {
        if (P.n_groups == 0) { tma_prefetch_desc(&P.tmA); tma_prefetch_desc(&P.tmB); }
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], CTA2 ? 16 : 8); }
        fence_mbar_init();
    }
    if (warp == 1) { if (CTA2) tmem_alloc2(tmem_slot, 512); else tmem_alloc(tmem_slot, 512); }
    tc_fence_before();
    if (CTA2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (tl && threadIdx.x == 0) tl[1] = clock64();
    pdl_enter();
    if (tl && threadIdx.x == 0) tl[2] = clock64();          // prologue done (barriers, TMEM, descriptors): only now wait for the previous kernel's results

    const int total_work = P.full_work + P.tail_tiles * P.tail_splits;      // (m_tiles counts 256-row pair tiles when CTA2)
    const int k_per_split = P.splits == 1 ? P.k_iters : (P.k_iters + P.splits - 1) / P.splits;
    const int m_sub = CTA2 ? 2 : 1;

    if (warp == 0) {
        // ================================ TMA producer (one thread) ================================
        // The inner loop is kept to: wait(empty) -> expect_tx -> TMA issues, with every coordinate advanced incrementally.
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            long long issued = 0;
            const uint32_t fb0_cluster = CTA2 ? mapa_rank(smem_u32(&full_bar[0]), 0) : 0u;   // leader's full barriers
            const bool a_mn = P.a_mn != 0, b_mn = P.b_mn != 0;
            const int b_chunks = (B_ROWS + 63) / 64;
            for (int work = unit; work < total_work; work += n_units) {
                const WorkItem wi = decode_work(P, work, k_per_split);
                const Prob pr = select_prob(P, wi.tile);
                const CUtensorMap* tmA = pr.tmA;
                const CUtensorMap* tmB = pr.tmB;
                const int m_blk = (pr.ltile % pr.m_tiles) * m_sub + (int)rank;     // 128-row tile index of THIS CTA
                const int n_blk = pr.ltile / pr.m_tiles;
                const int k_begin = wi.k_begin, k_end = wi.k_end;
                const int n_row0 = n_blk * BN + (CTA2 ? (int)rank * (BN / 2) : 0);  // first B row (N index) this CTA stages
                const int m_row0 = m_blk * BM;
                // GEGLU: accumulator columns [0, BN/2) = value rows, [BN/2, BN) = gate rows of the projection weight
                const int g_row0 = CTA2 ? (leader ? 0 : P.geglu_half) + n_blk * (BN / 2) : n_blk * (BN / 2);
                // conv forward: tile origin and running (tap, channel chunk) position
                int img = 0, h0 = 0, w0 = 0, cc = 0, tap_r = 0, tap_s = 0;
                if (P.mode == GM_CONV_FWD) {
                    int t = m_blk;
                    const int tw = t % P.tiles_w; t /= P.tiles_w;
                    const int th = t % P.tiles_h; img = t / P.tiles_h;
                    h0 = th * P.TH * P.stride - P.pad; w0 = tw * P.TW * P.stride - P.pad;
                    const int tap = k_begin / P.cin_chunks;
                    cc = k_begin - tap * P.cin_chunks;
                    tap_r = tap / P.taps_s; tap_s = tap - tap_r * P.taps_s;
                }
                // conv wgrad: fixed tap / channel origin per tile, running pixel-tile position
                int wg_c0 = 0, wg_dh = 0, wg_dw = 0, p_tw = 0, p_th = 0, p_im = 0;
                if (P.mode == GM_CONV_WGRAD) {
                    const int wg_tap = n_blk / P.n_tiles_per_tap;
                    wg_c0 = (n_blk - wg_tap * P.n_tiles_per_tap) * BN + (CTA2 ? (int)rank * (BN / 2) : 0);
                    const int r = wg_tap / P.taps_s, sft = wg_tap - r * P.taps_s;
                    wg_dh = r - P.pad; wg_dw = sft - P.pad;
                    int t = k_begin;
                    p_tw = t % P.tiles_w; t /= P.tiles_w;
                    p_th = t % P.tiles_h; p_im = t / P.tiles_h;
                }
                for (int kit = k_begin; kit < k_end; ++kit) {
                    if (!(P.dbg & 4)) mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * STAGE_BYTES;
                    uint8_t* sb = sa + A_BYTES;
                    uint64_t* fb = &full_bar[stage];
                    const uint32_t fbc = fb0_cluster + stage * 8;
                    if (CTA2) { if (leader) mbar_arrive_expect_tx(fb, 2 * STAGE_BYTES); }
                    else mbar_arrive_expect_tx(fb, STAGE_BYTES);
                    const int k0 = kit * BK;
                    if (P.mode == GM_LINEAR) {
                        if (!a_mn) { if (CTA2) tma2_load_2d(sa, tmA, fbc, k0, m_row0); else tma_load_2d(sa, tmA, fb, k0, m_row0); }
                        else {
#pragma unroll
                            for (int jj = 0; jj < BM / 64; ++jj) {
                                if (CTA2) tma2_load_2d(sa + jj * 8192, tmA, fbc, m_row0 + jj * 64, k0);
                                else tma_load_2d(sa + jj * 8192, tmA, fb, m_row0 + jj * 64, k0);
                            }
                        }
                    } else if (P.mode == GM_CONV_FWD) {
                        const int r = P.flip ? P.taps_s - 1 - tap_r : tap_r, sft = P.flip ? P.taps_s - 1 - tap_s : tap_s;
                        if (CTA2) tma2_load_4d(sa, tmA, fbc, cc * BK, w0 + sft, h0 + r, img);
                        else tma_load_4d(sa, tmA, fb, cc * BK, w0 + sft, h0 + r, img);
                        if (++cc == P.cin_chunks) { cc = 0; if (++tap_s == P.taps_s) { tap_s = 0; ++tap_r; } }
                    }
                    if (P.mode != GM_CONV_WGRAD) {
                        if (!b_mn) {
                            if (P.epi == EPI_GEGLU) {
                                if (CTA2) tma2_load_2d(sb, tmB, fbc, k0, g_row0);
                                else {
                                    tma_load_2d(sb, tmB, fb, k0, g_row0);
                                    tma_load_2d(sb + (BN / 2) * 128, tmB, fb, k0, P.geglu_half + g_row0);
                                }
                            } else {
                                if (CTA2) tma2_load_2d(sb, tmB, fbc, k0, n_row0); else tma_load_2d(sb, tmB, fb, k0, n_row0);
                            }
                        } else {
                            for (int jj = 0; jj < b_chunks; ++jj) {
                                if (CTA2) tma2_load_2d(sb + jj * 8192, tmB, fbc, n_row0 + jj * 64, k0);
                                else tma_load_2d(sb + jj * 8192, tmB, fb, n_row0 + jj * 64, k0);
                            }
                        }
                    } else {   // GM_CONV_WGRAD: K iteration = one 8x8 pixel tile of dy; both operands MN-major
                        const int hh = p_th * P.TH, ww = p_tw * P.TW;
#pragma unroll
                        for (int jj = 0; jj < BM / 64; ++jj) {
                            if (CTA2) tma2_load_4d(sa + jj * 8192, tmA, fbc, m_row0 + jj * 64, ww, hh, p_im);
                            else tma_load_4d(sa + jj * 8192, tmA, fb, m_row0 + jj * 64, ww, hh, p_im);
                        }
                        for (int jj = 0; jj < b_chunks; ++jj) {
                            if (CTA2) tma2_load_4d(sb + jj * 8192, tmB, fbc, wg_c0 + jj * 64, ww * P.stride + wg_dw, hh * P.stride + wg_dh, p_im);
                            else tma_load_4d(sb + jj * 8192, tmB, fb, wg_c0 + jj * 64, ww * P.stride + wg_dw, hh * P.stride + wg_dh, p_im);
                        }
                        if (++p_tw == P.tiles_w) { p_tw = 0; if (++p_th == P.tiles_h) { p_th = 0; ++p_im; } }
                    }
                    if (++stage == (uint32_t)STAGES) { stage = 0; phase ^= 1; }
                    if (tl && issued == 0) tl[3] = clock64();
                    ++issued;
                }
            }
            if (P.dbg & 2) {      // experiment mode: nobody waited for the loads -- drain them before the CTA may exit
                if (!CTA2 || leader) {
                    for (int sidx = 0; sidx < STAGES; ++sidx) {
                        const bool this_lap = (uint32_t)sidx < stage;
                        if (!this_lap && issued < (long long)STAGES) continue;
                        if (issued == 0) continue;
                        mbar_wait(&full_bar[sidx], this_lap ? phase : (phase ^ 1));
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer (leader CTA only in pair mode) ================================
        // The WHOLE warp runs this loop converged (barrier waits included) and one elected lane issues the tcgen05 instructions: with
        // `if (lane == 0)` around the loop ptxas kept the descriptors in vector registers and wrapped every tcgen05.mma / commit in an
        // ELECT + R2UR + BRA.U.ANY sequence (~15 dependent instructions per MMA), so the issuing THREAD paced the tensor pipe (found
        // with ncu's source view on the attention kernels in round 2; see elect_one_sync in common.cuh).  Converged, the descriptors
        // live in uniform registers and a K iteration is four back-to-back UTCHMMA.
        // Descriptors are advanced by integer adds on their low word.
        if (leader) {
            const uint32_t idesc = make_idesc_bf16(CTA2 ? 256 : BM, WIDE ? 256 : BN, P.a_mn, P.b_mn);
            const uint32_t idesc2 = make_idesc_bf16(256, 64, P.a_mn, P.b_mn);          // wide plan: accumulator columns [256, 320)
            const uint64_t hi = ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);   // SBO, version, SW128
            const uint32_t smem_lo = (smem_u32(smem) & 0x3ffffu) >> 4;
            const uint32_t a_lo0 = smem_lo | ((P.a_mn ? (8192u >> 4) : 1u) << 16);
            const uint32_t b_lo0 = (smem_lo + (uint32_t)(A_BYTES >> 4)) | ((P.b_mn ? (8192u >> 4) : 1u) << 16);
            const uint32_t a_kstep = (P.a_mn ? 2048u : 32u) >> 4, b_kstep = (P.b_mn ? 2048u : 32u) >> 4;
            const uint32_t stage_step = (uint32_t)STAGE_BYTES >> 4;
            uint32_t stage = 0, phase = 0;
            uint32_t acc = 0, acc_phase = 0;
            for (int work = unit; work < total_work; work += n_units) {
                const WorkItem wi = decode_work(P, work, k_per_split);
                const int k_begin = wi.k_begin, k_end = wi.k_end;
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (WIDE ? 0u : acc * 256);
                uint32_t accum = 0;
                for (int kit = k_begin; kit < k_end; ++kit) {
                    if (!(P.dbg & 2)) mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    if (tl && lane == 0 && kit == k_begin) tl[4] = clock64();
                    if (elect_one_sync()) {
                        const uint32_t alo = a_lo0 + stage * stage_step, blo = b_lo0 + stage * stage_step;
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) {
                            const uint64_t da = hi | (uint64_t)(alo + k * a_kstep);
                            const uint64_t db = hi | (uint64_t)(blo + k * b_kstep);
                            if (CTA2) umma2_bf16(tmem_d, da, db, idesc, k == 0 ? accum : 1u); else umma_bf16(tmem_d, da, db, idesc, k == 0 ? accum : 1u);
                            // B rows [128, 160) of each CTA start 16 KB into its B stage in either operand major
                            if (CTA2 && WIDE) umma2_bf16(tmem_d + 256, da, db + (16384u >> 4), idesc2, k == 0 ? accum : 1u);
                        }
                        // frees the smem slot (in both CTAs) when the MMAs retire
                        if (CTA2) umma2_commit_both(&empty_bar[stage]); else umma_commit(&empty_bar[stage]);
                    }
                    __syncwarp();
                    accum = 1;
                    if (++stage == (uint32_t)STAGES) { stage = 0; phase ^= 1; }
                }
                // accumulator complete (an empty split still signals the epilogue)
                if (elect_one_sync()) {
                    if (CTA2) umma2_commit_both(&tfull_bar[acc]); else umma_commit(&tfull_bar[acc]);
                }
                __syncwarp();
                if (tl && lane == 0) tl[5] = clock64();
                if (++acc == (WIDE ? 1u : 2u)) { acc = 0; acc_phase ^= 1; }      // the wide plan has ONE accumulator: tiles of a CTA pair do not overlap
            }
        }
        __syncwarp();
    } else {
        // ================================ epilogue (warps 2..9) ================================
        // two warps per TMEM lane quarter; they split the tile's 32-column chunks (even / odd)
        const int q = warp & 3;                       // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2;             // 0: even chunks, 1: odd chunks
        const int row_in_tile = q * 32 + lane;
        const uint32_t stg = smem_u32(bar_base + 1024) + (uint32_t)(warp - 2) * 4096;     // this warp's 4 KB transpose buffer
        uint32_t acc = 0, acc_phase = 0;
        for (int work = unit; work < total_work; work += n_units) {
            const WorkItem wi = decode_work(P, work, k_per_split);
            const int split = wi.split;
            const Prob pr = select_prob(P, wi.tile);
            const int m_blk = (pr.ltile % pr.m_tiles) * m_sub + (int)rank, n_blk = pr.ltile / pr.m_tiles;
            const bool empty_split = wi.k_end <= wi.k_begin;
            const RowMap rm = map_row(P, pr.M, m_blk, row_in_tile);
            const long long row = rm.row;
            const bool row_ok = rm.ok;
            const int group = rm.group;
            // column mapping
            int col0, col_limit;                          // first output column of this tile / exclusive limit
            long long col_shift = 0;                      // WGRAD: tap*Cin added to the column
            const int OUT_COLS = BN;
            if (P.mode == GM_CONV_WGRAD) {
                const int tap = n_blk / P.n_tiles_per_tap;
                col0 = (n_blk - tap * P.n_tiles_per_tap) * BN;
                col_limit = P.Cin;
                col_shift = (long long)tap * P.Cin;
            } else if (P.epi == EPI_GEGLU) {
                col0 = n_blk * (BN / 2);
                col_limit = P.geglu_half;
            } else {
                col0 = n_blk * BN;
                col_limit = pr.N;
            }

            // EPI_STORE with a residual: the residual rows do not depend on the accumulator, so the 64-byte row segments of the
            // first chunk are requested BEFORE waiting for the MMAs and every later chunk's one chunk ahead (a load placed next
            // to its use cost ~0.6 us of L2 latency per 8 rows: the epilogue, not the main loop, bounded the K <= 1280 GEMMs)
            const int lcol = (lane & 3) * 8;               // this lane's 8 columns inside a 32-column chunk (transposed layout)
            const bool pre_res = P.residual != nullptr && P.vec_ok && P.epi == EPI_STORE && wi.tail_slot < 0 && P.mode != GM_CONV_WGRAD;
            RowMap rmap[4];
            uint4 rnext[4];
#pragma unroll
            for (int st = 0; st < 4; ++st) {
                rmap[st] = map_row(P, pr.M, m_blk, q * 32 + st * 8 + (lane >> 2));
                rnext[st] = make_uint4(0u, 0u, 0u, 0u);
            }
            // wide plan: accumulator column -> output column.  CTA r holds B rows [160 r, 160 r + 160) of the tile, the first MMA
            // covers rows [0, 128) of both CTAs and the second rows [128, 160): accumulator columns [0, 128) = n [0, 128),
            // [128, 256) = n [160, 288), [256, 288) = n [128, 160), [288, 320) = n [288, 320)
            auto out_c = [&](int c) { return !WIDE ? c : c < 128 ? c : c < 256 ? c + 32 : c == 256 ? 128 : 288; };
            auto fetch_res = [&](int c) {
                const int col = col0 + out_c(c) + lcol;
#pragma unroll
                for (int st = 0; st < 4; ++st)
                    if (rmap[st].ok && col + 7 < col_limit)
                        rnext[st] = *reinterpret_cast<const uint4*>(P.residual + rmap[st].row * P.ldr + col);
            };
            if (pre_res && col0 + half * 32 < col_limit) fetch_res(half * 32);

            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            if (tl && warp == 2 && lane == 0) tl[6] = clock64();
            if (P.dbg & 1) goto epilogue_done;
            {
            const uint32_t taddr = tmem_base + (WIDE ? 0u : acc * 256) + ((uint32_t)(q * 32) << 16);

            if (P.epi == EPI_GEGLU) {
                // columns [0, BN/2) = value, [BN/2, BN) = gate (same output columns)
#pragma unroll 1
                for (int c = half * 32; c < BN / 2; c += 64) {
                    uint32_t rv[32], rg[32];
                    tmem_ld32(taddr + c, rv);
                    tmem_ld32(taddr + BN / 2 + c, rg);
                    tc_wait_ld();
                    float hv[4][8];
                    stage_chunk(stg, lane, rv);
                    __syncwarp();
#pragma unroll
                    for (int st = 0; st < 4; ++st) unstage8(stg, lane, st, hv[st]);
                    __syncwarp();
                    stage_chunk(stg, lane, rg);
                    __syncwarp();
                    const int col = col0 + c + lcol;
                    if (col < col_limit) {                   // aoz_gemm_bf16 requires N/2 % 8 == 0: col + 7 < col_limit too
                        uint32_t bh[4] = {0u, 0u, 0u, 0u}, bg[4] = {0u, 0u, 0u, 0u};
                        if (P.bias) {       // N/2 and the tile origin are multiples of 8, pointers checked: 16-byte aligned vectors
                            const uint4 t0 = __ldg(reinterpret_cast<const uint4*>(P.bias + col));
                            const uint4 t1 = __ldg(reinterpret_cast<const uint4*>(P.bias + P.geglu_half + col));
                            bh[0] = t0.x; bh[1] = t0.y; bh[2] = t0.z; bh[3] = t0.w;
                            bg[0] = t1.x; bg[1] = t1.y; bg[2] = t1.z; bg[3] = t1.w;
                        }
#pragma unroll
                        for (int st = 0; st < 4; ++st) {
                            float gv[8];
                            unstage8(stg, lane, st, gv);
                            if (!rmap[st].ok) continue;
                            const long long orow = rmap[st].row;
                            uint32_t ov[4], oh[4], og[4];
#pragma unroll
                            for (int e = 0; e < 8; e += 2) {
                                float h0 = hv[st][e] + bf16lo(bh[e >> 1]), h1 = hv[st][e + 1] + bf16hi(bh[e >> 1]);
                                float g0 = gv[e] + bf16lo(bg[e >> 1]), g1 = gv[e + 1] + bf16hi(bg[e >> 1]);
                                // autocast-faithful rounding points: linear out -> bf16, gelu -> bf16, product -> bf16
                                h0 = round_bf16(h0); h1 = round_bf16(h1); g0 = round_bf16(g0); g1 = round_bf16(g1);
                                oh[e >> 1] = pack_bf16(h0, h1);
                                og[e >> 1] = pack_bf16(g0, g1);
                                const float a0 = round_bf16(gelu_erf(g0)), a1 = round_bf16(gelu_erf(g1));
                                ov[e >> 1] = pack_bf16(h0 * a0, h1 * a1);
                            }
                            *reinterpret_cast<uint4*>(P.C + orow * P.ldc + col) = make_uint4(ov[0], ov[1], ov[2], ov[3]);
                            if (P.aux) {
                                *reinterpret_cast<uint4*>(P.aux + orow * P.ld_aux + col) = make_uint4(oh[0], oh[1], oh[2], oh[3]);
                                *reinterpret_cast<uint4*>(P.aux + orow * P.ld_aux + P.geglu_half + col) = make_uint4(og[0], og[1], og[2], og[3]);
                            }
                        }
                    }
                    __syncwarp();
                }
            } else if (wi.tail_slot >= 0) {
                // K slice of a tail tile: raw fp32 accumulator rows to the scratch buffer, [slice][128][BN]
                float* dstp = P.tail_ws + ((long long)(wi.tail_slot * m_sub + (int)rank) * BM + row_in_tile) * BN;
#pragma unroll 1
                for (int c = half * 32; c < BN; c += 64) {
                    uint32_t r[32];
                    if (!empty_split) {
                        tmem_ld32(taddr + c, r);
                        tc_wait_ld();
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) r[j] = 0u;
                    }
#pragma unroll
                    for (int j = 0; j < 32; j += 4) *reinterpret_cast<uint4*>(dstp + c + j) = make_uint4(r[j], r[j + 1], r[j + 2], r[j + 3]);
                }
            } else if (P.epi == EPI_PARTIAL) {
#pragma unroll 1
                for (int c = half * 32; c < OUT_COLS; c += 64) {
                    const int cbase = col0 + out_c(c);
                    if (cbase >= col_limit) { if (WIDE) continue; break; }          // warp-uniform
                    uint32_t r[32];
                    if (!empty_split) {
                        tmem_ld32(taddr + c, r);
                        tc_wait_ld();
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) r[j] = 0u;
                    }
                    if (!row_ok) continue;
                    float* dst = P.partial + ((long long)split * P.M + row) * P.N + col_shift + cbase;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        if (cbase + j + 3 < col_limit && ((((uintptr_t)(dst + j)) & 15) == 0)) {
                            *reinterpret_cast<uint4*>(dst + j) = make_uint4(r[j], r[j + 1], r[j + 2], r[j + 3]);
                        } else {
                            for (int e = 0; e < 4; ++e)
                                if (cbase + j + e < col_limit) dst[j + e] = __uint_as_float(r[j + e]);
                        }
                    }
                }
            } else if (P.vec_ok && !P.accumulate && P.rowgroup_bias == nullptr && P.mode != GM_CONV_WGRAD && col0 + BN <= col_limit &&
                       !empty_split && !(P.dbg & (8 | 16 | 32))) {
                // Fast store path (every Linear / conv-forward tile that lies inside the output: bias and / or residual, 16-byte
                // aligned rows).  The general loop below spends ~150 issued instructions per 8-column segment on per-segment address
                // arithmetic (64-bit row x stride products for C, the residual and the time-embedding rows), parameter re-loads and
                // the branches of epi_store8 -- with 8 epilogue warps on 4 schedulers that, not the store path, set the ~2500 cycles
                // per 32 x 32 chunk measured in round 1 (tools/gemm_timeline.py: 12.6 k cycles for a 320-wide tile).  Here the four
                // row pointers are formed once per tile, the bias vector travels with the residual prefetch and a segment is
                // 2 LDS + 8 FADD (+ 8 round + 8 FADD) + 4 pack + 1 STG.  Same operations in the same order: identical bits.
                const __nv_bfloat16* biasp = P.bias;
                const bool has_res = P.residual != nullptr;
                __nv_bfloat16* crow[4];
                const __nv_bfloat16* rrow[4];
#pragma unroll
                for (int st = 0; st < 4; ++st) {
                    crow[st] = pr.C + rmap[st].row * pr.ldc + col0 + lcol;
                    rrow[st] = has_res ? P.residual + rmap[st].row * P.ldr + col0 + lcol : nullptr;
                }
                uint4 bnext = make_uint4(0u, 0u, 0u, 0u);
                if (biasp) bnext = __ldg(reinterpret_cast<const uint4*>(biasp + col0 + out_c(half * 32) + lcol));
                // the accumulator chunk of the NEXT iteration is requested as soon as this one's registers are staged, so the
                // TMEM read (~300 cycles) runs under the four store steps
                uint32_t r[32];
                tmem_ld32(taddr + half * 32, r);
#pragma unroll 1
                for (int c = half * 32; c < BN; c += 64) {
                    uint4 rcur[4];
#pragma unroll
                    for (int st = 0; st < 4; ++st) rcur[st] = rnext[st];
                    const uint4 bcur = bnext;
                    if (c + 64 < BN) {
                        const int ocn = out_c(c + 64);
                        if (has_res) {
#pragma unroll
                            for (int st = 0; st < 4; ++st)
                                if (rmap[st].ok) rnext[st] = *reinterpret_cast<const uint4*>(rrow[st] + ocn);
                        }
                        if (biasp) bnext = __ldg(reinterpret_cast<const uint4*>(biasp + col0 + ocn + lcol));
                    }
                    tc_wait_ld();
                    stage_chunk(stg, lane, r);
                    __syncwarp();
                    if (c + 64 < BN) tmem_ld32(taddr + c + 64, r);
                    const int oc = out_c(c);
                    const uint32_t bw[4] = {bcur.x, bcur.y, bcur.z, bcur.w};
#pragma unroll
                    for (int st = 0; st < 4; ++st) {
                        float f[8];
                        unstage8(stg, lane, st, f);
                        if (biasp) {
#pragma unroll
                            for (int e = 0; e < 4; ++e) { f[2 * e] += bf16lo(bw[e]); f[2 * e + 1] += bf16hi(bw[e]); }
                        }
                        if (has_res) {
                            const uint32_t rw[4] = {rcur[st].x, rcur[st].y, rcur[st].z, rcur[st].w};
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                // round_bf16 of both values in one packed conversion (F2FP) instead of two F2F on the quarter-rate pipe
                                const uint32_t pk = pack_bf16(f[2 * e], f[2 * e + 1]);
                                f[2 * e] = bf16lo(pk) + bf16lo(rw[e]);
                                f[2 * e + 1] = bf16hi(pk) + bf16hi(rw[e]);
                            }
                        }
                        if (rmap[st].ok)
                            *reinterpret_cast<uint4*>(crow[st] + oc) =
                                make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
                    }
                    __syncwarp();
                }
            } else {
                // dbg 32 (experiments): CTA 0, first epilogue warp logs clock64 at its phase boundaries into the tail scratch
                const bool prof = (P.dbg & 32) && blockIdx.x == 0 && warp == 2 && lane == 0 && P.tail_ws != nullptr;
                long long* plog = reinterpret_cast<long long*>(P.tail_ws);
                int pslot = prof ? (int)plog[0] : 0;
                if (prof && pslot < 200) plog[1 + pslot++] = -clock64();         // negative: tile start (after the accumulator wait)
#pragma unroll 1
                for (int c = half * 32; c < OUT_COLS; c += 64) {
                    if (col0 + c >= col_limit) break;          // warp-uniform
                    uint4 rcur[4];
#pragma unroll
                    for (int st = 0; st < 4; ++st) rcur[st] = rnext[st];
                    if (pre_res && c + 64 < OUT_COLS && col0 + c + 64 < col_limit) fetch_res(c + 64);
                    uint32_t r[32];
                    if (!empty_split && !(P.dbg & 16)) {          // dbg 16 (experiments): epilogue without the TMEM read
                        tmem_ld32(taddr + c, r);
                        tc_wait_ld();
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) r[j] = 0u;
                    }
                    if (prof && pslot < 200) plog[1 + pslot++] = clock64();          // after the TMEM read
                    stage_chunk(stg, lane, r);
                    __syncwarp();
                    if (prof && pslot < 200) plog[1 + pslot++] = clock64();          // after staging
                    const int col = col0 + out_c(c) + lcol;
#pragma unroll
                    for (int st = 0; st < 4; ++st) {
                        float f[8];
                        unstage8(stg, lane, st, f);
                        if ((P.dbg & 8) && f[0] != 12345.678f) continue;      // dbg 8 (experiments): epilogue without the global stores
                        if (rmap[st].ok && col < col_limit)
                            epi_store8(P, pr.C, pr.ldc, rmap[st].row, rmap[st].group, col, col_limit, f, pre_res, rcur[st]);
                    }
                    __syncwarp();
                    if (prof && pslot < 200) plog[1 + pslot++] = clock64();          // after the four store steps
                }
                if (prof) plog[0] = pslot;
            }
            }
        epilogue_done:
            // release the accumulator buffer
            tc_fence_before();
            __syncwarp();
            if (tl && lane == 0) tl[8 + warp] = clock64();
            if (lane == 0) {
                if (CTA2 && !leader) mbar_arrive_cluster(mapa_rank(smem_u32(&tempty_bar[acc]), 0));
                else mbar_arrive(&tempty_bar[acc]);
            }
            if (++acc == (WIDE ? 1u : 2u)) { acc = 0; acc_phase ^= 1; }      // the wide plan has ONE accumulator: tiles of a CTA pair do not overlap
        }
    }

    tc_fence_before();
    if (CTA2) cluster_sync_all(); else __syncthreads();
    if (tl && threadIdx.x == 0) tl[7] = clock64();
    if (warp == 1) {
        tc_fence_after();
        if (CTA2) tmem_dealloc2(tmem_base, 512); else tmem_dealloc(tmem_base, 512);
    }
}

// ---- tail fix-up: sum the K slices of the tail tiles and apply the fused EPI_STORE epilogue -----------------------
// grid = tail_tiles x m_sub x 4 row blocks x (bn / 32) column blocks; a 128-thread block owns 32 rows x 32 columns:
// 4 lanes cover the 32 columns (128 B) of one row, so a warp reads 8 whole rows of a slice per step (coalesced) and
// writes 8 x 64-byte output segments.  Summing in the slices' own CTAs instead measured ~2.5 ms per step slower (DESIGN.md 4.2):
// the slices of a tile wait for the slowest sibling, and then few CTAs do the reduction this kernel spreads over thousands of threads.
__global__ void __launch_bounds__(128)
tail_fixup_kernel(const __grid_constant__ GemmParams P, int m_sub) {
    pdl_enter();
    const int chunks = P.bn / 32;
    int b = blockIdx.x;
    const int chunk = b % chunks; b /= chunks;
    const int rblk = b & 3; b >>= 2;
    const int sub = b % m_sub;
    const int t = b / m_sub;
    const Prob pr = select_prob(P, P.full_work + t);        // tail split implies splits == 1
    const int m_blk = (pr.ltile % pr.m_tiles) * m_sub + sub, n_blk = pr.ltile / pr.m_tiles;
    const int row_in_tile = rblk * 32 + (threadIdx.x >> 2);
    const int cq = (threadIdx.x & 3) * 8;                   // this lane's 8 columns inside the 32-column block
    const RowMap rm = map_row(P, pr.M, m_blk, row_in_tile);
    const int col = n_blk * P.bn + chunk * 32 + cq;
    if (!rm.ok || col >= pr.N) return;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    const long long slice_stride = (long long)m_sub * BM * P.bn;
    const float* src = P.tail_ws + ((long long)(t * P.tail_splits * m_sub + sub) * BM + row_in_tile) * P.bn + chunk * 32 + cq;
#pragma unroll 4
    for (int sp = 0; sp < P.tail_splits; ++sp) {
        const float4 v0 = *reinterpret_cast<const float4*>(src + sp * slice_stride);
        const float4 v1 = *reinterpret_cast<const float4*>(src + sp * slice_stride + 4);
        acc[0] += v0.x; acc[1] += v0.y; acc[2] += v0.z; acc[3] += v0.w;
        acc[4] += v1.x; acc[5] += v1.y; acc[6] += v1.z; acc[7] += v1.w;
    }
    epi_store8(P, pr.C, pr.ldc, rm.row, rm.group, col, pr.N, acc);
}

// ---- split-K reduction: sum fp32 partials, optional accumulate into existing bf16, optional OIHW permute ----
// partial: [splits][rows][cols] fp32.  out (bf16):
//   permute_taps == 0 : out[row*ld_out + col]                       (4 columns per thread, 128-bit loads)
//   permute_taps  > 0 : cols = taps*Cin, out is OIHW [rows=Cout][cin_real][taps]: one thread per (row, cin) gathers its
//                       taps (reads coalesced along cin) and writes them contiguously
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ partial, int splits, long long rows, long long cols,
                     __nv_bfloat16* __restrict__ out, long long ld_out, int permute_taps, int Cin, int cin_real, int accumulate) {
    pdl_enter();
    const long long total = rows * cols;
    if ((cols & 3) == 0 && (ld_out & 3) == 0 && ((((uintptr_t)out) & 7) == 0)) {
        const long long quads = total >> 2;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < quads; i += (long long)gridDim.x * blockDim.x) {
            const long long e = i << 2;
            float4 acc = *reinterpret_cast<const float4*>(partial + e);
            for (int k = 1; k < splits; ++k) {
                const float4 v = *reinterpret_cast<const float4*>(partial + (long long)k * total + e);
                acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
            }
            const long long row = e / cols, col = e - row * cols;
            __nv_bfloat16* o = out + row * ld_out + col;
            if (accumulate) {
                const uint2 old = *reinterpret_cast<const uint2*>(o);
                acc.x = round_bf16(acc.x) + bf16lo(old.x); acc.y = round_bf16(acc.y) + bf16hi(old.x);
                acc.z = round_bf16(acc.z) + bf16lo(old.y); acc.w = round_bf16(acc.w) + bf16hi(old.y);
            }
            *reinterpret_cast<uint2*>(o) = make_uint2(pack_bf16(acc.x, acc.y), pack_bf16(acc.z, acc.w));
        }
        return;
    }
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        float sum = 0.f;
        for (int k = 0; k < splits; ++k) sum += partial[(long long)k * total + i];
        const long long row = i / cols, col = i - row * cols;
        const long long o = row * ld_out + col;
        if (accumulate) sum = round_bf16(sum) + __bfloat162float(out[o]);
        out[o] = __float2bfloat16_rn(sum);
    }
}

// conv weight-gradient finish: partial [splits][rows][taps*Cin] fp32 -> OIHW bf16 [rows][cin_real][taps].
// One block = one output row x 128 input channels: per tap the 128 threads read 512 contiguous bytes of every split,
// the [cin][tap] block is transposed through shared memory (stride 9: conflict-free) and leaves as one contiguous run.
template <int TAPS>
__global__ void __launch_bounds__(128)
wgrad_permute_reduce_kernel(const float* __restrict__ partial, int splits, long long rows, int Cin, int cin_real,
                            __nv_bfloat16* __restrict__ out, int accumulate) {
    pdl_enter();
    __shared__ float sm[128 * TAPS];
    const long long row = blockIdx.y;
    const int c0 = blockIdx.x * 128, c = c0 + threadIdx.x;
    const long long cols = (long long)TAPS * Cin, total = rows * cols;
    if (c < Cin) {
        float sum[TAPS];
#pragma unroll
        for (int tap = 0; tap < TAPS; ++tap) sum[tap] = 0.f;
        const float* src = partial + row * cols + c;
        for (int k = 0; k < splits; ++k) {                      // all taps of a split in flight at once
#pragma unroll
            for (int tap = 0; tap < TAPS; ++tap) sum[tap] += __ldcs(src + (long long)k * total + (long long)tap * Cin);
        }
#pragma unroll
        for (int tap = 0; tap < TAPS; ++tap) sm[threadIdx.x * TAPS + tap] = sum[tap];
    }
    __syncthreads();
    const int nch = min(128, cin_real - c0);
    if (nch <= 0) return;
    __nv_bfloat16* o = out + (row * cin_real + c0) * TAPS;
    for (int i = threadIdx.x; i < nch * TAPS; i += 128) {
        float v = sm[i];
        if (accumulate) v = round_bf16(v) + __bfloat162float(o[i]);
        o[i] = __float2bfloat16_rn(v);
    }
}

static int g_dbg = 0;
static int g_force_bn = 0;        // > 0: experiments only (aoz_gemm_force_bn)
static int g_pair_mode = 1;       // 0 = single-CTA tiles only, 1 = the cost model may use CTA pairs (default), 2 = force pairs
// SMs the persistent GEMM / conv launches may occupy (0 = all).  Under data parallel NCCL's reduce-scatter / all-gather kernels run
// beside the reverse sweep: a persistent launch sized to all 148 SMs then has CTAs that cannot start until an NCCL CTA leaves their
// SM (231 KB of shared memory per GEMM CTA), and with static work assignment every such CTA holds the whole launch back.  Leaving
// NCCL its SMs (NCCL_MAX_CTAS of them) costs their share of the tensor throughput and removes the stall.
static int g_gemm_sm_budget = 0;
static inline int gemm_sms() {
    const int n = sm_count();
    return (g_gemm_sm_budget > 0 && g_gemm_sm_budget < n) ? g_gemm_sm_budget : n;
}
// Wide one-wave plan for outputs that are a little more than one wave of 256 x 256 pair tiles (4096 x 1280: 80 tiles on 74 pairs):
// 0 = off, 1 = the cost model may pick it (default), 2 = whenever the shape allows it.
static int g_wide_mode = 1;
static int g_wide_max_rounds = 2;       // rounds of 320-wide tiles the planner may consider (aoz_gemm_set_wide_max_rounds)
static int g_tail_mode = 1;       // 0 = never cut the last wave along K, 1 = the cost model may (default), 2 = whenever possible
static float* g_tail_ws = nullptr;        // caller-owned scratch for the tail slices (aoz_gemm_set_scratch)
static long long g_tail_bytes = 0;

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

template <bool CTA2>
static int launch_gemm_t(GemmParams& P, cudaStream_t stream) {
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncSetAttribute(gemm_bf16_kernel<CTA2>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_TOTAL);
        attr_set = true;
    }
    // P.m_tiles counts work-unit rows here (256-row pair tiles when CTA2); the planner's tail decision is in P.tail_*
    const int tiles = P.m_tiles * P.n_tiles;
    if (P.tail_tiles > 0) {
        P.full_work = tiles - P.tail_tiles;
        P.tail_ws = g_tail_ws;
    } else {
        P.full_work = tiles * P.splits;
        P.tail_tiles = 0; P.tail_splits = 1;
    }
    const int total_work = P.full_work + P.tail_tiles * P.tail_splits;
    if (total_work <= 0) return AOZ_OK;
    P.dbg = g_dbg;
    if (g_dbg & (32 | 64)) P.tail_ws = g_tail_ws;            // epilogue clock log goes to the scratch buffer
    const int b_rows = CTA2 ? P.bn / 2 : P.bn;
    const int stage_bytes = BM * BK * 2 + (P.b_mn ? ((b_rows + 63) / 64) * 8192 : b_rows * BK * 2);
    if (P.bn == 320) {
        const bool epi_ok = P.mode == GM_CONV_WGRAD ? P.epi == EPI_PARTIAL : P.epi == EPI_STORE;
        if (!CTA2 || !epi_ok || P.n_groups || P.tail_tiles) {
            set_error("gemm: the 320-wide plan needs CTA pairs, a store epilogue (fp32 partials for conv weight gradients) and no tail split");
            return AOZ_ERR_ARG;
        }
    }
    P.stages = SMEM_TILE_BYTES / stage_bytes;
    if (P.stages > MAX_STAGES) P.stages = MAX_STAGES;
    if (!CTA2) {
        const int grid = total_work < gemm_sms() ? total_work : gemm_sms();
        launch_k(gemm_bf16_kernel<false>, dim3(grid), dim3(GEMM_THREADS), (size_t)(GEMM_SMEM_TOTAL), stream, P);
    } else {
        const int pairs = gemm_sms() / 2;
        const int grid = 2 * (total_work < pairs ? total_work : pairs);
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(GEMM_THREADS); cfg.dynamicSmemBytes = GEMM_SMEM_TOTAL; cfg.stream = stream;
        cudaLaunchAttribute at[2];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[1].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = g_pdl ? 2 : 1;
        cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_bf16_kernel<true>, P);
        if (e != cudaSuccess) { set_error("gemm_bf16_kernel<pair> launch: %s", cudaGetErrorString(e)); return AOZ_ERR_CUDA; }
    }
    AOZ_CHECK_LAUNCH("gemm_bf16_kernel");
    if (P.tail_tiles > 0) {
        const int m_sub = CTA2 ? 2 : 1;
        launch_k(tail_fixup_kernel, dim3(P.tail_tiles * m_sub * 4 * (P.bn / 32)), dim3(128), (size_t)(0), stream, P, m_sub);
        AOZ_CHECK_LAUNCH("tail_fixup_kernel");
    }
    return AOZ_OK;
}

// ---- host-side tile / split selection ------------------------------------------------------------------------
// Cycle model per CTA (or CTA pair) and K iteration of 64: the MMA needs 2*bn cycles (128 x bn x 64 at 8192 FLOP/cycle/SM),
// shared memory must deliver the A (16 KB) and B (b_rows x 128 B) stage at 128 B/cycle.  A launch costs
// rounds x max(main loop, epilogue) + one exposed epilogue + fixed fill/drain; the N extent is covered by ceil(N / n_out) tiles.
struct TilePlan { int bn; bool pair; int n_tiles; double cycles; int tail_tiles, tail_splits; };

// `allow_tail`: the caller's epilogue is EPI_STORE with splits == 1, so the last (partial) wave may be cut along K instead
// (decode_work / tail_fixup_kernel): 80 tiles on 74 CTA pairs then cost ~1.1 tile times instead of 2.
// core: `units_of(pair, bn, &n_tiles)` = number of work units (tiles x splits) for a candidate tile shape
template <class UnitsFn>
static TilePlan plan_tiles_core(UnitsFn units_of, bool can_pair, int k_iters_per_unit, int splits, bool b_mn, bool geglu, bool allow_tail) {
    TilePlan best{128, false, 0, 1e300, 0, 1}, best_tail{128, false, 0, 1e300, 0, 1};
    const int sms = gemm_sms();
    const int step = b_mn ? 64 : 32;
    for (int pair = 0; pair <= 1; ++pair) {
        if (pair && (g_pair_mode == 0 || !can_pair)) continue;
        if (!pair && g_pair_mode == 2 && can_pair) continue;
        for (int bn = 64; bn <= 256; bn += step) {
            if (g_force_bn > 0 && bn != g_force_bn) continue;
            if (geglu && bn != 256 && bn != 128) continue;
            if (pair && (bn % (2 * step))) continue;
            int n_tiles = 0;
            const long long units = units_of(pair != 0, bn, &n_tiles);
            const int slots = pair ? sms / 2 : sms;
            const double rounds = (double)((units + slots - 1) / slots);
            // cycles per K iteration, calibrated on B200 (tools/gemm_sweep.py, profiles/r01_gemm_sweep.json): a ~540-cycle
            // floor per iteration, then growth with the tile width; a CTA pair shares B and grows more slowly
            const double cyc = pair ? fmax(535.0, 535.0 + (bn - 64) * 0.30 + fmax(0.0, bn - 128.0) * 0.85)
                                    : fmax(535.0, 535.0 + (bn - 64) * 0.60 + fmax(0.0, bn - 160.0) * 1.95);
            const double epi = (geglu ? 12.0 : 6.0) * bn + 400.0;
            const double main_loop = k_iters_per_unit * cyc;
            const double total = rounds * fmax(main_loop, epi) + epi + 3000.0;
            if (total < best.cycles) best = TilePlan{bn, pair != 0, n_tiles, total, 0, 1};
            // the same tiles with the last wave cut along K
            const int r = (int)(units % slots);
            if (allow_tail && g_tail_mode > 0 && splits == 1 && !geglu && r > 0 && g_tail_ws) {
                int ts_max = slots / r;
                if (ts_max > k_iters_per_unit / 2) ts_max = k_iters_per_unit / 2;
                if (ts_max > 16) ts_max = 16;
                for (int ts = 2; ts <= ts_max; ++ts) {
                    const long long ws_bytes = (long long)r * ts * (pair ? 2 : 1) * BM * bn * 4;
                    if (ws_bytes > g_tail_bytes) break;
                    const double full_rounds = (double)(units / slots);
                    const double slice = ceil_div(k_iters_per_unit, ts) * cyc;
                    const double fix = 6000.0 + (double)ws_bytes * 2.0 / 3000.0;         // extra launch + partial write / read
                    const double t2 = full_rounds * fmax(main_loop, epi) + slice + 4.0 * bn + 400.0 + epi + 3000.0 + fix;
                    if (t2 < best_tail.cycles) best_tail = TilePlan{bn, pair != 0, n_tiles, t2, r, ts};
                }
            }
        }
    }
    if (best_tail.tail_tiles > 0 && (g_tail_mode == 2 || best_tail.cycles < best.cycles)) return best_tail;
    return best;
}

// `allow_tail`: the caller's epilogue is EPI_STORE with splits == 1, so the last (partial) wave may be cut along K instead
// (decode_work / tail_fixup_kernel): 80 tiles on 74 CTA pairs then cost ~1.1 tile times instead of 2.
static TilePlan plan_tiles(int m_tiles128, int n_extent, int k_iters_per_unit, int splits, bool b_mn, bool geglu, int n_groups /*taps*/,
                           bool allow_tail = false) {
    auto units_of = [&](bool pair, int bn, int* n_tiles) -> long long {
        const int n_out = geglu ? bn / 2 : bn;
        *n_tiles = n_groups * ceil_div(n_extent, n_out);
        return (long long)(pair ? ceil_div(m_tiles128, 2) : m_tiles128) * (*n_tiles) * splits;
    };
    return plan_tiles_core(units_of, m_tiles128 >= 2, k_iters_per_unit, splits, b_mn, geglu, allow_tail);
}

// Wide one-wave plan (see the kernel's WIDE note): cycles by the model above, or 1e300 where the shape does not allow it.  One round:
// main loop (MMA-bound: 640 cycles per K iteration at full clock, calibrated like plan_tiles_core) + the exposed epilogue of a
// 320-wide tile + fill / drain.
static double wide_plan_cycles(int m_tiles128, int N, int k_iters) {
    if (g_wide_mode == 0 || g_pair_mode == 0 || g_force_bn != 0 || (N % 320) != 0 || m_tiles128 < 2) return 1e300;
    if (g_tail_mode == 2 && g_wide_mode != 2) return 1e300;             // a forced tail split (tests / experiments) keeps its plan
    const long long units = (long long)ceil_div(m_tiles128, 2) * (N / 320);
    const int slots = gemm_sms() / 2;
    const long long rounds = (units + slots - 1) / slots;
    if (rounds > g_wide_max_rounds) return 1e300;
    // one accumulator: main loop and epilogue of a pair's tiles run back to back
    return (double)rounds * ((double)k_iters * 775.0 + 2.0 * (6.0 * 320 + 400.0)) + 3000.0;
}

// split-K factor for un-fused GEMMs: trades wave quantisation against fp32 partial traffic.  `store_direct`: with one split
// the result is stored straight from the epilogue (Linear layers), so the tail split is available as an alternative to
// split-K; conv weight gradients always go through fp32 partials + the permuting reduce.
static int plan_splits(int m_tiles128, int n_extent, int k_iters, long long out_elems, bool b_mn, int n_groups, bool store_direct) {
    int best_s = 1;
    double best_c = 1e300;
    for (int s = 1; s <= 32 && s <= (k_iters + 1) / 2; ++s) {
        const int kit = ceil_div(k_iters, s);
        TilePlan tp = plan_tiles(m_tiles128, n_extent, kit, s, b_mn, false, n_groups, /*allow_tail=*/store_direct && s == 1);
        double c = tp.cycles;
        if (s == 1 && store_direct && n_groups == 1) c = fmin(c, wide_plan_cycles(m_tiles128, n_extent, k_iters));
        // partial write + reduce read, measured ~1.6 B/cycle/SM-equivalent on B200 (tools/kernel_times.py), + a launch
        if (s > 1 || !store_direct) c += (double)(2 * s + 1) * out_elems * 4.0 / 2400.0 / 2.0 + 4000.0;
        if (c < best_c) { best_c = c; best_s = s; }
    }
    return best_s;
}

static int launch_gemm(GemmParams& P, bool pair, cudaStream_t stream) {
    if (pair) {
        P.m_tiles = (P.m_tiles + 1) / 2;
        return launch_gemm_t<true>(P, stream);
    }
    return launch_gemm_t<false>(P, stream);
}

}  // namespace aoz

using namespace aoz;

extern "C" {

// 0 = single-CTA tiles only, 1 = cost model may choose CTA-pair (cta_group::2) tiles (default), 2 = force pairs
int aoz_gemm_set_pair_mode(int mode) { g_pair_mode = mode; return AOZ_OK; }
int aoz_gemm_set_sm_budget(int sms) { g_gemm_sm_budget = sms > 0 ? (sms & ~1) : 0; return AOZ_OK; }      // even: CTA pairs

// 0 = never split the last wave along K, 1 = cost model decides (default), 2 = split whenever the shape allows it
int aoz_gemm_set_tail_mode(int mode) { g_tail_mode = mode; return AOZ_OK; }
// 0 = never use the 320-wide one-wave plan, 1 = cost model decides (default), 2 = whenever the shape allows it
int aoz_gemm_set_wide_mode(int mode) { g_wide_mode = mode; return AOZ_OK; }
// rounds of 320-wide tiles the planner may consider (default 2; 1 = only one-wave launches)
int aoz_gemm_set_wide_max_rounds(int rounds) { g_wide_max_rounds = rounds < 1 ? 1 : rounds; return AOZ_OK; }

// Caller-owned fp32 scratch for the K slices of tail tiles (stream-ordered: every GEMM that uses it must run on the
// same stream).  Without it the tail split is off.  20 MB covers every shape (148 slices x 128 x 256 floats).
int aoz_gemm_set_scratch(void* ptr, long long bytes) {
    g_tail_ws = (float*)ptr;
    g_tail_bytes = ptr ? bytes : 0;
    return AOZ_OK;
}

int aoz_gemm_force_bn(int bn) { g_force_bn = bn; return AOZ_OK; }
int aoz_gemm_debug_flags(int flags) { g_dbg = flags; return AOZ_OK; }

// what the planner picks for C[M,N] = A[M,K] B with `splits` (<= 0: automatic): bn + 1000*pair + 10000*tail_splits +
// 1000000*tail_tiles + 100000000*splits  (tools / tests only)
long long aoz_gemm_describe_plan(int M, int N, int K, int b_mn, int splits) {
    const int mt = ceil_div(M, BM), kit = ceil_div(K, BK);
    if (splits <= 0) splits = plan_splits(mt, N, kit, (long long)M * N, b_mn != 0, 1, true);
    TilePlan tp = plan_tiles(mt, N, ceil_div(kit, splits), splits, b_mn != 0, false, 1, splits == 1);
    if (splits == 1) {
        const double cyc = wide_plan_cycles(mt, N, kit);
        if (cyc < 1e299 && (g_wide_mode == 2 || cyc < tp.cycles)) tp = TilePlan{320, true, N / 320, cyc, 0, 1};
    }
    return tp.bn + 1000LL * tp.pair + 10000LL * (tp.tail_tiles ? tp.tail_splits : 0) + 1000000LL * tp.tail_tiles + 100000000LL * splits;
}

// split-K factor aoz_gemm_bf16 will use when called with splits <= 0 (so the caller can size the workspace)
int aoz_gemm_auto_splits(int M, int N, int K, int b_mn) {
    return plan_splits(ceil_div(M, BM), N, ceil_div(K, BK), (long long)M * N, b_mn != 0, 1, true);
}
int aoz_conv_wgrad_auto_splits(int NB, int H, int W, int Cout, int Cin, int ks) {
    const int k_iters = NB * ceil_div(H, 8) * ceil_div(W, 8);
    return plan_splits(ceil_div(Cout, BM), Cin, k_iters, (long long)Cout * ks * ks * Cin, true, ks * ks, false);
}

// C[M,N] (bf16) = op(A) * op(B)^T-ish with fused epilogue.
//   a_mn == 0: A is [M, K] row-major (lda elements)       a_mn == 1: A is [K, M] row-major (lda)
//   b_mn == 0: B is [N, K] row-major (ldb)                 b_mn == 1: B is [K, N] row-major (ldb)
//   bias [N] / rowgroup_bias [M/rows_per_group, N] / residual [M, N] (ldr) optional (null = absent)
//   epi == EPI_GEGLU: B is [2*half, K]; C is [M, half]; aux (optional) receives the bf16 pre-activation [M, 2*half]
//   splits > 1: `workspace` must hold splits*M*N floats; the result is reduced into C afterwards
int aoz_gemm_bf16(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn, void* C, long long ldc,
                  int M, int N, int K, const void* bias, const void* rowgroup_bias, int rows_per_group, long long ld_rgb,
                  const void* residual, long long ldr, int epi, void* aux, long long ld_aux, int accumulate, int splits,
                  void* workspace, void* stream) {
    AOZ_CHECK_ARG(A && B && C, "aoz_gemm_bf16: null operand");
    AOZ_CHECK_ARG(M > 0 && N > 0 && K > 0, "aoz_gemm_bf16: bad extents M=%d N=%d K=%d", M, N, K);
    AOZ_CHECK_ARG((lda % 8) == 0 && (ldb % 8) == 0, "aoz_gemm_bf16: lda/ldb must be multiples of 8 elements (TMA 16-byte strides)");
    AOZ_CHECK_ARG((((uintptr_t)A | (uintptr_t)B) & 15) == 0, "aoz_gemm_bf16: operands must be 16-byte aligned");
    AOZ_CHECK_ARG(epi == EPI_STORE || epi == EPI_GEGLU, "aoz_gemm_bf16: bad epilogue %d", epi);
    const bool fused = bias || residual || rowgroup_bias || epi == EPI_GEGLU || accumulate;
    GemmParams P;
    memset(&P, 0, sizeof(P));
    P.mode = GM_LINEAR; P.epi = epi; P.a_mn = a_mn; P.b_mn = b_mn;
    P.M = M; P.N = N; P.K = K;
    P.k_iters = ceil_div(K, BK);
    P.m_tiles = ceil_div(M, BM);
    if (splits <= 0) splits = fused ? 1 : plan_splits(P.m_tiles, N, P.k_iters, (long long)M * N, b_mn != 0, 1, true);
    if (splits > P.k_iters) splits = P.k_iters;
    const bool geglu = epi == EPI_GEGLU;
    if (geglu) {
        AOZ_CHECK_ARG((N % 2) == 0 && !b_mn && splits == 1, "aoz_gemm_bf16: GEGLU needs even N, K-major B, no split");
        // the GEGLU epilogue loads bias and stores C / aux as 16-byte vectors of 8 columns with no scalar tail
        AOZ_CHECK_ARG(((N / 2) % 8) == 0, "aoz_gemm_bf16: GEGLU needs N/2 to be a multiple of 8 (got N=%d)", N);
        AOZ_CHECK_ARG(((((uintptr_t)C | (uintptr_t)aux | (uintptr_t)bias) & 15) == 0) && (ldc % 8) == 0 && (!aux || (ld_aux % 8) == 0),
                      "aoz_gemm_bf16: GEGLU needs 16-byte aligned C / aux / bias and ldc / ld_aux multiples of 8 elements");
        P.geglu_half = N / 2;
    }
    if (splits > 1) {
        AOZ_CHECK_ARG(workspace != nullptr, "aoz_gemm_bf16: split-K needs a workspace");
        AOZ_CHECK_ARG(!bias && !residual && !rowgroup_bias, "aoz_gemm_bf16: split-K does not fuse bias/residual");
    }
    const int kit = ceil_div(P.k_iters, splits);
    TilePlan tp = plan_tiles(P.m_tiles, geglu ? N / 2 : N, kit, splits, b_mn != 0, geglu, 1, /*allow_tail=*/splits == 1 && !geglu);
    if (!geglu && splits == 1) {
        const double cyc = wide_plan_cycles(P.m_tiles, N, kit);
        if (cyc < 1e299 && (g_wide_mode == 2 || cyc < tp.cycles)) tp = TilePlan{320, true, N / 320, cyc, 0, 1};
    }
    const int bn = tp.bn;
    const bool pair = tp.pair;
    P.bn = bn;
    P.n_tiles = tp.n_tiles;
    P.splits = splits;
    P.tail_tiles = tp.tail_tiles; P.tail_splits = tp.tail_splits;
    P.vec_ok = ((((uintptr_t)C | (uintptr_t)bias | (uintptr_t)rowgroup_bias | (uintptr_t)residual) & 15) == 0) && (ldc % 8) == 0 &&
               (ld_rgb % 8) == 0 && (ldr % 8) == 0;
    if (splits > 1) {
        P.epi = EPI_PARTIAL;
        P.partial = (float*)workspace;
    }
    P.C = (__nv_bfloat16*)C; P.ldc = ldc;
    P.bias = (const __nv_bfloat16*)bias;
    P.rowgroup_bias = (const __nv_bfloat16*)rowgroup_bias; P.rows_per_group = rows_per_group; P.ld_rgb = ld_rgb;
    P.residual = (const __nv_bfloat16*)residual; P.ldr = ldr;
    P.aux = (__nv_bfloat16*)aux; P.ld_aux = ld_aux;
    P.accumulate = accumulate;
    int rc;
    {   // A map
        uint64_t dims[2], strides[1]; uint32_t box[2];
        if (!a_mn) { dims[0] = K; dims[1] = M; box[0] = 64; box[1] = BM; }
        else       { dims[0] = M; dims[1] = K; box[0] = 64; box[1] = BK; }
        strides[0] = (uint64_t)lda * 2;
        if ((rc = make_tmap_bf16(&P.tmA, A, 2, dims, strides, box, nullptr)) != AOZ_OK) return rc;
    }
    {   // B map
        uint64_t dims[2], strides[1]; uint32_t box[2];
        const int b_rows = pair ? bn / 2 : bn;
        if (!b_mn) { dims[0] = K; dims[1] = N; box[0] = 64; box[1] = (uint32_t)((geglu && !pair) ? bn / 2 : b_rows); }
        else       { dims[0] = N; dims[1] = K; box[0] = 64; box[1] = BK; }
        strides[0] = (uint64_t)ldb * 2;
        if ((rc = make_tmap_bf16(&P.tmB, B, 2, dims, strides, box, nullptr)) != AOZ_OK) return rc;
    }
    if ((rc = launch_gemm(P, pair, (cudaStream_t)stream)) != AOZ_OK) return rc;
    if (splits > 1) {
        const long long total = ((long long)M * N + 3) / 4;
        int grid = (int)((total + 255) / 256); if (grid > sm_count() * 16) grid = sm_count() * 16;
        launch_k(splitk_reduce_kernel, dim3(grid), dim3(256), (size_t)(0), (cudaStream_t)stream, (const float*)workspace, splits, M, N, (__nv_bfloat16*)C,
                                                                    ldc, 0, 0, 0, accumulate);
        AOZ_CHECK_LAUNCH("splitk_reduce_kernel");
    }
    return AOZ_OK;
}

// Grouped GEMM: C_g[M_g, N_g] = op(A_g) op(B_g) for g in [0, n), n <= 10, ONE persistent launch.  All problems share K, the
// operand majors and the tile shape; plain bf16 store (no bias / residual / split-K).  Built for the weight gradients of
// one transformer block (dW = dy^T x for to_q/k/v, to_out, ff.*: ~900 tiles that fill 148 SMs in ~6 full waves).
// A_ptrs / B_ptrs / C_ptrs: HOST arrays of n device pointers (uint64); lda / ldb / ldc: HOST int64[n]; M / N: HOST int32[n].
int aoz_gemm_grouped_bf16(int n, const void* A_ptrs, const void* lda, const void* B_ptrs, const void* ldb, const void* C_ptrs,
                          const void* ldc, const void* M, const void* N, int K, int a_mn, int b_mn, void* stream) {
    AOZ_CHECK_ARG(n >= 1 && n <= MAX_GROUPS, "aoz_gemm_grouped_bf16: 1..%d problems per launch (got %d)", MAX_GROUPS, n);
    AOZ_CHECK_ARG(A_ptrs && B_ptrs && C_ptrs && lda && ldb && ldc && M && N && K > 0, "aoz_gemm_grouped_bf16: bad arguments");
    const uint64_t* Ap = (const uint64_t*)A_ptrs; const uint64_t* Bp = (const uint64_t*)B_ptrs; const uint64_t* Cp = (const uint64_t*)C_ptrs;
    const long long* la = (const long long*)lda; const long long* lb = (const long long*)ldb; const long long* lc = (const long long*)ldc;
    const int* Ms = (const int*)M; const int* Ns = (const int*)N;
    GemmParams P;
    memset(&P, 0, sizeof(P));
    P.mode = GM_LINEAR; P.epi = EPI_STORE; P.a_mn = a_mn; P.b_mn = b_mn;
    P.K = K; P.k_iters = ceil_div(K, BK);
    P.splits = 1;
    P.n_groups = n;
    bool can_pair = true, aligned = true;
    for (int g = 0; g < n; ++g) {
        AOZ_CHECK_ARG(Ap[g] && Bp[g] && Cp[g] && Ms[g] > 0 && Ns[g] > 0, "aoz_gemm_grouped_bf16: problem %d is empty", g);
        AOZ_CHECK_ARG((la[g] % 8) == 0 && (lb[g] % 8) == 0 && ((Ap[g] | Bp[g]) & 15) == 0, "aoz_gemm_grouped_bf16: problem %d operand alignment", g);
        if (Ms[g] <= BM) can_pair = false;
        if ((Cp[g] & 15) || (lc[g] % 8)) aligned = false;
    }
    auto units_of = [&](bool pair, int bn, int* n_tiles) -> long long {
        long long u = 0;
        for (int g = 0; g < n; ++g) u += (long long)ceil_div(Ms[g], pair ? 2 * BM : BM) * ceil_div(Ns[g], bn);
        *n_tiles = 1;
        return u;
    };
    const TilePlan tp = plan_tiles_core(units_of, can_pair, P.k_iters, 1, b_mn != 0, false, /*allow_tail=*/true);
    const int bn = tp.bn;
    const bool pair = tp.pair;
    P.bn = bn;
    P.vec_ok = aligned;
    int rc, tile_start = 0;
    for (int g = 0; g < n; ++g) {
        GroupDesc& d = P.grp[g];
        d.C = (__nv_bfloat16*)Cp[g]; d.ldc = lc[g]; d.M = Ms[g]; d.N = Ns[g];
        d.m_tiles = ceil_div(Ms[g], pair ? 2 * BM : BM);
        d.tile_start = tile_start;
        tile_start += d.m_tiles * ceil_div(Ns[g], bn);
        {
            uint64_t dims[2], strides[1]; uint32_t box[2];
            if (!a_mn) { dims[0] = K; dims[1] = Ms[g]; box[0] = 64; box[1] = BM; }
            else       { dims[0] = Ms[g]; dims[1] = K; box[0] = 64; box[1] = BK; }
            strides[0] = (uint64_t)la[g] * 2;
            if ((rc = make_tmap_bf16(&d.tmA, (const void*)Ap[g], 2, dims, strides, box, nullptr)) != AOZ_OK) return rc;
        }
        {
            uint64_t dims[2], strides[1]; uint32_t box[2];
            if (!b_mn) { dims[0] = K; dims[1] = Ns[g]; box[0] = 64; box[1] = (uint32_t)(pair ? bn / 2 : bn); }
            else       { dims[0] = Ns[g]; dims[1] = K; box[0] = 64; box[1] = BK; }
            strides[0] = (uint64_t)lb[g] * 2;
            if ((rc = make_tmap_bf16(&d.tmB, (const void*)Bp[g], 2, dims, strides, box, nullptr)) != AOZ_OK) return rc;
        }
    }
    // launch_gemm_t takes the tile count as m_tiles * n_tiles
    P.m_tiles = tile_start; P.n_tiles = 1;
    P.tail_tiles = tp.tail_tiles; P.tail_splits = tp.tail_splits;
    return pair ? launch_gemm_t<true>(P, (cudaStream_t)stream) : launch_gemm_t<false>(P, (cudaStream_t)stream);
}

// Implicit-GEMM convolution forward over NHWC bf16 (also used for dgrad with a flipped, transposed weight pack).
//   x      : [NB, Hin, Win, Cin]  (Cin multiple of 8; channel count seen by TMA)
//   wpack  : [Cout, taps * cin_chunks*64] bf16, K index = tap*(cin_chunks*64) + cin  (zero padded)
//   y      : [NB, H, W, Cout] with H = (Hin + 2*pad - ks)/stride + 1
//   flip   : traverse the taps mirrored (dgrad)
int aoz_conv_fwd_bf16(const void* x, int NB, int Hin, int Win, int Cin, const void* wpack, int Cout, int ks, int stride,
                      int pad, int flip, void* y, const void* bias, const void* rowgroup_bias, const void* residual,
                      int accumulate, void* stream) {
    AOZ_CHECK_ARG(x && wpack && y, "aoz_conv_fwd_bf16: null operand");
    AOZ_CHECK_ARG(ks == 3 || ks == 1, "aoz_conv_fwd_bf16: kernel size %d", ks);
    AOZ_CHECK_ARG(stride == 1 || stride == 2, "aoz_conv_fwd_bf16: stride %d", stride);
    AOZ_CHECK_ARG((Cin % 8) == 0, "aoz_conv_fwd_bf16: Cin must be a multiple of 8 (got %d)", Cin);
    const int H = (Hin + 2 * pad - ks) / stride + 1, W = (Win + 2 * pad - ks) / stride + 1;
    GemmParams P;
    memset(&P, 0, sizeof(P));
    P.mode = GM_CONV_FWD; P.epi = EPI_STORE;
    P.NB = NB; P.H = H; P.W = W;
    P.TW = W >= 16 ? 16 : 8; P.TH = BM / P.TW;
    if (stride == 2) { P.TW = 8; P.TH = 16; }              // box extents are limited to 256 along each dim
    P.tiles_h = ceil_div(H, P.TH); P.tiles_w = ceil_div(W, P.TW);
    P.taps_s = ks; P.pad = pad; P.stride = stride; P.flip = flip;
    P.cin_chunks = ceil_div(Cin, 64);
    P.k_iters = ks * ks * P.cin_chunks;
    P.M = NB * H * W; P.N = Cout; P.K = P.k_iters * 64;
    P.m_tiles = NB * P.tiles_h * P.tiles_w;
    TilePlan tp = plan_tiles(P.m_tiles, Cout, P.k_iters, 1, false, false, 1, /*allow_tail=*/true);
    {   // the 320-wide plan (one or two rounds of 256 x 320 tiles): 1280- and 640-channel convolutions at 32 x 32 / 64 x 64
        const double cyc = wide_plan_cycles(P.m_tiles, Cout, P.k_iters);
        if (cyc < 1e299 && (g_wide_mode == 2 || cyc < tp.cycles)) tp = TilePlan{320, true, Cout / 320, cyc, 0, 1};
    }
    const int bn = tp.bn;
    const bool pair = tp.pair;
    P.bn = bn;
    P.n_tiles = tp.n_tiles;
    P.splits = 1;
    P.tail_tiles = tp.tail_tiles; P.tail_splits = tp.tail_splits;
    P.vec_ok = ((((uintptr_t)y | (uintptr_t)bias | (uintptr_t)rowgroup_bias | (uintptr_t)residual) & 15) == 0) && (Cout % 8) == 0;
    P.C = (__nv_bfloat16*)y; P.ldc = Cout;
    P.bias = (const __nv_bfloat16*)bias;
    P.rowgroup_bias = (const __nv_bfloat16*)rowgroup_bias; P.ld_rgb = Cout;
    P.residual = (const __nv_bfloat16*)residual; P.ldr = Cout;
    P.accumulate = accumulate;
    int rc;
    {
        uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)Win, (uint64_t)Hin, (uint64_t)NB};
        uint64_t strides[3] = {(uint64_t)Cin * 2, (uint64_t)Win * Cin * 2, (uint64_t)Hin * Win * Cin * 2};
        uint32_t box[4] = {64, (uint32_t)(P.TW * stride), (uint32_t)(P.TH * stride), 1};
        uint32_t es[4] = {1, (uint32_t)stride, (uint32_t)stride, 1};
        if ((rc = make_tmap_bf16(&P.tmA, x, 4, dims, strides, box, es)) != AOZ_OK) return rc;
    }
    {
        uint64_t dims[2] = {(uint64_t)P.K, (uint64_t)Cout};
        uint64_t strides[1] = {(uint64_t)P.K * 2};
        uint32_t box[2] = {64, (uint32_t)(pair ? bn / 2 : bn)};
        if ((rc = make_tmap_bf16(&P.tmB, wpack, 2, dims, strides, box, nullptr)) != AOZ_OK) return rc;
    }
    return launch_gemm(P, pair, (cudaStream_t)stream);
}

// Convolution weight gradient: dW[cout][tap][cin] = sum_pixels dy[pix][cout] * x[pix*stride + tap - pad][cin].
//   dy : [NB, H, W, Cout], x : [NB, Hin, Win, Cin], grad_w : OIHW bf16 [Cout, cin_real, ks, ks] (the parameter layout;
//   cin_real <= Cin drops zero-padded input channels, e.g. conv_in's 4 real channels of 8)
//   workspace : splits * Cout * taps*Cin floats
int aoz_conv_wgrad_bf16(const void* dy, const void* x, int NB, int H, int W, int Cout, int Hin, int Win, int Cin, int ks,
                        int stride, int pad, int cin_real, void* grad_w, int accumulate, int splits, void* workspace, void* stream) {
    AOZ_CHECK_ARG(dy && x && grad_w && workspace, "aoz_conv_wgrad_bf16: null operand");
    if (cin_real <= 0 || cin_real > Cin) cin_real = Cin;
    AOZ_CHECK_ARG((Cin % 8) == 0 && (Cout % 8) == 0, "aoz_conv_wgrad_bf16: channel counts must be multiples of 8");
    GemmParams P;
    memset(&P, 0, sizeof(P));
    P.mode = GM_CONV_WGRAD; P.epi = EPI_PARTIAL; P.a_mn = 1; P.b_mn = 1;
    P.NB = NB; P.H = H; P.W = W; P.TH = 8; P.TW = 8;
    P.tiles_h = ceil_div(H, 8); P.tiles_w = ceil_div(W, 8);
    P.taps_s = ks; P.pad = pad; P.stride = stride;
    P.Cin = Cin;
    const int taps = ks * ks;
    P.M = Cout; P.N = taps * Cin; P.K = NB * H * W;
    P.k_iters = NB * P.tiles_h * P.tiles_w;
    P.m_tiles = ceil_div(Cout, BM);
    if (splits <= 0) splits = plan_splits(P.m_tiles, Cin, P.k_iters, (long long)Cout * taps * Cin, true, taps, false);
    if (splits > P.k_iters) splits = P.k_iters;
    TilePlan tp = plan_tiles(P.m_tiles, Cin, ceil_div(P.k_iters, splits), splits, true, false, taps);
    if (g_wide_mode > 0 && g_pair_mode != 0 && g_force_bn == 0 && (Cin % 320) == 0 && P.m_tiles >= 2 && !(g_tail_mode == 2 && g_wide_mode != 2)) {
        // 320-wide tiles: any number of rounds (a K iteration is 64 pixels, the single accumulator's exposed epilogue is small against it)
        const long long units = (long long)ceil_div(P.m_tiles, 2) * taps * (Cin / 320) * splits;
        const int slots = gemm_sms() / 2;
        const double cyc = (double)((units + slots - 1) / slots) * ((double)ceil_div(P.k_iters, splits) * 775.0 + 2.0 * (6.0 * 320 + 400.0)) + 3000.0;
        if (g_wide_mode == 2 || cyc < tp.cycles) tp = TilePlan{320, true, taps * (Cin / 320), cyc, 0, 1};
    }
    const int bn = tp.bn;
    P.bn = bn;
    P.n_tiles_per_tap = ceil_div(Cin, bn);
    P.n_tiles = taps * P.n_tiles_per_tap;
    P.splits = splits;
    P.partial = (float*)workspace;
    int rc;
    {
        uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)W, (uint64_t)H, (uint64_t)NB};
        uint64_t strides[3] = {(uint64_t)Cout * 2, (uint64_t)W * Cout * 2, (uint64_t)H * W * Cout * 2};
        uint32_t box[4] = {64, 8, 8, 1};
        if ((rc = make_tmap_bf16(&P.tmA, dy, 4, dims, strides, box, nullptr)) != AOZ_OK) return rc;
    }
    {
        uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)Win, (uint64_t)Hin, (uint64_t)NB};
        uint64_t strides[3] = {(uint64_t)Cin * 2, (uint64_t)Win * Cin * 2, (uint64_t)Hin * Win * Cin * 2};
        uint32_t box[4] = {64, (uint32_t)(8 * stride), (uint32_t)(8 * stride), 1};
        uint32_t es[4] = {1, (uint32_t)stride, (uint32_t)stride, 1};
        if ((rc = make_tmap_bf16(&P.tmB, x, 4, dims, strides, box, es)) != AOZ_OK) return rc;
    }
    if ((rc = launch_gemm(P, tp.pair, (cudaStream_t)stream)) != AOZ_OK) return rc;
    if (taps == 9)
        launch_k(wgrad_permute_reduce_kernel<9>, dim3(ceil_div(Cin, 128), Cout), dim3(128), (size_t)(0), (cudaStream_t)stream,
                 (const float*)workspace, splits, (long long)Cout, Cin, cin_real, (__nv_bfloat16*)grad_w, accumulate);
    else
        launch_k(wgrad_permute_reduce_kernel<1>, dim3(ceil_div(Cin, 128), Cout), dim3(128), (size_t)(0), (cudaStream_t)stream,
                 (const float*)workspace, splits, (long long)Cout, Cin, cin_real, (__nv_bfloat16*)grad_w, accumulate);
    AOZ_CHECK_LAUNCH("wgrad_permute_reduce_kernel");
    return AOZ_OK;
}

}  // extern "C"
