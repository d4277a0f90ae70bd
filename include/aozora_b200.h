/* aozora_b200.h -- C ABI of libaozora_b200.so: the B200-native SDXL UNet training-step kernels.
 *
 * The reference (Hysocs/Aozora_SDXL_Training) is pure Python and has no FFI; its hot path reaches the GPU only
 * through library calls made by diffusers / PyTorch.  Each entry point below replaces one such call site
 * (cited as reference file:line; "[3P]" = inside diffusers' UNet2DConditionModel, reached from train.py:2760).
 *
 * Conventions: every function returns 0 on success or a negative code (see AOZ_ERR_*), with the message
 * available from aoz_last_error() (thread-local).  Pointers are raw DEVICE pointers unless stated; the caller
 * owns every buffer including workspaces; no hidden allocation, no hidden synchronisation; `stream` is a
 * cudaStream_t passed as void*.  bf16 tensors are channels-last ("NHWC" / [rows, C]) unless stated.
 * Dtype codes: 0 = fp32, 1 = bf16, 2 = fp16.
 */
#ifndef AOZORA_B200_H
#define AOZORA_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define AOZ_OK 0
#define AOZ_ERR_ARG -1
#define AOZ_ERR_CUDA -2
#define AOZ_ERR_UNSUPPORTED -3

/* ---- plumbing ------------------------------------------------------------------------------------------- */
const char* aoz_last_error(void);
int aoz_abi_version(void);
int aoz_sm_count(void);
int aoz_set_pdl(int on);               /* programmatic dependent launch between consecutive kernels (default off: no gain under graph replay) */
long long aoz_launch_count(void);      /* kernels launched by this library so far (every launch site counts itself) */

/* ---- optimizer: RavenAdamW.step / TitanAdamW.step (training_utils/optimizers/raven.py:89-149,
 *      titan.py:237-296) and torch.nn.utils.clip_grad_norm_ (train.py:2772-2781) ----------------------------
 * Multi-tensor tables (device arrays): p/g/m/v_ptrs[n] = uint64 device addresses, numel[n] int64,
 * chunk_start[n+1] int32 (first chunk of tensor t), chunk_tensor[n_chunks] int32, chunk = aoz_mt_chunk_elems()
 * elements.  hyper[n] = 8 floats {beta1, 1-beta1, beta2, 1-beta2, eps, step_size, 1/sqrt_bc2, wd_factor}.
 * clip_coef: optional device float (multiplied into the gradient with torch's dtype rounding). */
int aoz_mt_chunk_elems(void);
int aoz_raven_step_mt(int n_tensors, int n_chunks, const void* p_ptrs, const void* g_ptrs, const void* m_ptrs,
                      const void* v_ptrs, const void* numel, const void* chunk_start, const void* chunk_tensor,
                      const void* hyper, const void* clip_coef, int p_dtype, int g_dtype, int m_dtype, void* stream);
/* out3 = {total_norm, clip_coef = min(1, max_norm/(norm+1e-6)), sum_of_squares}; partial: n_chunks floats */
int aoz_gradnorm_mt(int n_tensors, int n_chunks, const void* g_ptrs, const void* numel, const void* chunk_start,
                    const void* chunk_tensor, void* partial, float max_norm, int emulate_bf16, void* out3,
                    int g_dtype, void* stream);
int aoz_clip_coef_from_sumsq(const void* sumsq, float max_norm, int emulate_bf16, void* out2, void* stream);
/* Gradient accumulation (train.py:2765 with GRADIENT_ACCUMULATION_STEPS > 1: torch adds each micro-step's bf16 gradient into
 * p.grad): y[t] = copy ? b[t] : a[t] + b[t] for every tensor t, bf16, one launch over the multi-tensor tables above.  Each
 * element is bit-identical to aoz_add on the same pair (fp32 add, one round to nearest even).  y may alias a or b.  a_ptrs may
 * be null when copy != 0.  Tensors need only bf16 alignment: chunks whose pointers are all 16-byte aligned are vectorised.
 * The tables must be aligned to their element size; n_tensors must be positive. */
int aoz_grad_accum_mt(int n_tensors, int n_chunks, const void* a_ptrs, const void* b_ptrs, const void* y_ptrs,
                      const void* numel, const void* chunk_start, const void* chunk_tensor, int copy, void* stream);

/* ---- dense contractions [3P]: nn.Linear (to_q/k/v, to_out.0, proj_in/out, ff.net.0.proj + GEGLU, ff.net.2,
 *      time/add embedding MLPs) forward, dgrad, wgrad; nn.Conv2d 3x3/1x1 as implicit GEMM -------------------- */
int aoz_gemm_set_pair_mode(int mode);
/* SMs the persistent GEMM / conv launches may occupy (0 = all, rounded down to even): data-parallel runs leave NCCL's CTAs their own
 * SMs (set NCCL_MAX_CTAS to the difference) so that no persistent CTA waits behind a collective kernel.  Nothing is cached: every
 * GEMM / conv call plans its tiles (CTA pairs, tail split, wide plan) for the budget in force at that call, while launches already
 * captured into a CUDA graph keep the plan they were captured with. */
int aoz_gemm_set_sm_budget(int sms);
int aoz_gemm_force_bn(int bn);
/* tail split: tiles of the last, partly filled wave are cut along K across the idle SMs (fp32 slices in the caller-owned
 * scratch, finished by a fix-up kernel).  mode 0 = off, 1 = cost model decides (default), 2 = whenever possible.
 * The scratch (>= 20 MB covers every shape) is used stream-ordered: all GEMM / conv calls must share one stream. */
int aoz_gemm_set_tail_mode(int mode);
/* wide one-wave plan: outputs that are slightly more than one wave of 256 x 256 pair tiles (4096 x 1280 = 80 tiles on 74 SM pairs)
 * run as ONE round of 256 x 320 tiles (a single 320-column accumulator, two MMAs per K step).  mode 0 = off, 1 = cost model
 * decides (default), 2 = whenever the shape allows it (N % 320 == 0, tiles <= SM pairs, store epilogue, no split-K).
 * The second MMA has N = 64: for MN-major B it reads half a 64-wide swizzle atom per CTA. */
int aoz_gemm_set_wide_mode(int mode);
/* rounds of 320-wide tiles per SM pair the planner may consider (default 2; the single accumulator serialises a pair's tiles) */
int aoz_gemm_set_wide_max_rounds(int rounds);
int aoz_gemm_set_scratch(void* ptr, long long bytes);
int aoz_gemm_debug_flags(int flags);
int aoz_gemm_auto_splits(int M, int N, int K, int b_mn);
long long aoz_gemm_describe_plan(int M, int N, int K, int b_mn, int splits);   /* planner introspection for tools / tests */
int aoz_conv_wgrad_auto_splits(int NB, int H, int W, int Cout, int Cin, int ks);
int aoz_gemm_bf16(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn, void* C, long long ldc,
                  int M, int N, int K, const void* bias, const void* rowgroup_bias, int rows_per_group, long long ld_rgb,
                  const void* residual, long long ldr, int epi, void* aux, long long ld_aux, int accumulate, int splits,
                  void* workspace, void* stream);
/* Grouped GEMM (one persistent launch for up to 10 problems sharing K, operand majors and tile shape; plain bf16 store):
 * the weight gradients dW = dy^T x of one BasicTransformerBlock [3P].  A_ptrs/B_ptrs/C_ptrs: HOST arrays of n device
 * pointers (uint64); lda/ldb/ldc: HOST int64[n]; M/N: HOST int32[n]. */
int aoz_gemm_grouped_bf16(int n, const void* A_ptrs, const void* lda, const void* B_ptrs, const void* ldb, const void* C_ptrs,
                          const void* ldc, const void* M, const void* N, int K, int a_mn, int b_mn, void* stream);
int aoz_conv_fwd_bf16(const void* x, int NB, int Hin, int Win, int Cin, const void* wpack, int Cout, int ks, int stride,
                      int pad, int flip, void* y, const void* bias, const void* rowgroup_bias, const void* residual,
                      int accumulate, void* stream);
int aoz_conv_wgrad_bf16(const void* dy, const void* x, int NB, int H, int W, int Cout, int Hin, int Win, int Cin, int ks,
                        int stride, int pad, int cin_real, void* grad_w, int accumulate, int splits, void* workspace, void* stream);
int aoz_pack_conv_weight(const void* w, int Cout, int Cin, int ks, int CinPad, int CoutPad, void* wf, void* wd, void* stream);

/* ---- attention [3P]: Attention.attn1 / attn2 via AttnProcessor2_0 = F.scaled_dot_product_attention
 *      (train.py:213-229), head_dim 64, no mask, no dropout; forward and backward ---------------------------
 * q: [B, Tq, H, 64] with row stride ldq (elements), k/v: [B, Tk, H, 64] strides ldk / ldv; o: [B, Tq, H, 64] ldo;
 * lse: [B, H, Tq] fp32 (log-sum-exp of the scaled scores, natural log). */
int aoz_attn_fwd(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv, void* o, long long ldo,
                 void* lse, int B, int H, int Tq, int Tk, float scale, void* stream);
/* backward form: 2 = one kernel, dQ (and with a single KV tile dK / dV) summed over CTAs in fp32 by bulk reduce-add (default;
 * not bit-reproducible), 0 = dK/dV kernel + dQ kernel (bit-reproducible; also taken under 2 when Tq % 4 != 0).  Any other
 * value returns AOZ_ERR_ARG and leaves the form unchanged. */
int aoz_attn_set_bwd_mode(int fused);
long long aoz_attn_bwd_workspace_floats(int B, int H, int Tq);
int aoz_attn_bwd(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv, const void* o,
                 long long ldo, const void* d_o, long long lddo, const void* lse, void* dq, long long lddq, void* dk,
                 long long lddk, void* dv, long long lddv, int B, int H, int Tq, int Tk, float scale, void* workspace,
                 void* stream);

/* ---- normalisation [3P]: GroupNorm(32)(+SiLU) in ResnetBlock2D / Transformer2DModel.norm / conv_norm_out,
 *      LayerNorm in BasicTransformerBlock ------------------------------------------------------------------- */
/* experiment switch: 1 = single-launch slab kernels where a (image, group) slab fits in shared memory (default), 0 = always
 * the statistics + apply kernels */
int aoz_groupnorm_set_slab(int on);
long long aoz_groupnorm_workspace_floats(int NB, int HW, int C);
int aoz_groupnorm_fwd(const void* x, const void* gamma, const void* beta, int NB, int HW, int C, float eps, int silu,
                      void* y, void* mean, void* rstd, void* workspace, void* stream);
int aoz_groupnorm_bwd(const void* dy, const void* x, const void* gamma, const void* beta, const void* mean, const void* rstd,
                      int NB, int HW, int C, int silu, const void* dres, void* dx, void* dgamma, void* dbeta, int accumulate,
                      void* workspace, void* stream);
int aoz_layernorm_fwd(const void* x, const void* gamma, const void* beta, long long rows, int C, float eps, void* y, void* mean,
                      void* rstd, void* stream);
long long aoz_layernorm_bwd_workspace_floats(int C);
int aoz_layernorm_bwd(const void* dy, const void* x, const void* gamma, const void* mean, const void* rstd, long long rows, int C,
                      const void* dres, void* dx, void* dgamma, void* dbeta, int accumulate, void* workspace, void* stream);
/* The same, additionally dcolsum[c] = sum_r dx[r, c] (of the stored bf16 dx; null: not wanted): dx of a pre-LN transformer sublayer
 * is the gradient of the previous Linear's output, so this is that layer's bias gradient without the column-sum launch */
int aoz_layernorm_bwd_colsum(const void* dy, const void* x, const void* gamma, const void* mean, const void* rstd, long long rows, int C,
                             const void* dres, void* dx, void* dgamma, void* dbeta, int accumulate, void* dcolsum, void* workspace,
                             void* stream);

/* ---- step glue: noising + target (train.py:2743-2758; DDPMScheduler.add_noise/get_velocity [3P]),
 *      weighted_sdxl_mse_loss + dL/dpred (train.py:2408-2416, 2765), layout and elementwise pieces [3P] ------- */
int aoz_nchw_to_nhwc(const void* src, int src_f32, int NB, int C, int HW, int Cpad, void* dst, void* stream);
int aoz_nhwc_to_nchw(const void* src, int NB, int C, int HW, int ld, void* dst, int dst_f32, void* stream);
int aoz_noise_target(const void* latents, const void* noise, const void* tickets, const void* alphas_cumprod, const void* jitter,
                     int mode, int NB, int C, int HW, int Cpad, void* xt, void* target, void* cond, void* stream);
int aoz_mse_loss(const void* pred, long long p_sn, long long p_sc, long long p_shw, const void* target, const void* tickets,
                 const void* table, int table_len, int NB, int C, int HW, float denom, const void* grad_scale_ptr, float grad_scale,
                 void* per_sample, void* weights, void* loss_out, void* dpred, long long d_sn, long long d_sc, long long d_shw,
                 void* stream);
int aoz_geglu_bwd(const void* dy, const void* aux, long long M, int half, void* daux, void* stream);
int aoz_silu_fwd(const void* x, long long n, void* y, void* stream);
int aoz_silu_bwd(const void* dy, const void* x, long long n, void* dx, void* stream);
int aoz_add(const void* a, const void* b, long long n, void* y, void* stream);
int aoz_upsample2x_fwd(const void* x, int NB, int H, int W, int C, void* y, void* stream);
int aoz_upsample2x_bwd(const void* dy, int NB, int H, int W, int C, void* dx, void* stream);
int aoz_zero_insert2x(const void* x, int NB, int H, int W, int C, int Hout, int Wout, void* y, void* stream);
int aoz_copy_channels(const void* src, long long src_ld, int src_off, void* dst, long long dst_ld, int dst_off, long long rows, int ch,
                      int accumulate, void* stream);
long long aoz_colsum_workspace_floats(int groups, int N);
int aoz_colsum(const void* x, int groups, long long M, int N, long long ld, long long group_stride, void* out, int accumulate,
               void* workspace, void* stream);
int aoz_timestep_embedding(const void* t, int n, int dim, void* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AOZORA_B200_H */
