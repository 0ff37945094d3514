/*
 * tair_b200 — C ABI of the B200-native TeReDiff patch-denoising hot path.
 *
 * This is the drop-in boundary: every entry point takes plain device pointers,
 * explicit sizes and a cudaStream_t (passed as void*), enqueues work on that
 * stream without synchronising, and returns 0 on success or a negative code
 * (the message is available from tair_last_error()).  Outputs are always
 * caller-allocated.  There is no CPU fallback: a missing / unloadable library
 * is a hard error on the Python side (tair_b200/_lib.py).
 *
 * Reference interfaces replaced (paths relative to the yinnhao/TAIR tree):
 *   - testr/adet/layers/csrc/vision.cpp:52-55, DeformAttn/ms_deform_attn.h:20-40
 *       `_C.ms_deform_attn_forward`                      -> tair_msda_forward
 *   - terediff/sampler/spaced_sampler.py:141-147,123-131,167-189 (p_sample math)
 *                                                        -> tair_sampler_update
 *   - DDIM / DPM-Solver++(2M) update (DiffBIR's samplers; not in TAIR)
 *                                                        -> tair_sampler_multistep_update
 *   - val_patches.py:114-206 (merge_patches_with_overlap) -> tair_blend_tiles
 *   - terediff/model/unet.py:203-223 / util.py:182-193 (GroupNorm32+SiLU)
 *                                                        -> tair_groupnorm_nhwc
 *   - terediff/model/attention.py:252-254 (nn.LayerNorm) -> tair_layernorm
 *   - nn.Linear / 1x1 nn.Conv2d call sites (attention.py:181-186,206,301-331;
 *     unet.py:170-176,189-197; controlnet.py:318-321)    -> tair_gemm_bf16
 *   - 3x3 nn.Conv2d call sites (unet.py:67,99,152,178; controlnet.py:168-175)
 *                                                        -> tair_conv3x3_bf16
 *   - F.scaled_dot_product_attention (attention.py:206)  -> tair_attention_bf16
 *
 * Layout convention: activations are channels-last bf16, i.e. a (B,C,H,W)
 * reference tensor is held as a row-major [B*H*W, C] matrix.  Weights are
 * repacked once at load time to [Cout, K] bf16 with K contiguous
 * (K = Cin for linear/1x1, K = 9*Cin ordered (ky,kx,ci) for 3x3).
 */
#ifndef TAIR_B200_H_
#define TAIR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TAIR_OK 0
#define TAIR_ERR_INVALID (-1)
#define TAIR_ERR_CUDA (-2)
#define TAIR_ERR_UNSUPPORTED (-3)

/* Thread-local message of the last failing call on this thread ("" if none). */
const char* tair_last_error(void);
/* ABI version of this header; bumped on any signature change. */
int tair_abi_version(void);
/* Number of kernel launches issued through this library by the calling process
 * since load (or since the last reset).  bench.py reports it as gpu_launches. */
int64_t tair_launch_count(void);
void tair_launch_count_reset(void);

/* ---- epilogue shared by the tensor-core GEMM and the implicit-GEMM conv ---- */
enum {
  TAIR_ACT_NONE = 0,
  TAIR_ACT_GEGLU = 1, /* out[:, j] = v[:, j] * gelu(g[:, j]); weight rows tile-interleaved, see DESIGN.md */
  TAIR_ACT_GELU = 2,
  TAIR_ACT_SILU = 3,
  TAIR_ACT_RELU = 4
};

typedef struct tair_epilogue {
  void* out;               /* [M, ldc] bf16 (or fp32 when out_fp32 != 0)              */
  int64_t ldc;             /* elements between consecutive output rows                 */
  int32_t out_fp32;        /* 0: bf16 output, 1: fp32 output                           */
  int32_t act;             /* TAIR_ACT_*; applied after bias / row-group add           */
  const float* bias;       /* [N] fp32 or NULL                                         */
  const void* residual;    /* [M, ldr] bf16 added after the activation, or NULL        */
  int64_t ldr;
  const void* rowgroup;    /* fp32 (bf16 when rowgroup_bf16 != 0) [G, ldg] added before act, or NULL.  rows_per_group > 0: row m uses
                              rowgroup[m / rows_per_group] (timestep-embedding add: one row per image);
                              rows_per_group < 0: periodic, row m uses rowgroup[m % -rows_per_group]
                              (positional-embedding projections shared by every image)     */
  int64_t ldg;
  int32_t rows_per_group;
  int32_t rowgroup_bf16;   /* 0: fp32 rows.  1: bf16 rows, prefetched like the residual (half the L2 traffic of the fp32
                              form; TESTR's per-query positional projections).  Needs a 16-byte aligned bf16 output,
                              N % 32 == 0, rows 16-byte aligned (ldg % 8 == 0), act == NONE, no residual, no folded
                              LayerNorm; TAIR_ERR_INVALID otherwise.  Not on the split-K path of
                              tair_conv3x3_bf16 either (see `workspace`): a conv whose output image is at most 8x8 with
                              K >= 4096, given a workspace, returns TAIR_ERR_INVALID for bf16 rows (fp32 rows work).  */
  void* workspace;         /* optional scratch (16-byte aligned, private to the stream) or NULL.  When given and large
                              enough (3 * M * N * 4 bytes), tair_conv3x3_bf16 computes layers whose OUTPUT image is at
                              most 8x8 with K >= 4096 as a 3-way split-K: fp32 partial tiles in the workspace, then
                              a fixed-order reduction + epilogue kernel.  The split depends on the layer geometry
                              only, never on the batch, so results stay batch-independent.                     */
  int64_t workspace_bytes;
  /* LayerNorm folded into the GEMM that consumes it (attention.py:252-254,264-272: norm1 -> attn1 q|k|v, norm2 -> attn2
     to_q, norm3 -> GEGLU): A holds the RAW rows x, W holds W * gamma, and with ln_row_stats != NULL the accumulator is
     rescaled per row BEFORE bias / activation:   acc' = rstd[m] * (acc - mean[m] * ln_col_sum[n])
     ln_row_stats: fp32 [M, 2] = (mean, rstd) from tair_row_stats; ln_col_sum: fp32 [N] = sum_k W'[n, k] (of the bf16 values);
     the caller folds beta into the bias: bias'[n] = bias[n] + sum_k beta[k] W[n, k].  GEMM only (not conv / split-K). */
  const float* ln_row_stats;
  const float* ln_col_sum;
} tair_epilogue;

/* out = epilogue(A[M,K] * W[N,K]^T).  A, W bf16, K contiguous; lda/ldw in elements
 * (multiples of 8).  fp32 accumulation in tensor memory (tcgen05).
 * Tile autotuning: the first un-captured call for a new problem shape times every legal N tile on the caller's stream and
 * synchronises that stream ONCE (results are bit-identical for every candidate); later calls, and calls made while the
 * stream is being captured, enqueue without synchronising.  TAIR_AUTOTUNE=0 disables tuning (closed-form tile pick). */
int tair_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, int32_t M, int32_t N,
                   int32_t K, const tair_epilogue* epi, void* stream);

/* 3x3 convolution, stride 1 or 2, as an implicit GEMM:
 *   x  [B, H, W, Cin] bf16 channels-last (Cin % 64 == 0)
 *   w  [Cout, 9*Cin]  bf16, K ordered (ky, kx, ci)
 *   pad = zeros on the top/left (0 or 1); one zero row/column is always available on the bottom/right.
 *         pad 1 == PyTorch padding=1; pad 0 == F.pad(x,(0,1,0,1)) + padding=0 (VAE downsampler).
 *   out rows are output pixels in (b, ho, wo) order; M = B*Ho*Wo, N = Cout. */
int tair_conv3x3_bf16(const void* x, const void* w, int32_t B, int32_t H, int32_t W, int32_t Cin,
                      int32_t Cout, int32_t stride, int32_t pad, const tair_epilogue* epi, void* stream);

/* softmax(Q K^T * scale) V per (batch, head); flash-style, head_dim must be 64.
 *   q [B*Lq, ldq], k/v [B*Lk, ldk/ldv], o [B*Lq, ldo]  bf16; head h occupies columns [64h, 64h+64)
 *   of each row (so q/k/v may be column slices of one fused projection buffer).  causal != 0 (Lq == Lk): query i
 *   sees keys j <= i only (the attn_mask of the OpenCLIP text transformer). */
int tair_attention_bf16(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                        void* o, int64_t ldo, int32_t B, int32_t H, int32_t Lq, int32_t Lk,
                        int32_t head_dim, float scale, int32_t causal, void* stream);

/* ---- memory-bound kernels ------------------------------------------------------------------ */

/* GroupNorm over channels-last bf16 x [B, HW, C] with optional fused SiLU / GELU (act = TAIR_ACT_*).
 * gamma/beta fp32 [C]; workspace >= tair_groupnorm_workspace_bytes(B, groups) bytes of device memory. */
int64_t tair_groupnorm_workspace_bytes(int32_t B, int32_t groups);
int tair_groupnorm_nhwc(const void* x, void* y, const float* gamma, const float* beta, int32_t B, int32_t HW,
                        int32_t C, int32_t groups, float eps, int32_t act, void* workspace, void* stream);

/* Per-row LayerNorm statistics: out[m] = (mean, 1/sqrt(var + eps)) of x[m, :C]; bf16 rows, fp32 [M,2] out.  Feeds
 * tair_epilogue.ln_row_stats of the GEMM that consumes the LayerNorm (the normalised tensor is never materialised). */
int tair_row_stats(const void* x, int64_t ldx, float* out, int32_t M, int32_t C, float eps, void* stream);

/* Row LayerNorm: y[m,:] = (x[m,:]-mean)/sqrt(var+eps)*gamma+beta; bf16 in/out, fp32 statistics. */
int tair_layernorm(const void* x, int64_t ldx, void* y, int64_t ldy, const float* gamma, const float* beta,
                   int32_t M, int32_t C, float eps, void* stream);

/* One ancestral-sampling update, all tensors fp32 [B, per_sample]:
 *   v      = v_uncond ? v_uncond + cfg_scale*(v_cond - v_uncond) : v_cond      (cfg_scale_dev, a 1-element DEVICE
 *            scalar, overrides cfg_scale when non-NULL: a captured CUDA graph then serves every guidance scale)
 *   x0     = A[t]*x - B[t]*v        v-parameterisation: A = sqrt_alphas_cumprod, B = sqrt_one_minus_alphas_cumprod;
 *                                   eps-parameterisation: pass A = sqrt_recip_alphas_cumprod, B = sqrt_recipm1_alphas_cumprod
 *                                   (spaced_sampler.py:133-147)
 *   x_prev = coef1[t]*x0 + coef2[t]*x + (t != 0) * sqrt(post_var[t]) * noise
 * t is the int64 [B] index into the respaced schedule tables (device pointers).  pred_x0 may be NULL. */
int tair_sampler_update(const float* x, const float* v_cond, const float* v_uncond, float cfg_scale,
                        const float* cfg_scale_dev, const float* noise, float* x_prev, float* pred_x0, const int64_t* t,
                        const float* sqrt_alphas_cumprod, const float* sqrt_one_minus_alphas_cumprod,
                        const float* posterior_mean_coef1, const float* posterior_mean_coef2,
                        const float* posterior_variance, int32_t B, int32_t per_sample, void* stream);

/* One multistep (DDIM / DPM-Solver++(2M)) update, all tensors fp32 [B, per_sample]:
 *   v      = v_uncond ? v_uncond + cfg_scale*(v_cond - v_uncond) : v_cond      (cfg_scale_dev as in tair_sampler_update)
 *   x0     = P[t]*x - Q[t]*v            (same order of operations as tair_sampler_update)
 *   x_next = ((b[t]*x0 + a[t]*x) + c[t]*x0_hist) + d[t]*noise
 *   x0_hist <- x0                        (in place; x0_hist may be NULL only where every c[t] used is 0)
 * x0_hist is not read for a sample whose c[t] == 0, so stale or NaN history never reaches the result.  x_next must not
 * alias x, v_cond, v_uncond or x0_hist.  t is the int64 [B] index into the per-step tables (device pointers). */
int tair_sampler_multistep_update(const float* x, const float* v_cond, const float* v_uncond, float cfg_scale,
                                  const float* cfg_scale_dev, const float* noise, float* x_next, float* x0_hist,
                                  const int64_t* t, const float* P, const float* Q, const float* a, const float* b,
                                  const float* c, const float* d, int32_t B, int32_t per_sample, void* stream);

/* out[b, :] = cos(t*f) || sin(t*f), f_k = exp(-ln(max_period) k/half); t int64 [B]; out bf16 [B, dim]. */
int tair_timestep_embedding(const int64_t* t, void* out, int32_t B, int32_t dim, float max_period, void* stream);

/* (B,C,HW) fp32 -> [B*HW, Cpad] bf16 (zero channel padding) and back ([B*HW, ld] bf16 -> (B,C,HW) fp32). */
int tair_nchw_to_nhwc_bf16(const float* in, void* out, int32_t B, int32_t C, int32_t HW, int32_t Cpad, void* stream);
int tair_nhwc_to_nchw_f32(const void* in, int64_t ld, float* out, int32_t B, int32_t C, int32_t HW, void* stream);

/* out[M, C1+C2] = [a | b (+ c)] (c may be NULL); out = a + b over n elements; nearest x2 upsample. All bf16. */
int tair_concat_add(const void* a, const void* b, const void* c, void* out, int64_t M, int32_t C1, int32_t C2,
                    void* stream);
int tair_add_bf16(const void* a, const void* b, void* out, int64_t n, void* stream);
int tair_upsample2x_nhwc(const void* in, void* out, int32_t B, int32_t H, int32_t W, int32_t C, void* stream);

/* Multi-scale deformable attention forward; argument meaning as _C.ms_deform_attn_forward:
 *   value [B,S,M,D] (fp32, or bf16 when value_bf16), spatial_shapes int64 [L,2] (H,W) and
 *   level_start_index int64 [L] on the DEVICE, sampling_loc fp32 [B,Lq,M,L,P,2] (x,y in [0,1]),
 *   attn_weight fp32 [B,Lq,M,L,P]  ->  out [B,Lq,M*D] (fp32, or bf16 when out_bf16).
 * Unlike the reference there is no im2col_step and no batch-divisibility constraint. */
int tair_msda_forward(const void* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                      const float* sampling_loc, const float* attn_weight, void* out, int32_t B, int32_t S,
                      int32_t M, int32_t D, int32_t L, int32_t Lq, int32_t P, int32_t value_bf16,
                      int32_t out_bf16, void* stream);

/* Window attention of the Swin blocks (terediff/model/swinir.py:120-149): n_windows back-to-back sequences of L <= 64
 * tokens, H heads in 64-column slots (narrower heads zero-padded), packed 128/L per tensor-core tile and attended
 * block-diagonally.  bias (or NULL): fp32 [bias_nw, H, L (key), L (query)], added to q.k BEFORE the scale, i.e. the
 * caller stores (relative_position_bias + shift mask) / scale; window w uses table w % bias_nw. */
int tair_attention_windows_bf16(const void* q, const void* k, const void* v, int64_t ld, void* o, int64_t ldo,
                                int32_t H, int32_t L, int64_t n_windows, const float* bias, int32_t bias_nw,
                                float scale, void* stream);

/* LayerNorm over the first C_valid channels of rows padded to C (C % 8 == 0, C <= 256); pad channels are written as 0.
 * SwinIR keeps its 180 channels in 192-wide rows (swinir.py norm1 / norm2 / patch_embed.norm / norm). */
int tair_layernorm_ragged(const void* x, int64_t ldx, void* y, int64_t ldy, const float* gamma, const float* beta,
                          int32_t M, int32_t C, int32_t C_valid, float eps, void* stream);

/* y[r, :cols] = x[idx[r], :cols] (bf16 rows, cols % 8 == 0): window partition / reverse and cyclic shift of the Swin
 * blocks as a single index map (swinir.py:37-66,262-281). */
int tair_gather_rows_bf16(const void* x, int64_t ldx, const int32_t* idx, void* y, int64_t ldy, int64_t rows,
                          int32_t cols, void* stream);

/* y = x >= 0 ? x : slope * x on n bf16 values (n % 8 == 0): nn.LeakyReLU of the SwinIR upsampler (swinir.py:777-801). */
int tair_leaky_relu_bf16(const void* x, void* y, int64_t n, float slope, void* stream);

/* Tile front-end: crop P tiles of `tile` x `tile` pixels (origins[p] = {y, x}, device int32) out of the zero-padded
 * 8-bit RGB image [Hp, Wp, 3] and resize each to out x out exactly as PIL's Image.resize(BICUBIC) does (two passes,
 * 22-bit fixed point, 8-bit intermediate), then divide by 255: dst [P, 3, out, out] fp32.  bounds [out, 2] =
 * {first tap, taps} and coeffs [out, ksize] int32 are PIL's per-output-index tables (same for both passes of a square
 * tile; tair_b200.tiles.pil_bicubic_coeffs).  tmp: P * tile * out * 3 bytes.  Replaces the per-tile
 * T.Resize(BICUBIC) + T.ToTensor() of val_patches.py:291-294,318. */
int tair_tiles_bicubic_u8(const void* image, int32_t Hp, int32_t Wp, const int32_t* origins, int32_t P, int32_t tile,
                          int32_t out, const int32_t* bounds, const int32_t* coeffs, int32_t ksize, void* tmp,
                          float* dst, void* stream);

/* Blend n_tiles fp32 tiles [n_tiles, C, tile, tile] laid out row-major on an n_h x n_w grid with the given
 * overlap (stride = tile - overlap) into out [C, out_h, out_w] (top-left crop of the canvas). */
int tair_blend_tiles(const float* tiles, float* out, int32_t n_tiles, int32_t n_h, int32_t n_w, int32_t C,
                     int32_t tile, int32_t overlap, int32_t out_h, int32_t out_w, void* stream);

/* MSDeformAttn core fused with its pre-processing (ms_deform_attn.py:136-149): proj rows hold the raw
 * sampling_offsets (M*L*P*2) followed by the raw attention logits (M*L*P) of one query; the kernel applies the
 * softmax over L*P and forms loc = ref + offset/(W,H) (ref_dim 2) or ref_xy + offset/P * ref_wh * 0.5 (ref_dim 4).
 * ref is fp32 [(B,) Lq/q_per_ref, L, ref_dim]; ref_batch_stride (elements) is 0 when shared by all images.
 * proj is fp32, or bf16 when proj_bf16 != 0.  value bf16 [B,S,M,D] -> out bf16 [B*Lq, M*D]. */
int tair_msda_fused(const void* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                    const void* proj, int64_t ldp, int32_t proj_bf16, const float* ref, int32_t ref_dim,
                    int64_t ref_batch_stride, int32_t q_per_ref, void* out, int32_t B, int32_t S, int32_t M,
                    int32_t D, int32_t L, int32_t Lq, int32_t P, void* stream);

/* Self-attention over many short strided sequences (head slots of 64 columns; narrower heads are zero-padded by the
 * caller): q/k/v are column offsets into one row-major [rows, ld] bf16 matrix (fused in_proj output); sequence (o, i),
 * o < n_outer, i < n_inner starts at row o*outer_stride + i*inner_stride, token t at + t*tok_stride.  Output rows
 * follow the same addressing in o [rows, ldo].  Replaces the nn.MultiheadAttention cores of the TESTR decoder
 * (deformable_transformer.py:454-466,485-503) without the swapdims copies. */
int tair_attention_seq_bf16(const void* q, const void* k, const void* v, int64_t ld, void* o, int64_t ldo, int32_t H,
                            int32_t L, int64_t n_outer, int32_t n_inner, int64_t outer_stride, int64_t inner_stride,
                            int64_t tok_stride, float scale, void* stream);

/* The same, for 32-wide heads and sequences of at most 128 tokens, on UNPADDED projections (head h in columns
 * [32h, 32h + 32) of q / k / v / o; ld >= 32 H).  This is what the TESTR decoder calls: 16 control points / 25 characters
 * per object, 100 objects per tile, 8 heads of 32 channels - far below one 128-row tensor-core tile, so the kernel is
 * register-level mma.sync per (sequence, head) and bound by the bytes it reads (csrc/attn_small.cu). */
int tair_attention_seq32_bf16(const void* q, const void* k, const void* v, int64_t ld, void* o, int64_t ldo, int32_t H,
                              int32_t L, int64_t n_outer, int32_t n_inner, int64_t outer_stride, int64_t inner_stride,
                              int64_t tok_stride, float scale, void* stream);

/* Detection post-processing of the TESTR head (transformer_detector.py:123-152 + spaced_sampler.py:298-306) for n_items =
 * tiles x queries: scores[i] = sigmoid(mean_p pred_logits[i,p]) (one class), polygons[i, 2p+{0,1}] = ctrl point p in pixels
 * (x * image_w, y * image_h), recs[i,c] = arg-max character of position c (uint8).  pred_logits fp32 [n_items, n_pts],
 * pred_ctrl_points fp32 [n_items, n_pts, 2], pred_texts fp32 [n_items, n_chars, voc].  The score threshold is applied by
 * the caller after ONE device->host copy of the three compact outputs. */
int tair_testr_postprocess(const float* pred_logits, const float* pred_ctrl_points, const float* pred_texts,
                           float* scores, float* polygons, uint8_t* recs, int32_t n_items, int32_t n_pts,
                           int32_t n_chars, int32_t voc, float image_w, float image_h, void* stream);

/* y[r,:] = softmax(scale * x[r,:]) over bf16 rows (cols % 8 == 0, <= 8192); bf16 [R,C] -> [C,R] batched transpose.
 * Used by the single-head 512-wide VAE attention (terediff/model/vae.py:253-281), evaluated as GEMM-softmax-GEMM. */
int tair_softmax_rows_bf16(const void* x, int64_t ldx, void* y, int64_t ldy, int32_t rows, int32_t cols, float scale,
                           void* stream);
int tair_transpose_bf16(const void* in, int64_t ldi, int64_t in_batch_stride, void* out, int64_t ldo,
                        int64_t out_batch_stride, int32_t batch, int32_t R, int32_t C, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TAIR_B200_H_ */
