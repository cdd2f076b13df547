/* b200sr — C ABI of the B200-native (sm_100a) diffusion-denoiser kernels.
 *
 * This is the drop-in boundary of the hot path: plain pointers, sizes and a CUDA stream; no
 * torch types.  Every entry point
 *   - takes DEVICE pointers (bf16 activations are raw uint16 storage, "NHWC" = [N, H, W, C],
 *     token matrices are row-major [rows, ld]),
 *   - enqueues work on `stream` (a cudaStream_t passed as void*) and returns immediately,
 *   - never allocates, never synchronises, never throws,
 *   - returns 0 on success or a negative errno-style code:
 *       -22 (EINVAL)  bad shape / alignment / flag combination
 *       -19 (ENODEV)  no sm_100 device or driver entry point unavailable
 *        -5 (EIO)     CUDA launch error
 *
 * The reference (Bluear7878/Remote-Sensing-Vision-Language-Diffusion-Model) has no native code and
 * no FFI; the interface each function replaces is the torch op sequence at the cited
 * reference file:line.  The Python binding a maintainer would add is shown in INTEGRATION.md
 * (ctypes) and implemented in b200sr/_lib.py.
 */
#ifndef B200SR_H_
#define B200SR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Library / device introspection. */
#define B200SR_ABI_VERSION 6  /* what b200sr_abi_version() returns */
int b200sr_abi_version(void);         /* bumps on any signature change */
int b200sr_num_sms(void);             /* SM count of the current device, <0 on error */

/* Fused epilogue description shared by the GEMM and implicit-GEMM convolution entry points:
 *   out = alpha * (acc + bias[n]) + rowvec[group(m), n] + residual[m, n]          (geglu == 0)
 *   out[m, j] = (acc[m, v(j)] + bias[v(j)]) * gelu_erf(acc[m, g(j)] + bias[g(j)])  (geglu == 1)
 * where for GEGLU the weight rows were packed by interleaving value / gate rows in groups of 16
 * (rows 32k..32k+15 = value features 16k..16k+15, rows 32k+16..32k+31 = their gates), the output
 * has N/2 columns, and alpha / rowvec / residual are not allowed.
 * group(m) = m / rows_per_group (GEMM) or the image index (convolution).                      */
typedef struct b200sr_epilogue {
  const float* bias;        /* [N] fp32 or NULL */
  const float* rowvec;      /* [groups, N] fp32 or NULL (ResBlock emb add, openaimodel.py:337-348) */
  int32_t rows_per_group;   /* GEMM only; 0 = single group */
  int64_t ld_rowvec;        /* elements between rowvec rows; 0 = N (rowvec may be a column window of a wider matrix) */
  const void* residual;     /* bf16 [M, ldr] or NULL */
  int64_t ldr;
  void* out;                /* bf16 (or fp32 when out_fp32) [M, ldc] */
  int64_t ldc;
  int32_t out_fp32;
  int32_t geglu;
  float alpha;
  int32_t act;              /* applied to the final value: 0 = none, 1 = SiLU (ZeroSFT mlp_shared, SR_modules.py:75-78),
                               2 = GELU (erf; open_clip text tower MLP), 3 = quick GELU x*sigmoid(1.702x) (CLIP-L text tower) */
  /* Cross-attention against a context that is constant over the sampler steps (the text embedding,
   * attention.py:222-285), with to_q folded into the keys and to_out into the values:
   *   P = softmax_per_head(x K'^T)   one GEMM, N = heads * 80, epilogue = softmax over each 80-column
   *                                  segment of a row, of which the first softmax_valid (77) take part
   *                                  (the others are written as 0); exp2 is applied to the accumulator
   *                                  as is, i.e. K' carries scale * log2(e)
   *   out = P V' + bias + residual   a plain GEMM with K = heads * 80
   * K' / V' differ per batch element: rows [g * w_rows_per_group, (g + 1) * w_rows_per_group) of A are
   * multiplied with weight rows [g * w_group_stride, g * w_group_stride + N).                          */
  int32_t softmax_valid;       /* 0 = off; GEMM only, bf16 output, no other epilogue term */
  int32_t w_dynamic;           /* set when W is an activation written by an earlier kernel on the stream (e.g. K or V of
                                  an attention expressed as GEMMs): constant weights are otherwise prefetched before the
                                  kernel's programmatic dependency on its predecessor resolves */
  int32_t w_rows_per_group;    /* 0 = one weight for all rows; otherwise a multiple of 256 */
  int64_t w_group_stride;      /* in weight rows */
  /* b200sr_conv3x3_bf16, stride 1, W % 8 == 0, H >= 16 only: GroupNorm(+SiLU) of the INPUT fused into the convolution
   * (ResBlock in_layers / out_layers openaimodel.py:254-258, :289-300; first-stage ResnetBlock model.py:127-141; SR3 Block
   * unet.py:81-92): x is the raw tensor, a_gn_stats = (mean, rstd) per (image, group) from b200sr_group_norm_stats; every
   * staged input tile is rewritten as silu(x * rstd * w + (b - mean * rstd * w)) in shared memory before the MMAs read it
   * (zero padding stays zero), so the normalised tensor never travels through HBM.  NULL = off.                       */
  const float* a_gn_stats;     /* [N, groups, 2] fp32 */
  const float* a_gn_weight;    /* [Cin] */
  const float* a_gn_bias;      /* [Cin] */
  int32_t a_gn_groups;
  int32_t a_gn_silu;
  /* b200sr_gemm_bf16 only: the LayerNorm in front of a Linear (BasicTransformerBlock norm1/2/3 -> to_q/k/v, GEGLU proj,
   * attention.py:376-486) folded around the GEMM, so the normalised activations never exist in HBM and no LayerNorm
   * kernel runs.  With W' = W * gamma (rounded to bf16; this is the W passed in), colsum[n] = sum_k W'[n, k] and
   * shift[n] = sum_k W[n, k] * beta[k] (+ the Linear's bias):
   *     LN(x) W^T + b  =  rstd[m] * (x W'^T - mean[m] * colsum) + shift
   * The GEMM runs on the RAW rows x; (mean, rstd) of each row come from ln_parts partial (sum, sum of squares) pairs,
   * ln_stats[q * M + m], which the GEMM that produced x wrote through ln_stats_out (one pair per N tile of that
   * GEMM: ln_parts = ceil(N_producer / b200sr_gemm_n_tile(M, N_producer, K_producer)), taken over the bf16 values it
   * stored).  colsum / shift are [weight groups, N] (one row unless w_rows_per_group > 0).  Works with every epilogue
   * term, including geglu and the per-head softmax.  NULL = off.                                                  */
  const float* ln_stats;       /* [ln_parts, M, 2] fp32 */
  int32_t ln_parts;
  const float* ln_colsum;
  const float* ln_shift;
  float ln_eps;
  float* ln_stats_out;         /* [n tiles, M, 2] fp32 or NULL; bf16 output, no geglu / softmax */
  /* b200sr_gemm_bf16 only: softmax over WHOLE rows of alpha * A W^T in two passes of the same GEMM, for the single-head
   * attention of width 512 (SR3 SelfAttention, sr3_modules/unet.py:114-143; first-stage AttnBlock, model.py:158-199) whose
   * output accumulator leaves no tensor memory for a flash-style kernel.  The fp32 score matrix never exists:
   *   row_softmax = 1  statistics pass: no output matrix (out may be NULL); for every row and N tile the pair
   *                    (max, sum of 2^(x - max)) of x = alpha * acc over the tile's valid columns -> ln_stats_out
   *   row_softmax = 2  apply pass: the tile is recomputed and written as bf16 2^(x - M) / L, with (M, L) folded from the
   *                    ln_parts pairs in ln_stats (= pass 1's ln_stats_out)
   * alpha carries scale * log2(e); columns >= row_softmax_valid (0 = N) take no part and are written as 0.  No other
   * epilogue term may be set.                                                                                       */
  int32_t row_softmax;
  int32_t row_softmax_valid;
} b200sr_epilogue;

/* D = A[M,K] * W[N,K]^T with fused epilogue; bf16 operands, fp32 accumulate (tcgen05 / TMEM).
 * Replaces nn.Linear / 1x1 nn.Conv2d: sgm/modules/attention.py:213-218 (to_q/k/v, to_out),
 * :84-91 (GEGLU), :106 (FF out), :587/:611 (proj_in/out); openaimodel.py:283-287 (emb_layers),
 * :311 (skip 1x1), :657-691 (time_embed/label_emb); SR_modules.py:84 (zero_conv).
 * lda in elements; K % 8 == 0; N % 8 == 0; force_bn = 0 lets the library pick the N tile.    */
int b200sr_gemm_bf16(const void* A, int64_t lda, const void* W, int32_t M, int32_t N, int32_t K,
                     const b200sr_epilogue* epi, int32_t force_bn, void* stream);

/* The N tile b200sr_gemm_bf16 uses for an [M, K] x [N, K]^T product with force_bn = 0 and no softmax epilogue
 * (the number of ln_stats_out partials per row is ceil(N / tile)).  0 on invalid sizes.                          */
int b200sr_gemm_n_tile(int32_t M, int32_t N, int32_t K);

/* 3x3 convolution, pad 1, stride 1 or 2, NHWC bf16, weights [Cout, 3, 3, Cin] bf16, as an
 * implicit GEMM on the same tcgen05 mainloop (each tap = one shifted TMA box, zero fill = pad).
 * Replaces nn.Conv2d 3x3: openaimodel.py:121 (Upsample.conv), :190-197 (Downsample.op),
 * :257 / :294-300 (ResBlock), SR_modules.py:76-80 (ZeroSFT mlp_shared / zero_mul / zero_add),
 * sr3_modules/unet.py:59-92; the first-stage convolutions sgm/modules/diffusionmodules/model.py:53-143.
 * Cin % 64 == 0, Cout % 8 == 0.  pad_lo = 1: pad 1 on every side.  pad_lo = 0 (stride 2 only): pad 0 on top / left and
 * 1 on bottom / right — the first stage's Downsample, F.pad(x, (0, 1, 0, 1)) + conv(stride 2, padding 0),
 * model.py:70-88.                                                                                          */
int b200sr_conv3x3_bf16(const void* x, const void* w, int32_t N, int32_t H, int32_t W, int32_t Cin, int32_t Cout,
                        int32_t stride, int32_t pad_lo, const b200sr_epilogue* epi, int32_t force_bn, void* stream);

/* Direct 3x3 convolution (pad 1, stride 1) for tiny channel counts: Cin <= 8 (Cout % 8 == 0),
 * or Cout <= 4 (Cin % 8 == 0).  `addend` (bf16 NHWC, few-in only) is added to the result
 * (GLVControl `h += guided_hint`, SR_modules.py:521-531).  out_nchw_f32 (few-out only) writes
 * fp32 NCHW (UNet `out`, openaimodel.py:941-947; wrappers.py:110 `.float()`).                 */
int b200sr_conv3x3_small(const void* x, const void* w, const float* bias, const void* addend, void* y, int32_t N,
                         int32_t H, int32_t W, int32_t Cin, int32_t Cout, int32_t out_nchw_f32, void* stream);

/* GroupNorm over NHWC bf16 with optional fused SiLU and ZeroSFT modulation:
 *   y = GN(x) * w + b ; [SiLU] ; [y = y * (1 + gamma) + beta ; y = y*s + raw*(1-s)]
 * util.py:258-276, attention.py:122-125, openaimodel.py:254-258; SR_modules.py:101-110.
 * workspace: b200sr_group_norm_workspace_bytes() bytes of device scratch.  Its first 1 KiB holds
 * per-image arrival counters: zero it once after allocation; every call leaves it zeroed.
 * Calls that may run concurrently (different streams) need distinct workspaces.                */
size_t b200sr_group_norm_workspace_bytes(int32_t N, int32_t HW, int32_t C, int32_t groups);
/* kernels one b200sr_group_norm_nhwc call of this shape enqueues: 1 (tensors that fit the SMs' shared memory: statistics,
 * per-image barrier and apply in one kernel) or 2 (statistics kernel + apply kernel); 0 for invalid shapes. */
int b200sr_group_norm_launches(int32_t N, int32_t HW, int32_t C, int32_t groups);
int b200sr_group_norm_nhwc(const void* x, void* y, const float* weight, const float* bias, int32_t N, int32_t HW,
                           int32_t C, int32_t groups, float eps, int32_t silu, const void* sft_gamma,
                           const void* sft_beta, const void* raw, float control_scale, void* workspace, void* stream);

/* The statistics pass of b200sr_group_norm_nhwc alone: stats_out[n, g] = (mean, 1/sqrt(var + eps)), fp32 [N, groups, 2],
 * for a convolution that applies the normalisation itself (b200sr_epilogue.a_gn_*).  Same workspace contract.      */
int b200sr_group_norm_stats(const void* x, int32_t N, int32_t HW, int32_t C, int32_t groups, float eps, float* stats_out,
                            void* workspace, void* stream);

/* LayerNorm over the last dim of a bf16 [M, C] matrix (attention.py:437-439). */
int b200sr_layer_norm(const void* x, void* y, const float* weight, const float* bias, int32_t M, int32_t C, float eps,
                      void* stream);

/* softmax(Q K^T * scale) V for head_dim 64 (attention.py:222-285, SR_modules.py:135-149).
 * q/k/v are column windows of row-major bf16 matrices: head h of q lives at columns
 * [q_col + 64h, q_col + 64h + 64) of a [B, Nq, ldq] matrix (so a fused QKV projection is
 * consumed in place); out is [B, Nq, ldo] with head h at columns [64h, 64h + 64).
 * workspace: b200sr_attention_d64_workspace_bytes() bytes of device scratch (NULL allowed when that is
 * 0).  The tiles of the last, partial wave of CTAs are split over the key range and merged through
 * it; its first 2 KiB are arrival counters: zero them once after allocation, every call leaves them
 * zeroed.  Calls that may run concurrently (different streams) need distinct workspaces.
 * causal != 0 (Nq == Nk <= 128): key k takes part in query q only if k <= q — the text towers of the conditioner
 * (transformers CLIPTextModel / open_clip attn_mask, sgm/modules/encoders/modules.py:436-613).    */
size_t b200sr_attention_d64_workspace_bytes(int32_t B, int32_t H, int32_t Nq, int32_t Nk);
int b200sr_attention_d64(const void* q, int64_t ldq, int32_t q_col, const void* k, int64_t ldk, int32_t k_col,
                         const void* v, int64_t ldv, int32_t v_col, void* out, int64_t ldo, int32_t B, int32_t H,
                         int32_t Nq, int32_t Nk, float scale, int32_t causal, void* workspace, void* stream);

/* Between the two passes of a row_softmax GEMM: fold the [n_parts, rows, 2] (max, sum) pairs of pass 1 into one
 * (M, L) pair per row, out [rows, 2]; pass 2 then takes ln_stats = out, ln_parts = 1.                             */
int b200sr_row_softmax_fold(const float* parts, int32_t n_parts, int64_t rows, float* out, void* stream);

/* y = softmax(x * scale) over the first valid_cols entries of each row (the rest are written as 0: zero-
 * padded keys); x fp32 [rows, cols], y bf16.  SR3 SelfAttention (one head of width C, scores from
 * b200sr_gemm_bf16 with fp32 output): models/sr3_model/sr3_modules/unet.py:133-138. */
int b200sr_softmax_rows(const float* x, void* y, int32_t rows, int32_t cols, int32_t valid_cols, float scale,
                        void* stream);

/* Layout conversion at the nn.Module boundary. */
int b200sr_nchw_f32_to_nhwc_bf16(const float* x, void* y, int32_t N, int32_t C, int32_t HW, float scale, void* stream);
int b200sr_nhwc_bf16_to_nchw_f32(const void* x, float* y, int32_t N, int32_t C, int32_t HW, void* stream);
/* same, from a source with Cs >= C channels per pixel (the first C are converted): the result of a convolution to <= 4
 * channels that ran on the tensor cores with its output padded to 8 (UNet `out` openaimodel.py:941-947 + wrappers.py:110
 * `.float()`; SR3 final_conv; the first stage's decoder conv_out). */
int b200sr_nhwc_bf16_to_nchw_f32_strided(const void* x, float* y, int32_t N, int32_t C, int32_t Cs, int32_t HW, void* stream);

/* Nearest x2 upsample, NHWC bf16 (openaimodel.py:125-145; sr3 unet.py:59-66). */
int b200sr_upsample2x_nhwc(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);

/* out[:, :Ca] = a ; out[:, Ca:] = b (+ c).  Rows of bf16 channels (SR_modules.py:88-100,
 * openaimodel.py:1001, sr3 unet.py:257).  c may be NULL.                                      */
int b200sr_concat_add(const void* a, int32_t Ca, const void* b, int32_t Cb, const void* c, void* out, int64_t rows,
                      void* stream);

/* y = a + alpha * b, bf16. */
int b200sr_axpy_bf16(const void* a, const void* b, void* y, float alpha, int64_t n, void* stream);

/* y[rows, Cpad] = [x[rows, C] | zeros], bf16: pads the 4-channel latent to a 64-channel K chunk so the stem
 * convolutions (openaimodel.py:695-701, SR_modules.py:478-480) use b200sr_conv3x3_bf16. */
int b200sr_pad_channels(const void* x, void* y, int32_t C, int32_t Cpad, int64_t rows, void* stream);

/* y = silu(x), bf16 (embedding path: openaimodel.py:281-283, :660-662). */
int b200sr_silu_bf16(const void* x, void* y, int64_t n, void* stream);

/* out[b, t, :] = tok[ids[b, t], :] + pos[t, :] (fp32 tables, int64 ids, bf16 out): token + position embedding of
 * the conditioner's text towers (sgm/modules/encoders/modules.py:473-493, :569-571). */
int b200sr_embed_tokens(const int64_t* ids, const float* tok, const float* pos, void* out, int32_t B, int32_t T, int32_t C,
                        int32_t vocab, void* stream);

/* Sinusoidal embedding of t[B] (fp32) to bf16 [B, dim]; sin_first = 0: cos|sin (util.py:206-230),
 * sin_first = 1: sin|cos (sr3 unet.py:19-32).                                                 */
int b200sr_sinusoid_embedding(const float* t, void* out, int32_t B, int32_t dim, float max_period, int32_t sin_first,
                              void* stream);

/* Sampler step around the network call (sampling.py:598-621, denoiser.py:67-78, guiders.py:59-74).
 * scalars (device, fp32[6]) = {sigma, sigma_hat, sigma_next, sigma_quantised, cfg_scale, s_noise}.
 *   pre : x_hat = x + noise*s_noise*sqrt(sigma_hat^2 - sigma^2) (fp32 NCHW);
 *         net_in[k] = x_hat / sqrt(sigma_q^2 + 1) for k < cfg_copies (bf16 NHWC [cfg_copies*B,...])
 *   post: denoised = CFG(eps * -sigma_q + x_hat); x_next = x_hat + (x_hat - denoised)/sigma_hat *
 *         (sigma_next - sigma_hat); eps is fp32 NCHW [2B,...] (uncond first) when use_cfg.      */
int b200sr_sampler_pre(const float* x, const float* noise, const float* scalars, float* x_hat, void* net_in, int32_t B,
                       int32_t C, int32_t HW, int32_t cfg_copies, void* stream);
int b200sr_sampler_post(const float* eps, const float* x_hat, const float* scalars, float* denoised_out, float* x_next,
                        int32_t B, int32_t C, int32_t HW, int32_t use_cfg, void* stream);
int b200sr_euler_from_denoised(const float* denoised, const float* x_hat, const float* scalars, float* x_next,
                               int64_t n, void* stream);

/* Tile blend (sampling.py:753-756, :830-847): acc[win] += tile * weight, cnt[win] += weight; out = acc / cnt.
 * The product and the sum are rounded separately (no FMA), so a weighted strip formed by
 * b200sr_tile_weighted_strip on another GPU and added by b200sr_strip_add gives the same bits.  cnt may be
 * NULL (the weight sum is data independent and can be kept by the caller).                               */
int b200sr_tile_accumulate(const float* tile, const float* weight, float* acc, float* cnt, int32_t BC, int32_t th,
                           int32_t tw, int32_t H, int32_t W, int32_t h0, int32_t w0, void* stream);
int b200sr_tile_normalize(const float* acc, const float* cnt, float* out, int64_t n, void* stream);

/* Tile-sharded blend across GPUs (the reference loops over tiles sequentially, sampling.py:727-756): the
 * part of a window's weighted result that lies inside another rank's window travels as a packed strip.
 *   strip[bc, y, x] = tile[bc, y0 + y, x0 + x] * weight[y0 + y, x0 + x]       (sender)
 *   acc[bc, h0 + y, w0 + x] += strip[bc, y, x]                                (owner, in global window order) */
int b200sr_tile_weighted_strip(const float* tile, const float* weight, float* strip, int32_t BC, int32_t th, int32_t tw,
                               int32_t y0, int32_t x0, int32_t sh, int32_t sw, void* stream);
int b200sr_strip_add(const float* strip, float* acc, int32_t BC, int32_t sh, int32_t sw, int32_t H, int32_t W,
                     int32_t h0, int32_t w0, void* stream);

/* First-stage (SDXL VAE) glue at the latent (sgm/models/autoencoder.py:298-318, models/SR_model.py:58-85):
 *   pointwise_small: 1x1 convolution between <= 8 channels (quant_conv 8->8, post_quant_conv 4->4), bf16 NHWC in,
 *                    w fp32 [Cout, Cin], out = (w x + bias) * scale as bf16 NHWC or fp32 NCHW [rows / HW, Cout, HW]
 *   diag_gaussian:   DiagonalGaussianDistribution on moments fp32 NCHW [N, 2C, HW] (mean | logvar, logvar clamped to
 *                    [-30, 20]): z = (mean + exp(logvar / 2) * noise) * scale, or mean * scale when noise is NULL (mode) */
int b200sr_pointwise_small(const void* x, const float* w, const float* bias, void* y, int32_t Cin, int32_t Cout,
                           int64_t rows, int32_t HW, int32_t out_nchw_f32, float scale, void* stream);
int b200sr_diag_gaussian(const float* moments, const float* noise, float* z, int32_t N, int32_t C, int32_t HW,
                         float scale, void* stream);

/* Output side (utils/colorfix.py:73-119, models/util.py:159-166), fp32 NCHW images:
 *   wavelet_level: low = depthwise 3x3 [1 2 1; 2 4 2; 1 2 1] / 16 blur of img with dilation `radius` and replicate
 *                  padding; if high != NULL: high = (first ? 0 : high) + (img - low)   (one level of wavelet_decomposition)
 *   add_f32:       out = a + b                                   (content_high_freq + style_low_freq)
 *   image_to_u8:   bicubic resize (align_corners False, A = -0.75) of one [C, H, W] image in [-1, 1] to [OH, OW],
 *                  * 127.5 + 127.5, clip, truncate -> uint8 [OH, OW, C]                              (Tensor2PIL) */
int b200sr_wavelet_level(const float* img, float* low, float* high, int32_t first, int32_t BC, int32_t H, int32_t W,
                         int32_t radius, void* stream);
int b200sr_add_f32(const float* a, const float* b, float* out, int64_t n, void* stream);
int b200sr_image_to_u8(const float* x, void* out, int32_t C, int32_t H, int32_t W, int32_t OH, int32_t OW, void* stream);

/* Stage-1 -> stage-2 hand-off (infer.py:133-138 tensor2img; models/util.py:132-156 PIL2Tensor), uint8 images HWC:
 *   tensor2img_u8:    fp32 [C, H, W] -> uint8 [H, W, C]: t = (clamp(x, -1, 1) + 1) / 2 in fp32, rint(t * 255) in fp32
 *                     (round half to even, as numpy .round()); SR3's tensor2img, utils/tensor2img.py:4-21
 *   resample_u8:      one axis of PIL.Image.resize(..., Image.BICUBIC) (libImaging/Resample.c, 8 bits per channel):
 *                     src viewed as [outer, in_len, inner] bytes -> dst [outer, out_len, inner]; the horizontal pass
 *                     of an [H, W, C] image is (outer, inner) = (H, C), the vertical pass (1, W * C).  bounds int32
 *                     [out_len, 2] = (first tap, tap count), coeffs int32 [out_len, ksize] in 22-bit fixed point,
 *                     both built on the host (b200sr.ops.pillow_bicubic_tables); dst[o] = clamp((2^21 + sum of
 *                     src * coeff) >> 22, 0, 255).  src and dst must not overlap.
 *   img_u8_to_tensor: uint8 [H, W, C] -> fp32 [C, H, W]: (float)(x / 255.0 * 2.0 - 1.0) evaluated in double */
int b200sr_tensor2img_u8(const float* x, void* out, int32_t C, int32_t H, int32_t W, void* stream);
int b200sr_resample_u8(const void* src, void* dst, int32_t outer, int32_t in_len, int32_t out_len, int32_t inner,
                       const int32_t* bounds, const int32_t* coeffs, int32_t ksize, void* stream);
int b200sr_img_u8_to_tensor(const void* in, float* out, int32_t C, int32_t H, int32_t W, void* stream);

/* Up to 8 small device-to-device copies in one launch (bytes % 4 == 0, 4-byte aligned): the per-step loader of
 * the sampler engine (latent, noise, this step's row of the scalar table sampling.py:598-606 and of the
 * precomputed timestep-embedding projections openaimodel.py:281-287) into the buffers a CUDA graph reads. */
typedef struct b200sr_copy {
  const void* src;
  void* dst;
  int64_t bytes;
} b200sr_copy;
int b200sr_copy_batch(const b200sr_copy* copies, int32_t n, void* stream);

/* First-block-cache similarity (DFBCache.py:98-134): result[0] = mean|prev-cur| / (mean|prev| + 1e-6),
 * result[1] = (result[0] < threshold[0]).  workspace = 2 zeroed doubles (re-zeroed on return). */
int b200sr_rel_l1_similarity(const void* prev, const void* cur, int64_t n, const float* threshold, void* workspace,
                             float* result, void* stream);

/* SR3 ancestral update (sr3_modules/diffusion.py:142-176); scalars (device fp32[5]) =
 * {sqrt_recip_alphas_cumprod[t], sqrt_recipm1_alphas_cumprod[t], coef1[t], coef2[t], log_var[t]}. */
int b200sr_sr3_update(const float* x, const float* eps, const float* noise, const float* scalars, float* out,
                      int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200SR_H_ */
