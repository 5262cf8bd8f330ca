/* tld_b200.h — C ABI of libtld_b200.so, the B200-native (sm_100a) hot path of
 * apapiu/transformer_latent_diffusion.
 *
 * The reference is pure Python and has NO FFI boundary of its own (SURVEY.md §8b); its boundary is the
 * Python class API.  Each entry point below therefore names the reference method whose body it replaces
 * (paths relative to /root/reference).  The Python mirror of that API lives in
 * transformer_latent_diffusion_b200/{denoiser,diffusion}.py and binds these symbols with ctypes
 * (see INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - plain pointers and sizes only; every data pointer is a DEVICE pointer unless stated otherwise
 *   - all tensors are contiguous, row-major, fp32 at the boundary (the reference's default dtype);
 *     bf16 exists only inside the library as the tensor-core operand format (fp32 accumulate)
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); calls on one handle are not re-entrant
 *   - return 0 on success; non-zero on error, message via tld_last_error() (thread-local)
 *   - there is no CPU fallback: without a CUDA device every compute entry point returns an error
 */
#ifndef TLD_B200_H
#define TLD_B200_H

#include <stdint.h>

#if defined(__GNUC__)
#define TLD_API __attribute__((visibility("default")))
#else
#define TLD_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tld_denoiser tld_denoiser; /* opaque */

/* Constructor arguments of tld.denoiser.Denoiser (tld/denoiser.py:86-97).  dropout is accepted for
 * signature parity and must be 0 for the inference path (the reference evaluates with model.eval()). */
typedef struct tld_config {
  int32_t image_size;       /* latent H = W                         */
  int32_t noise_embed_dims; /* sinusoidal embedding width E         */
  int32_t patch_size;
  int32_t embed_dim;        /* D, multiple of 64, heads = D/64      */
  int32_t n_layers;
  int32_t text_emb_size;
  int32_t mlp_multiplier;
  int32_t n_channels;
  float dropout;
} tld_config;

TLD_API const char* tld_last_error(void);
TLD_API int tld_version(void);
/* Process-wide tuning switches (tests / experiments): "gemm_ctas" = 0 auto | 1 single-CTA tiles | 2 CTA-pair
 * (cta_group::2) tiles;  "attention_impl" = 0 auto | 1 mma.sync kernel | 3 tcgen05 persistent;
 * "attention_exp_emu" = 0|4|6|8|10 of every 16 exp2 pairs of kernel 3 evaluated on the FMA pipe instead of MUFU;  "attention_bwd_impl" = 0 | 1 mma.sync backward kernels (default, faster) | 2 tcgen05 backward kernel when tokens per
 * sample % 256 == 0;
 * "fused_mlp" = 1 (default) up-projection + depthwise conv + GELU as one
 * kernel for 16x16 token grids | 0 three separate kernels;  "ln_fold" = 1 norm1 / norm3 folded into the neighbouring GEMMs (their
 * statistics ride on the residual epilogues; measured slower on B200, see csrc/api.cu) | 0 (default) separate LayerNorm kernels;  "pdl" = 1 launch
 * the step kernels with programmatic dependent launch (prologues overlap the previous kernel's tail) | 0 plain launches (default: measured no gain);
 * "fused_qkv" = 1 (default) qkv projection + self-attention + residual as one CTA-pair kernel at 256 tokens per sample | 0 GEMM + attention kernel;
 * "qkv_exp_emu" = 0|4|6|8 the same exp2 split for that kernel;  "fused_xattn" = 1 (default) norm2 + 2-token cross-attention (q folded into the keys)
 * + residual + norm3 as one row-wise kernel (embed_dim % 128 == 0) | 0 LayerNorm, q GEMM with the 2-key epilogue, LayerNorm;
 * variants of that row kernel, all measured within 10 % of each other (DESIGN.md 3.4b): "xattn_rows" = 4 (default) | 2 rows per warp
 * (8 | 16 warps), "xattn_ctas" = 1 (default) | 2 CTAs per SM, "xattn_mma" = 0 (default) FFMA dot products | 1 | 2 | 3 the dots as
 * tf32 mma.sync with x truncated | x split hi + lo | x and the folded keys split (embed_dim <= 768, tokens % 8 == 0);
 * "share_cfg_prefix" = 1 (default) the sampler runs block 0's norm1 + self-attention once per CFG pair and copies the rows (bit-identical) | 0. */
TLD_API int tld_set_option(const char* key, int value);

/* ---- lifetime --------------------------------------------------------------------------------
 * Replaces Denoiser.__init__ + .to(device) (tld/denoiser.py:86-114, tld/diffusion.py:145-155). */
TLD_API int tld_denoiser_create(const tld_config* cfg, int device, tld_denoiser** out);
TLD_API void tld_denoiser_destroy(tld_denoiser* h);

/* Replaces load_state_dict for ONE entry (tld/diffusion.py:152-153).  `key` is the reference state_dict key
 * (e.g. "denoiser_trans_block.decoder_blocks.0.mlp.mlp.1.weight"); `data` is fp32 (host or device pointer,
 * `numel` elements).  The library copies/packs into its own arena (bf16 for GEMM operands, fp32 otherwise). */
TLD_API int tld_denoiser_set_param(tld_denoiser* h, const char* key, const float* data, int64_t numel);
/* The same for n parameters at once from DEVICE-resident fp32 tensors, enqueued on `stream` without any host
 * synchronisation (copies / conversion kernels straight from the sources).  The Python mirror calls it before every forward,
 * generate and training step: in-place updates by optimisers and EMA code are not reliably visible in torch's version
 * counters (fused Adam; `.data` arithmetic as in tld/train.py:55-58), so the packed copy is refreshed, not cached. */
TLD_API int tld_denoiser_set_params_async(tld_denoiser* h, int n, const char* const* keys, const float* const* data,
                                          const int64_t* numels, void* stream);
/* Counter bumped by every forward-like call on the handle (tld_denoiser_forward, tld_sampler_generate, tld_sampler_edit,
 * tld_train_forward).
 * The activations tld_train_backward differentiates live in per-handle buffers: the caller stores the value returned right
 * after tld_train_forward and may only run the backward while it is unchanged (tld_train_backward re-checks it). */
TLD_API long long tld_forward_serial(tld_denoiser* h);
/* Number of parameters still missing after the set_param calls (0 = ready). */
TLD_API int tld_denoiser_missing_params(tld_denoiser* h);

/* ---- Denoiser.forward (tld/denoiser.py:116-126) ---------------------------------------------
 * x[B,C,H,W], noise_level[B,1], label[B,text_emb] -> out[B,C,H,W]; all fp32 device pointers. */
TLD_API int tld_denoiser_forward(tld_denoiser* h, const float* x, const float* noise_level, const float* label,
                         float* out, int batch, void* stream);

/* ---- DiffusionGenerator.generate minus the VAE decode (tld/diffusion.py:54-89) --------------
 * labels[num_imgs,text_emb] (the cond half; the zero uncond half is implicit, diffusion.py:61),
 * seeds[num_imgs,C,H,W] initial noise (diffusion.py:105-120), latent_out[num_imgs,C,H,W] = final x0_pred.
 * noise_levels: HOST pointer to the n_levels >= 2 noise levels the model is called at, i.e. the list built at
 * diffusion.py:50-52 (the caller computes it: the sinusoidal embedding multiplies the level by up to 2*pi*1000,
 * so the levels must be bit-identical to the reference's fp32 torch.arange/pow values; [0] is forced to 0.99
 * here as well).  n_levels model calls are made (n_levels-1 updates + the final prediction, diffusion.py:66,85).
 * One diffusion step (2B-sample CFG forward + guidance + multistep update) is one CUDA-graph launch. */
TLD_API int tld_sampler_generate(tld_denoiser* h, const float* labels, const float* seeds, float* latent_out,
                                 int num_imgs, const double* noise_levels, int n_levels, float class_guidance,
                                 float sharp_f, float bright_f, int use_ddpm_plus, void* stream);
/* ---- image-to-image and masked inpainting on the same sampler ----------------------------------
 * init_latent[num_imgs,C,H,W]: the known latent x0k in denoiser space (VAE latent / scale_factor); noise[num_imgs,C,H,W]:
 * eps; mask[num_imgs,1,H,W] or NULL: 1 = regenerate, 0 = keep, clamped to [0,1] on the device (no host check).  All fp32
 * device pointers.  noise_levels (HOST, n_levels >= 2) are the tail sig[i0:] of the generate schedule and are used
 * verbatim; from_pure_noise = 1 means i0 == 0: the first level is forced to 0.99 and sampling starts from eps.
 *   start:  x = eps (from_pure_noise) or sig[0]*eps + (1-sig[0])*x0k (the training corruption, tld/train.py:130)
 *   loop:   the generate loop over the given levels (DPM-Solver++ ratios from these levels, first step first order); with a
 *           mask, after each update to level next: x = m*x + (1-m)*(next*eps + (1-next)*x0k), the same eps every step
 *   output: latent_out = m*x0 + (1-m)*x0k (x0 without a mask); no sharp / bright shifts.
 * Without a mask and with from_pure_noise = 1 the result is bit-identical to tld_sampler_generate with sharp_f = bright_f = 0.
 * Unmasked edits replay the generate step graph; masked edits use a second cached graph.  One launch more than generate. */
TLD_API int tld_sampler_edit(tld_denoiser* h, const float* labels, const float* noise, const float* init_latent,
                             const float* mask, float* latent_out, int num_imgs, const double* noise_levels, int n_levels,
                             int from_pure_noise, float class_guidance, int use_ddpm_plus, void* stream);
/* Device time of the sampling loop of the last tld_sampler_generate / tld_sampler_edit call (ms, CUDA events) and number of
 * kernel launches (graph nodes x replays + prologue) it issued. */
TLD_API int tld_sampler_last_stats(tld_denoiser* h, float* loop_ms, int64_t* kernel_launches);

/* ---- single ops, exported for the parity tests (tests/test_ops_gpu.py) -----------------------
 * Same kernels the forward uses, one at a time.  bf16 tensors are passed as raw uint16 device pointers. */
/* out = A[M,K] * W[N,K]^T with epilogue `epi`: 0 bf16 | 1 +bias bf16 | 2 x_f32 += acc+bias | 4 f32 */
TLD_API int tld_op_gemm(int epi, const uint16_t* A, const uint16_t* W, int M, int N, int K, void* out,
                const float* bias, void* stream);
/* C[M,N] = A^T B with A stored [K,M] and B stored [K,N] (bf16, row-major over K): the weight-gradient product
 * dW = dY^T X of the training step (tld/train.py:169 via autograd) on MN-major tcgen05 operands, no transposed copies.
 * epi 0: bf16 out, 4: fp32 out. */
TLD_API int tld_op_gemm_mn(int epi, const uint16_t* A, const uint16_t* B, int M, int N, int K, void* out, void* stream);
/* C[M,N] = A B with A [M,K] and B stored [K,N]: the data-gradient product dX = dY W with the weight as stored (MN-major B). */
TLD_API int tld_op_gemm_nn(int epi, const uint16_t* A, const uint16_t* B, int M, int N, int K, void* out, void* stream);
/* q-projection GEMM fused with the 2-key cross-attention and residual add (transformer_blocks.py:70-72,137):
 * x[M,D] += softmax2(q k0, q k1)(v0,v1) with q = A Wq^T; kv0/kv1 [rows, 2D] fp32 (K | V). */
TLD_API int tld_op_gemm_xattn(const uint16_t* A, const uint16_t* Wq, int M, int D, float* x, const float* kv0,
                      const float* kv1, int n_tok, void* stream);
/* LayerNorm folding (norm1 -> qkv_linear, norm3 -> mlp.0; transformer_blocks.py:136,138): the LayerNorm kernels disappear.
 * Consumer: out_bf16[M,N] = rstd_r (A Wf^T - mean_r col_s) + col_c with A = bf16 of the UN-normalised rows, Wf = bf16(gamma (.) W),
 * col_s[n] = sum_k Wf[n,k], col_c[n] = sum_k beta[k] W[n,k] (+ bias); mean_r / rstd_r from row_part [M, n_part] partial (sum, sum of
 * squares) of the fp32 rows (n_part = K/32, fixed summation order: deterministic). */
TLD_API int tld_op_gemm_lnfold(const uint16_t* A, const uint16_t* Wf, int M, int N, int K, uint16_t* out, const float* col_c,
                               const float* col_s, const float* row_part, int n_part, void* stream);
/* Producers: x_f32[M,N] = x + A W^T + bias written back explicitly, plus xb_out = bf16(x_new) and part_out [M, N/32] = per-32-column
 * (sum, sum of squares) of the new rows - what the consumer above needs; the cross-attention variant adds the 2-key SDPA instead. */
TLD_API int tld_op_gemm_bias_resid_lnp(const uint16_t* A, const uint16_t* W, int M, int N, int K, float* x, const float* bias,
                                       uint16_t* xb_out, float* part_out, void* stream);
TLD_API int tld_op_gemm_xattn_lnp(const uint16_t* A, const uint16_t* Wq, int M, int D, float* x, const float* kv0,
                                  const float* kv1, int n_tok, uint16_t* xb_out, float* part_out, void* stream);
/* fp32 rows -> bf16 copy + [rows, D/32] partials (the patch embedding's rows); gamma-folded weight + its column constants */
TLD_API int tld_op_rowstats_cast(const float* x, uint16_t* xb, float* part, int rows, int D, void* stream);
TLD_API int tld_op_ln_fold_weights(const float* W, const float* gamma, const float* beta, const float* bias, uint16_t* Wf,
                                   float* s, float* c, int N, int K, void* stream);
TLD_API int tld_op_layernorm(const float* x, const float* gamma, const float* beta, uint16_t* y, int rows, int D,
                     void* stream);
/* x[T,D] += softmax(q k^T/8) v per (sample, head) from qkv[T,3D]; impl 0 = auto, 1 = mma.sync kernel,
 * 3 = tcgen05 persistent pipelined kernel (needs n_tok % 128 == 0; auto picks it when that holds) */
TLD_API int tld_op_self_attention(const uint16_t* qkv, float* x, int batch, int n_tok, int D, int impl, void* stream);
/* norm2 + CrossAttention over the two conditioning tokens + residual + norm3 in ONE row-wise kernel (transformer_blocks.py:
 * 62-75,137,138): x[batch*n_tok, D] += softmax2(q k0, q k1) (v0, v1) with q = LN2(x) Wq^T folded into the keys (u = Wq_h^T k_h
 * per head, so q is never formed), y = bf16(LN3(x_new)).  kv0 / kv1 [batch, 2D] (K | V rows of the noise and label tokens),
 * uk_scratch [2 * batch, D / 64, D] fp32.  Needs D % 128 == 0 (<= 1024) and n_tok % 32 == 0. */
TLD_API int tld_op_ln_xattn_ln(float* x, const float* g2, const float* b2, const float* g3, const float* b3, const uint16_t* Wq,
                               const float* kv0, const float* kv1, int batch, int n_tok, int D, float* uk_scratch, uint16_t* y,
                               void* stream);
/* SelfAttention of a block in ONE kernel for 256-token samples (transformer_blocks.py:51-59,24-48,136): x[batch*256, D] +=
 * softmax(q k^T / 8) v per (sample, head) with [q|k|v] = xn[batch*256, D] Wqkv[3D, D]^T computed inside the kernel by the CTA
 * pair that owns the (sample, head): the qkv tensor is never written.  Needs n_tok == 256 and D % 64 == 0. */
TLD_API int tld_op_qkv_attention(const uint16_t* xn, const uint16_t* Wqkv, float* x, int batch, int n_tok, int D, void* stream);
/* MLPSepConv front half in one kernel for 16x16-token samples (transformer_blocks.py:95-103): out[batch*256, N] bf16 =
 * GELU(dwconv3x3(A[batch*256, K] W[N, K]^T + col_c) + dw_b) with the hidden tensor kept on chip (CTA-pair tile = one image,
 * halo row exchanged through distributed shared memory).  Optional LayerNorm fold: row_sums [batch*256, 2] = (sum, sum of
 * squares) of the un-normalised fp32 rows that A is the bf16 copy of, col_s [N] = sum_k W_nk (W already scaled by gamma):
 * value = rstd (acc - mean col_s) + col_c.  Pass NULL for both for the plain bias epilogue.  N % 256 == 0. */
TLD_API int tld_op_gemm_up_dwconv_gelu(const uint16_t* A, const uint16_t* W, const float* col_c, const float* col_s,
                                       const float* row_sums, const float* dw_w9, const float* dw_b, uint16_t* out, int batch,
                                       int K, int N, void* stream);
TLD_API int tld_op_dwconv_gelu(const uint16_t* h, const float* w9, const float* bias, uint16_t* g, int batch, int grid,
                       int channels, void* stream);

/* ---- VAE decoder row-wise kernels (diffusers AutoencoderKL.decode, called at tld/diffusion.py:91) ------------
 * NHWC bf16 activations (== torch channels_last).  y = act(GroupNorm_groups(x + pre_bias) * gamma + beta), act = SiLU
 * if silu != 0; x,y [batch, hw, channels]; pre_bias (nullable: the producing conv's bias, folded in), gamma, beta
 * fp32 [channels]. */
TLD_API int tld_vae_group_norm(const uint16_t* x, const float* pre_bias, const float* gamma, const float* beta,
                               uint16_t* y, int batch, int hw, int channels, int groups, float eps, int silu,
                               void* stream);
/* out = x + h + bias[c] (ResnetBlock2D tail; bias nullable), NHWC bf16, numel elements */
TLD_API int tld_vae_add_bias(const uint16_t* x, const uint16_t* h, const float* bias, uint16_t* out, long long numel,
                             int channels, void* stream);
/* 3x3 'same' convolution as an implicit GEMM on the tcgen05 core (4-D TMA boxes shifted per tap, zero fill = padding):
 * x NHWC bf16 [batch,h,w,cin], w bf16 [cout, 9*cin] with K order (ky,kx,cin), bias fp32 [cout] or NULL,
 * out NHWC bf16 [batch,h,w,cout]; cin,cout multiples of 64, h*w multiple of 128. */
TLD_API int tld_vae_conv3x3(const uint16_t* x, const uint16_t* w, const float* bias, uint16_t* out, int batch, int h,
                            int w_px, int cin, int cout, void* stream);
/* The same convolution with the ResnetBlock tail in its epilogue: out = conv(x) + bias + residual (residual NHWC bf16
 * [batch,h,w,cout] or NULL), and - if gn_partials is not NULL - the GroupNorm statistics partials of the STORED output,
 * gn_partials fp32 [batch*h*w/32, cout/4, 2] = (sum, sum of squares) per 32-pixel slab and 4-channel quad, for
 * tld_vae_group_norm_from_conv.  bias must not be NULL here. */
TLD_API int tld_vae_conv3x3_fused(const uint16_t* x, const uint16_t* w, const float* bias, uint16_t* out, int batch, int h,
                                  int w_px, int cin, int cout, const uint16_t* residual, float* gn_partials, void* stream);
/* act(GroupNorm(x)) with the statistics taken from the producing convolution's partials (x is read once, not twice) */
TLD_API int tld_vae_group_norm_from_conv(const uint16_t* x, const float* conv_partials, const float* gamma, const float* beta,
                                         uint16_t* y, int batch, int hw, int channels, int groups, float eps, int silu,
                                         void* stream);
/* softmax(q k^T / sqrt(channels)) v of the mid-block attention (ONE head as wide as the channel count): q, k, v, out bf16
 * [batch, n_tok, channels] (rows = pixels); per image a tcgen05 GEMM, a row softmax and a tcgen05 GEMM.  n_tok, channels % 64 == 0. */
TLD_API int tld_vae_attention_core(const uint16_t* q, const uint16_t* k, const uint16_t* v, uint16_t* out, int batch, int n_tok,
                                   int channels, void* stream);
/* decoder.conv_out (3x3 'same', 128 -> 3 channels): an HBM-bound direct convolution on the CUDA cores (nothing for a tensor core
 * to do with 3 output channels).  x NHWC bf16 [batch,h,w,128] (device); w_host [3,128,3,3] and b_host [3] are HOST fp32 arrays
 * (the 3456 weights travel in the kernel-parameter constant bank); out fp32 NCHW [batch,3,h,w] (device) = the final image. */
TLD_API int tld_vae_conv_out3(const uint16_t* x, const float* w_host, const float* b_host, float* out, int batch, int h, int w,
                              void* stream);
/* nearest-neighbour 2x upsample, NHWC bf16: x [batch,h,w,channels] -> y [batch,2h,2w,channels] */
TLD_API int tld_vae_upsample2x(const uint16_t* x, uint16_t* y, int batch, int h, int w, int channels, void* stream);
/* Image post-processing on the device (tld/diffusion.py:185, tld/train.py:36): img [batch,3,h,w] in [-1,1] (fp32, or bf16 when
 * is_bf16) -> ONE uint8 HWC grid out[GH, GW, 3] in torchvision.make_grid layout (min(ncol,batch) images per row, `pad`
 * black pixels around each; GH = rows*(h+pad)+pad, GW = cols*(w+pad)+pad), value = trunc(clip((x+1)/2, 0, 1) * 255) as
 * ToPILImage does.  Lets the caller copy 1 byte per sample to the host instead of 4. */
/* uint8 latent storage of the reference's dataset files (tld/data.py:51-60), bit-exact with the reference's arithmetic:
 * quantize: out[i] = trunc(((clip(lat[i], -c, c) / c + 1) / 2) * 255), lat fp32 or (is_fp16) fp16 with per-step fp16 rounding;
 * dequantize: out_fp16[i] = ((half(q[i]) / 255) * 2 - 1) * c, every step rounded to fp16. */
TLD_API int tld_latent_quantize(const void* lat, int is_fp16, uint8_t* out, long long n, float clip_val, void* stream);
TLD_API int tld_latent_dequantize(const uint8_t* q, uint16_t* out_fp16, long long n, float clip_val, void* stream);
TLD_API int tld_image_grid_u8(const void* img, int is_bf16, uint8_t* out, int batch, int h, int w, int ncol, int pad,
                              void* stream);

/* ---- CLIP text tower (tld/diffusion.py:136-140,160,177: clip_model.encode_text(clip.tokenize(prompt)); openai/CLIP model.py) ----
 * The linear layers run on tld_op_gemm (bias / bias + residual epilogues) and the LayerNorms on tld_op_layernorm; these are the
 * remaining row-wise pieces.  ids / eot: int64 device arrays ([batch, n_ctx] token ids; [batch] index of the EOT token).
 *   tld_clip_embed            x[b,t,:] = token_embedding[ids[b,t]] + positional_embedding[t]   (fp32 [batch*n_ctx, D])
 *   tld_clip_causal_attention out = softmax(q k^T / 8 + causal mask) v per (prompt, head) from qkv bf16 [batch*n_ctx, 3D]
 *                             (q | k | v as nn.MultiheadAttention's in_proj lays them out), head_dim 64, n_ctx <= 128
 *   tld_clip_quick_gelu       out = in * sigmoid(1.702 in), bf16, n elements (even)
 *   tld_clip_final            out[b] = LayerNorm(x[b, eot[b]]) @ proj   (proj fp32 [D, P] row-major = CLIP's text_projection) */
TLD_API int tld_clip_embed(const int64_t* ids, const float* token_embedding, const float* positional_embedding, float* x,
                           int batch, int n_ctx, int D, int vocab, void* stream);
TLD_API int tld_clip_causal_attention(const uint16_t* qkv, uint16_t* out, int batch, int n_ctx, int D, void* stream);
TLD_API int tld_clip_quick_gelu(const uint16_t* in, uint16_t* out, long long n, void* stream);
TLD_API int tld_clip_final(const float* x, const int64_t* eot, const float* gamma, const float* beta, const float* proj, float* out,
                           int batch, int n_ctx, int D, int P, void* stream);

/* ---- training step (tld/train.py:160-170: pred = model(x_noisy, sigma, label); loss.backward()) ---------------
 * tld_train_forward == tld_denoiser_forward but keeps the activations; tld_train_backward turns d(loss)/d(pred) into
 * the fp32 gradient of every parameter, read back per reference state_dict key with tld_train_get_grad (the caller
 * owns loss, optimiser, EMA and the data-parallel all-reduce, exactly as in the reference).  <= 256 tokens/sample. */
TLD_API int tld_train_forward(tld_denoiser* h, const float* x, const float* noise_level, const float* label, float* out,
                              int batch, void* stream);
TLD_API int tld_train_backward(tld_denoiser* h, const float* d_pred, int batch, void* stream);
TLD_API int tld_train_get_grad(tld_denoiser* h, const char* key, float* dst, int64_t numel, void* stream);
/* Data-parallel training (tld/train.py:109,169: accelerate/DDP all-reduces gradient buckets while the backward is still
 * running).  All gradients live in ONE device arena; tld_train_grad_layout returns it as n_layers + 2 ranges
 * (out[2i] = element offset, out[2i+1] = elements): range l < n_layers = decoder block l (without kv_linear), range n_layers =
 * all kv_linear weights, range n_layers + 1 = everything else.  tld_train_wait_grad makes `stream` wait (device-side only)
 * until range `segment` of the backward enqueued last is final (segment >= n_layers: the whole backward), so the caller can
 * all-reduce block l in place on a side stream while blocks l-1..0 are still being differentiated. */
/* Creates the gradient arena (layout only, no activations) so that tld_train_grad_layout / _offset can be queried before the
 * first training forward: the fused optimiser lays its parameter / moment / EMA arenas out exactly like the gradients. */
TLD_API int tld_train_prepare(tld_denoiser* h);
TLD_API int tld_train_grad_layout(tld_denoiser* h, float** arena, int64_t* total, int64_t* out, int n_segments);
TLD_API int tld_train_wait_grad(tld_denoiser* h, int segment, void* stream);
/* element offset / size of the gradient of `key` inside that arena (lets the caller snapshot all gradients with one copy) */
TLD_API int tld_train_grad_offset(tld_denoiser* h, const char* key, int64_t* offset, int64_t* numel);

/* ---- optimizer.step() + update_ema (tld/train.py:170,172-173,55-58) as ONE pass over flat fp32 arenas -------------
 * torch.optim.Adam's arithmetic (exp_avg.lerp_, exp_avg_sq.mul_.addcmul_, bias corrections 1 - beta^step as python floats,
 * param.addcdiv_) followed by ema = alpha * ema + (1 - alpha) * param on the UPDATED parameters.  All pointers are device
 * fp32 arrays of n elements laid out identically (the gradient arena of tld_train_grad_layout is the natural `grad`);
 * `ema` may be NULL (ranks other than 0 keep no EMA, tld/train.py:104-106,172).  `step` is the 1-based step count,
 * `grad_scale` multiplies the gradient first (1 = none).  weight_decay is Adam's L2 form (grad += wd * param). */
TLD_API int tld_adam_ema_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* ema, int64_t n,
                              double lr, double beta1, double beta2, double eps, double weight_decay, int64_t step,
                              double ema_alpha, double grad_scale, void* stream);

/* ---- backward-pass ops of the training step (autograd through tld/transformer_blocks.py:135-139, driven by
 * tld/train.py:160-170), exported for the parity tests (tests/test_backward_gpu.py) ------------------------------
 * in fp32 [rows,cols] -> out bf16 [rows,cols] (nullable) and outT bf16 [cols,rows] (nullable): operands of dgrad/wgrad */
TLD_API int tld_bwd_cast_transpose(const float* in, uint16_t* out, uint16_t* outT, int rows, int cols, void* stream);
/* out[c] = sum_r in[r,c] (bias gradients) */
TLD_API int tld_bwd_colsum(const float* in, float* out, int rows, int cols, void* stream);
/* LayerNorm backward: dx += dLN(dy; x, gamma); dgamma, dbeta [D] overwritten */
TLD_API int tld_bwd_layernorm(const float* dy, const float* x, const float* gamma, float* dx, float* dgamma, float* dbeta,
                              int rows, int D, void* stream);
/* depthwise-3x3 + GELU backward (token grid NHWC bf16): hid = conv input, dg = grad of the GELU output ->
 * dhid (grad of conv input), dw9 [9,C] tap-major, db [C]; du_tmp is a scratch buffer shaped like hid */
TLD_API int tld_bwd_dwconv_gelu(const uint16_t* hid, const uint16_t* dg, const float* w9, const float* bias,
                                uint16_t* du_tmp, uint16_t* dhid, float* dw9, float* db, int batch, int grid, int channels,
                                void* stream);
/* 2-key cross-attention backward: q bf16 [B*n_tok, D], go = d(out) fp32, kv0/kv1 [B, 2D] (K|V) -> dq bf16,
 * dkv0/dkv1 [B, 2D] accumulated with atomicAdd (zero them first) */
TLD_API int tld_bwd_xattn(const uint16_t* q, const float* go, const float* kv0, const float* kv1, uint16_t* dq, float* dkv0,
                          float* dkv1, int batch, int n_tok, int D, void* stream);
/* self-attention backward (n_tok <= 256): qkv bf16 [T,3D], d_out fp32 [T,D] (= residual gradient), x_before/x_after the
 * residual stream around the attention (O = x_after - x_before) -> dqkv bf16 [T,3D] */
TLD_API int tld_bwd_self_attention(const uint16_t* qkv, const float* d_out, const float* x_before, const float* x_after,
                                   uint16_t* dqkv, int batch, int n_tok, int D, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TLD_B200_H */
