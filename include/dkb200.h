/* dkb200 — C ABI of the B200-native denoise + decode engine behind DiffusionKit's
 * `diffusionkit.mlx` DiffusionPipeline / FluxPipeline API.
 *
 * The reference (argmaxinc/DiffusionKit @ 498e5dba) has no FFI boundary: its hot path sits behind a
 * Python class API and bottoms out in MLX library calls.  This header is the boundary a maintainer
 * would bind instead (ctypes stub in INTEGRATION.md).  Each entry point cites the reference code it
 * replaces (paths relative to python/src/diffusionkit/mlx/).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; dk_last_error() gives the message
 *     (thread-local).  No C++ exception crosses this boundary.
 *   - all pointers are DEVICE pointers unless a name ends in _host; buffers are caller-owned
 *     (torch tensors on the Python side); the library borrows them for the duration of a call
 *     (weights: until the model handle is destroyed).
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it.
 *   - dtype: DK_BF16 (FLUX: __init__.py:610) or DK_FP16 (SD3: __init__.py:76) for weights and
 *     activations; sampler state is fp32 (__init__.py:761-788).
 *   - layouts follow the reference: latents/images NHWC (mmdit.py:188-266, vae.py:386-401),
 *     Linear weights (out,in) (mlx nn.Linear), conv weights (O,kh,kw,I) (mlx nn.Conv2d).
 *
 * Why the boundary is at the OPERATOR level (and not dk_mmdit_forward / dk_vae_decode)
 *   The reference's own boundary to its accelerator library is the operator level: mmdit.py / vae.py are
 *   Python modules that call mx.fast.scaled_dot_product_attention, mx.fast.layer_norm, nn.Linear,
 *   nn.Conv2d, nn.GroupNorm one by one; model structure (block lists, which stream skips its post-attention
 *   path, the modulation cache keyed by timestep, the img2img branch) lives in Python and is what its
 *   maintainers edit.  This header replaces exactly that layer — every MLX call on the path has one entry
 *   point here, with the fusions expressed as epilogue/prologue arguments of those calls — so a binding keeps
 *   the reference's module code and swaps its library calls.  A model-level entry point would have to freeze
 *   the parameter-tree naming, six model configurations, the modulation cache and the quirk flags of
 *   SURVEY.md App. A.4 into a C struct.  The cost of staying at the operator level is launch overhead, which
 *   the host layer removes by capturing each forward / decode in a CUDA graph (one cudaGraphLaunch per
 *   MMDiT forward or VAE decode: diffusionkit_b200/mmdit.py, vae.py); a non-Python host does the same with
 *   cudaStreamBeginCapture around its own sequence of dk_* calls — every entry point is capture-safe (no
 *   allocation, no synchronisation, no host-side state beyond the launch counter).
 */
#ifndef DKB200_H
#define DKB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DK_BF16 0
#define DK_FP16 1

#define DK_ACT_NONE 0
#define DK_ACT_GELU_ERF 1 /* mlx nn.GELU() exact erf — mmdit.py:421,835 */
#define DK_ACT_SILU 2
#define DK_ACT_QUICK_GELU 3 /* x * sigmoid(1.702 x): mlx nn.gelu_fast_approx, CLIP-L "quick_gelu" — clip.py:11 */

typedef struct dk_ctx dk_ctx;

const char* dk_version(void);
const char* dk_last_error(void);
int dk_ctx_create(int device, dk_ctx** out);
void dk_ctx_destroy(dk_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
long long dk_ctx_launch_count(dk_ctx* ctx);

/* ---------------------------------------------------------------------------------------------
 * K1  tcgen05 GEMM with fused epilogue — replaces every nn.Linear on the path
 *     (mmdit.py:471-473 q/k/v, :532 o_proj, :830-835 FFN, :430-435 adaLN, :56-59 context_embedder,
 *      :357-361/:372-376 embedders, :771-774 final linear; vae.py:36-39 attention projections).
 *     out[row(m), n] = res[rrow(m), n] + gate[m / rows_per_batch, n] * act(sum_k A[m,k] W[n,k] + bias[n])
 *     row(m)  = (m / rows_per_batch) * out_batch_rows + out_row_off + m % rows_per_batch
 *     rrow(m) = (m / rows_per_batch) * res_batch_rows + res_row_off + m % rows_per_batch
 *     (the row maps let a stream's GEMM write straight into the joint [text|image] sequence buffer,
 *      mmdit.py:594-625, and let a per-position table broadcast over the batch, mmdit.py:334-349.)
 * ------------------------------------------------------------------------------------------- */
typedef struct dk_gemm_args {
  int dtype;
  int M, N, K;
  const void* A; /* [M, K] row-major, leading dim lda (elements) */
  long long lda;
  const void* W; /* [N, K] row-major (nn.Linear weight), leading dim ldw; if w_n_major: [K, N] */
  long long ldw;
  void* out; /* 16-bit output */
  long long ldc;
  const void* bias; /* [N] or NULL */
  const void* gate; /* [batches, gate_ld] or NULL */
  long long gate_ld;
  const void* res; /* residual or NULL (may alias out) */
  long long ldres;
  int rows_per_batch; /* 0 => M */
  int out_batch_rows, out_row_off;
  int res_batch_rows, res_row_off;
  int act;       /* DK_ACT_* applied to (acc + bias) */
  int w_n_major; /* 1: W is [K, N] row-major (exercises the MN-major operand path used for V) */
  /* fused epilogue for a packed [q | k | v] projection (N = 3 * qk_heads * qk_head_dim), qk_head_dim = 0 disables:
   * per head of the q and k thirds  x = RMSNorm(x; weight, qk_eps)  (mmdit.py:754-764; NULL weight = no norm)
   * then RoPE with table qk_rope[pos][pair] = (cos, sin), pos = out_row_off + m % rows_per_batch (mmdit.py:934-942;
   * NULL = no RoPE).  Replaces a separate dk_qk_norm_rope pass over the QKV buffer. */
  const void* qk_q_weight;
  const void* qk_k_weight;
  const float* qk_rope;
  int qk_heads, qk_head_dim;
  float qk_eps;
} dk_gemm_args;
int dk_gemm(dk_ctx* ctx, const dk_gemm_args* args, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2  LayerNorm (no affine, eps) + adaLN modulate: y = LN(x) * (1 + scale[b]) + shift[b]
 *     replaces affine_transform / mx.fast.layer_norm — mmdit.py:958-972, :838-849.
 *     x, y: [B*rows_per_batch, h]; shift/scale: row b at ptr + b*mod_ld (16-bit).
 * ------------------------------------------------------------------------------------------- */
int dk_ln_modulate(dk_ctx* ctx, int dtype, const void* x, void* y, const void* shift, const void* scale,
                   long long mod_ld, int rows, int rows_per_batch, int h, float eps, void* stream);

/* ---------------------------------------------------------------------------------------------
 * QK-RMSNorm (mmdit.py:754-764, eps 1e-6, learned weight) + FLUX RoPE (mmdit.py:934-942) applied
 * in place to the q and k thirds of a packed [rows, 3h] QKV buffer.
 *   rows = B * S; row r -> sequence position r % S.
 *   q_w/k_w: norm weights [d] for positions < split, q_w2/k_w2 for positions >= split (the text and
 *   image streams of a MultiModalTransformerBlock own separate QKNorm modules); NULL => no norm.
 *   rope: fp32 [S, d/2, 2] (cos, sin) or NULL (SD3: no RoPE).
 * ------------------------------------------------------------------------------------------- */
int dk_qk_norm_rope(dk_ctx* ctx, int dtype, void* qkv, int rows, int S, int heads, int d, int split, const void* q_w,
                    const void* k_w, const void* q_w2, const void* k_w2, const float* rope, float eps, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K3  attention forward: softmax(scale * Q K^T) V, no mask — replaces
 *     mx.fast.scaled_dot_product_attention (mmdit.py:562-563,643,687-688,736).
 *     qkv: packed [B*S, 3*heads*d] (q | k | v thirds, head-major inside a third).
 *     output row (b, s): s < split -> out0[(b*split + s) * ld0 + head*d ...]
 *                        else      -> out1[(b*(S-split) + s-split) * ld1 + head*d ...]
 *     (split = S with out1 = NULL writes one [B*S, ld0] buffer.)  d in {64, 128}.
 * ------------------------------------------------------------------------------------------- */
int dk_attention_fwd(dk_ctx* ctx, int dtype, const void* qkv, int B, int S, int heads, int d, float scale, int split,
                     void* out0, long long ld0, void* out1, long long ld1, void* stream);
/* Tuning hook for same-process A/B measurements of the K3 variants (no reference counterpart): split P publication
 * (0/1), exponentials per four evaluated on the FMA pipe (0..2), streamed exponential pass (0/1; 2 / 3 select the 64-key
 * double-buffered kernel of attention_v6.cu with two threads / one thread per row); a negative value
 * restores the built-in default / environment setting.  Results are bit-identical for every setting of split and
 * stream; poly changes P below its 16-bit rounding. */
int dk_attention_tuning(int split, int poly, int stream);

/* ---------------------------------------------------------------------------------------------
 * elementwise / layout kernels on the MMDiT path
 * ------------------------------------------------------------------------------------------- */
/* c[t*B + b, :] = silu(y[b, :] + temb[t, :])  — input of every adaLN Linear (mmdit.py:94-96, :430-431) */
int dk_silu_add(dk_ctx* ctx, int dtype, const void* y, const void* temb, void* c, int n_t, int B, int h, void* stream);
/* act(x) elementwise, 16-bit (MLP embedders: mmdit.py:357-361, :372-376) */
int dk_act(dk_ctx* ctx, int dtype, const void* x, void* y, long long n, int act, void* stream);
/* latent NHWC (B,H,W,C) 16-bit -> patch rows [B*(H/2)*(W/2), 4C].
 * order 0: (c, ph, pw)  FLUX reshape patchify (mmdit.py:292-302)
 * order 1: (ph, pw, c)  SD3 conv k2 s2 im2col, matches weight (O,kh,kw,I) (mmdit.py:285-290) */
int dk_patchify(dk_ctx* ctx, int dtype, const void* latent, void* rows, int B, int H, int W, int C, int order,
                void* stream);
/* rows [B*(H/2)*(W/2), 4C] 16-bit -> NHWC (B,H,W,C) 16-bit.  order 0: FLUX unpack (mmdit.py:304-321);
 * order 1: SD3 unpatchify (p, q, c) (mmdit.py:975-988) */
int dk_unpatchify(dk_ctx* ctx, int dtype, const void* rows, void* latent, int B, int H, int W, int C, int order,
                  void* stream);
/* crop of the learned position table (mmdit.py:334-349): table [max_hw*max_hw, h] -> out [hp*wp, h] */
int dk_pos_embed_crop(dk_ctx* ctx, int dtype, const void* table, void* out, int max_hw, int hp, int wp, int h,
                      void* stream);
/* copy [B, rows, h] blocks into a wider sequence buffer: dst[b, dst_off + r, :] = src[b, r, :] */
int dk_copy_rows(dk_ctx* ctx, int dtype, const void* src, void* dst, int B, int rows, int h, int dst_rows, int dst_off,
                 int src_rows, int src_off, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K6  sampler step (fp32 state) — CFGDenoiser + Euler update, __init__.py:691-719, :775-782,
 *     sampler.py:37-39.
 *   dk_sampler_prepare: xin[(k*B + b)] = cast16(x[b]) for k in 0..reps-1  (reps = 2 when cfg > 0, :700-706)
 *   dk_sampler_step:    den = float(xin) - float(out) * sigma; if cfg: den = den_neg + w (den_text - den_neg)
 *                       x += ((x - den) / sigma) * (sigma_next - sigma)
 * ------------------------------------------------------------------------------------------- */
int dk_sampler_prepare(dk_ctx* ctx, int dtype, const float* x, void* xin, long long n_per_rep, int reps, void* stream);
int dk_sampler_step(dk_ctx* ctx, int dtype, float* x, const void* xin, const void* out, long long n, float sigma,
                    float sigma_next, float cfg_weight, void* stream);
/* y = x * a + b (fp32): latent_format.process_out (__init__.py:732-733) and noise scaling (sampler.py:41-42) */
int dk_axpb_f32(dk_ctx* ctx, const float* x, float* y, long long n, float a, float b, void* stream);
/* ---- text encoders (SURVEY.md §8 row f2): CLIP-L/G (mlx/clip.py) and the T5-XXL encoder (mlx/t5.py) ------------- */
/* out[i] = table[ids[i]] (+ pos[i % pos_len]); table [vocab, d], pos [pos_len, d] or NULL   (clip.py:97-98, t5.py:322) */
int dk_embedding(dk_ctx* ctx, int dtype, const void* table, const int* ids, const void* pos, void* out, long long n,
                 int d, int vocab, int pos_len, void* stream);
/* y = LN(x) * weight + bias, biased variance, fp32 statistics (mlx nn.LayerNorm; clip.py:32-33,78) */
int dk_layernorm(dk_ctx* ctx, int dtype, const void* x, void* y, const void* weight, const void* bias, int rows, int h,
                 float eps, void* stream);
/* T5 RMSNorm over the fp32 residual stream: y = (dtype)(weight * x * rsqrt(mean(x^2) + eps))   (t5.py:150-170) */
int dk_rmsnorm_f32(dk_ctx* ctx, int dtype, const float* x, const void* weight, void* y, int rows, int d, float eps,
                   void* stream);
/* x (fp32) += y (16-bit): T5 keeps the residual stream in fp32 (t5.py:214-221) */
int dk_add_f32_16(dk_ctx* ctx, int dtype, float* x, const void* y, long long n, void* stream);
/* out[r, f] = gelu_erf(h[r, f]) * h[r, F + f], h [rows, 2F] = x @ [wi_0 | wi_1]^T   (t5.py:195-199) */
int dk_glu_gelu(dk_ctx* ctx, int dtype, const void* h, void* out, long long rows, int F, void* stream);
/* short-sequence attention (S <= 512, head dim 64) over a packed (q | k | v) projection [B*S, 3*heads*64]:
 * out = softmax(scale * q k^T + rel_bias[head][j - i + S - 1] + (causal ? -6e4 * [j > i] : 0)) v
 * rel_bias [heads, 2S-1] 16-bit or NULL (T5 relative-position bias, t5.py:21-102); causal: CLIP mask (clip.py:84-90) */
int dk_attention_small(dk_ctx* ctx, int dtype, const void* qkv, const void* rel_bias, void* out, int B, int S, int heads,
                       int head_dim, float scale, int causal, void* stream);
/* MLX affine 4-bit Linear weights -> dense 16-bit (the `*-4bit-quantized` model versions, reference
 * mlx/model_io.py:728-734, 772-775: nn.quantize with MLX defaults group_size 64, bits 4).
 * wq [N, K/8] uint32 (8 nibbles per word, element 0 in the low bits); scales, biases [N, K/group_size] 16-bit;
 * out[n, k] = scales[n, k/group] * q[n, k] + biases[n, k/group]  (one fp32 FMA, rounded once to `dtype`) */
int dk_dequant_q4(dk_ctx* ctx, int dtype, const uint32_t* wq, const void* scales, const void* biases, void* out,
                  long long N, int K, int group_size, void* stream);
/* read_image (__init__.py:536-551): uint8 [pixels, src_channels >= 3] -> 16-bit [pixels, cpad]; channels 0..2 =
 * u8 / 255 * 2 - 1, the padding channels are zero */
int dk_image_pre(dk_ctx* ctx, int dtype, const uint8_t* img, void* out, long long pixels, int src_channels, int cpad,
                 void* stream);
/* out = a * x + b * y (fp32): img2img noise scaling sigma * noise + (1 - sigma) * latent (sampler.py:41-42) */
int dk_axpby_f32(dk_ctx* ctx, const float* x, const float* y, float* out, long long n, float a, float b, void* stream);
/* VAE-encoder posterior sample + process_in: hidden [pixels, 2C] 16-bit = (mean | logvar);
 * out = ((mean + exp(0.5 * clip(logvar, -30, 20)) * noise) - shift) * scale   (__init__.py:586-594, :729-730) */
int dk_vae_sample_latent(dk_ctx* ctx, int dtype, const void* hidden, const float* noise, float* out, long long pixels,
                         int C, float shift, float scale, void* stream);
/* fp32 <-> 16-bit casts */
int dk_cast_f32_to_16(dk_ctx* ctx, int dtype, const float* x, void* y, long long n, void* stream);
int dk_cast_16_to_f32(dk_ctx* ctx, int dtype, const void* x, float* y, long long n, void* stream);

/* ---------------------------------------------------------------------------------------------
 * VAE decoder kernels (vae.py:20-149, 336-401)
 * ------------------------------------------------------------------------------------------- */
/* K7a GroupNorm statistics (nn.GroupNorm(32, C, pytorch_compatible=True), eps 1e-5; vae.py:34,72,78):
 *     stats[(b*G + g)*2 + {0,1}] = mean, rstd over (H*W, C/G); x NHWC 16-bit.
 *     ws: scratch of dk_groupnorm_ws_floats(B, G) floats (two-stage deterministic reduction, no atomics). */
int dk_groupnorm_ws_floats(int B, int G);
int dk_groupnorm_stats(dk_ctx* ctx, int dtype, const void* x, float* stats, float* ws, int B, int HW, int C, int G,
                       float eps, void* stream);
/* GroupNorm apply (+ optional SiLU): y = act((x - mean) * rstd * gamma[c] + beta[c]) */
int dk_groupnorm_apply(dk_ctx* ctx, int dtype, const void* x, void* y, const float* stats, const void* gamma,
                       const void* beta, int B, int HW, int C, int G, int silu, void* stream);
/* K7  conv 3x3, stride 1, zero pad 1, NHWC, as an im2col-free implicit GEMM: the 9 taps are 9 shifted TMA
 *     boxes of the input (out-of-bounds = zero fill = the padding), accumulated in TMEM.
 *     x [B,H,W,Cin] (Cin % 64 == 0), w [Cout,3,3,Cin] (Cout % 8 == 0), bias [Cout], res NHWC [B,H,W,Cout] or NULL
 *     (the ResnetBlock2D skip, vae.py:99).  replaces nn.Conv2d 3x3 (vae.py:73-81,134-136,349-351,384) */
int dk_conv3x3(dk_ctx* ctx, int dtype, const void* x, const void* w, const void* bias, const void* res, void* out,
               int B, int H, int W, int Cin, int Cout, void* stream);
/* 3x3 convolution with stride 2 and mlx's (0,1),(0,1) bottom/right zero padding — the VAE encoder's downsample
 * (vae.py:130-132,142-144).  x [B,H,W,Cin] (H, W even) -> out [B,H/2,W/2,Cout].  Same TMA implicit GEMM; the tap tile is
 * a 4-D box traversed with element stride 2. */
int dk_conv3x3_s2(dk_ctx* ctx, int dtype, const void* x, const void* w, const void* bias, void* out, int B, int H, int W,
                  int Cin, int Cout, void* stream);
/* K7f fused ResNet-path convolution (csrc/conv_fused.cu): [GroupNorm-apply + SiLU on the input] -> [nearest 2x] ->
 *     conv 3x3 (+ bias, + skip) -> output AND the GroupNorm partial statistics of the output, in ONE kernel.
 *     replaces nn.GroupNorm + nn.SiLU + nn.Conv2d (+ skip) of ResnetBlock2D (vae.py:60-101) and
 *     upsample_nearest + nn.Conv2d of the upsample stages (vae.py:20-25,146-147).
 *     x NHWC [B,H,W,Cin] RAW (pre-norm); gn_stats [B,G,2] (mean, rstd) + gamma/beta [Cin] normalise it on the fly while
 *     the 64-channel halo tile sits in shared memory (NULL: no norm); silu != 0 applies x*sigmoid(x) after the affine.
 *     up == 0: w [Cout,3,3,Cin], out [B,H,W,Cout].   up == 1: conv3x3(nearest2x(x)) by sub-pixel phases,
 *     w = the phase weights made by dk_conv_up_weights [4*Cout, 4*Cin], out [B,2H,2W,Cout].  res like out, or NULL.
 *     out_partial [B, slots, out_G, 2], slots = output pixels / 128: (sum, sum of squares) of the STORED output per
 *     128-pixel row segment and channel group, folded by dk_groupnorm_finalize (NULL: not wanted).
 *     Shapes: W % 128 == 0, H % 4 == 0, Cin % 64 == 0 (<= 512), Cout % 128 == 0 — dk_conv_fused_supported says. */
int dk_conv_fused_supported(int H, int W, int Cin, int Cout);
int dk_conv3x3_fused(dk_ctx* ctx, int dtype, const void* x, const void* w, const void* bias, const void* res, void* out,
                     int B, int H, int W, int Cin, int Cout, int up, const float* gn_stats, const void* gamma,
                     const void* beta, int G, int silu, float* out_partial, int out_G, void* stream);
/* Phase weights of conv3x3(nearest2x(.)): w [Cout,3,3,Cin] -> wp [4][Cout][2x2][Cin]; the 3x3 taps that fall on the
 * same source pixel are added in fp32 and rounded once (2.25x fewer FLOPs than convolving the upsampled tensor). */
int dk_conv_up_weights(dk_ctx* ctx, int dtype, const void* w, void* wp, int Cout, int Cin, void* stream);
/* Second stage of the GroupNorm statistics: partial [B, slots, G, 2] (sum, sumsq) -> stats [B, G, 2] (mean, rstd);
 * count = elements per (image, group).  Deterministic (fixed order, double accumulation). */
int dk_groupnorm_finalize(dk_ctx* ctx, const float* partial, float* stats, int B, int G, int slots, double count,
                          float eps, void* stream);
/* nearest 2x upsample NHWC (vae.py:20-25) */
int dk_upsample_nearest2x(dk_ctx* ctx, int dtype, const void* x, void* y, int B, int H, int W, int C, void* stream);
/* row softmax in place: x[r, :n] = softmax(scale * x[r, :n]); fp32 math, 16-bit storage (vae.py:49-52) */
int dk_softmax_rows(dk_ctx* ctx, int dtype, void* x, long long rows, int n, long long ld, float scale, void* stream);
/* clip(x/2 + 0.5, 0, 1) (and optional trunc(x*255) -> uint8): __init__.py:583, :526.
 * x NHWC [.., C_in_stride] 16-bit, takes the first 3 channels. */
int dk_image_post(dk_ctx* ctx, int dtype, const void* x, int c_stride, float* img_f32, uint8_t* img_u8, long long pixels,
                  void* stream);

/* ---------------------------------------------------------------------------------------------
 * masked img2img (inpainting).  No reference counterpart: the reference has no inpainting.  These compose with its
 * img2img flow: noise_scaling (sampler.py:41-42), the Euler step (__init__.py:779-781) and the decode tail
 * (__init__.py:583, :526).
 * ------------------------------------------------------------------------------------------- */
/* after an Euler step to sigma_next, re-noise the kept latent cells to the image's trajectory:
 * x = mask ? x : sigma_next * noise + (1 - sigma_next) * x0   (fp32; x0 = process_in of the posterior sample)
 * x0, noise, x [pixels, C] (C % 4 == 0, 16-byte aligned); mask one byte per latent pixel, non-zero = regenerate:
 * those cells of x are left untouched */
int dk_inpaint_blend(dk_ctx* ctx, const float* x0, const float* noise, const uint8_t* mask, float* x, long long pixels,
                     int C, float sigma_next, void* stream);
/* inpainting composite: img_u8 = mask ? dk_image_post's uint8 (bit-identical) : orig
 * x NHWC [.., c_stride] 16-bit decoder output, orig [pixels, 3] uint8, mask one byte per pixel (non-zero = decoded) */
int dk_image_post_masked(dk_ctx* ctx, int dtype, const void* x, int c_stride, const uint8_t* orig, const uint8_t* mask,
                         uint8_t* img_u8, long long pixels, void* stream);

/* ---------------------------------------------------------------------------------------------
 * one-time weight broadcast for multi-GPU batch sharding (no per-step collective).
 * The Python host uses torch.distributed (NCCL) for the rendezvous; these are thin NCCL wrappers
 * for hosts without torch.
 * ------------------------------------------------------------------------------------------- */
int dk_comm_unique_id(uint8_t id_host[128]);
int dk_comm_init(dk_ctx* ctx, int rank, int world, const uint8_t id_host[128]);
int dk_comm_broadcast(dk_ctx* ctx, void* ptr, size_t bytes, int root, void* stream);
int dk_comm_destroy(dk_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* DKB200_H */
