/*
 * sdb200 — C ABI of the B200-native latent-diffusion kernels.
 *
 * The reference (CompVis/stable-diffusion) has no FFI: its plug-in boundary is `instantiate_from_config`
 * (ldm/util.py:78-93) plus the duck-typed nn.Module contracts around the denoising loop. This header is the
 * boundary a maintainer binds instead (ctypes stub in INTEGRATION.md): plain pointers and sizes, no torch
 * types. Every entry point enqueues work on `stream` and returns immediately; 0 = OK, non-zero = error
 * (text via sdb_last_error()). All device pointers are owned by the caller.
 *
 * Each function cites the reference operation(s) it replaces.
 */
#ifndef SDB200_H
#define SDB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* sdb_stream_t; /* cudaStream_t */

const char* sdb_last_error(void);
int sdb_version(void);
int sdb_sm_count(void);
long long sdb_launch_count(void); /* kernels launched through this library since load */
/* Debug only: subsequent sdb_gemm launches write per-CTA phase timestamps (8-word launch header + 8 words per CTA,
 * 1288 words per launch) into the device buffer `buf` of n_words uint64; NULL switches tracing off. Returns the
 * number of words handed out since the previous call. Used by scripts/timeline_unet.py. The stamps are written only by
 * a library built with -DSDB_TRACE (SDB_BUILD_TRACE=1 python build.py); the production build leaves the buffer untouched. */
long long sdb_debug_trace(void* buf, int64_t n_words);

/* ---- epilogue activations ---- */
enum {
  SDB_ACT_NONE = 0,
  SDB_ACT_GEGLU = 1,      /* out[:, j] = x_j * gelu_erf(gate_j); ldm/modules/attention.py:37-45 (weights packed
                             so each accumulator tile holds [x half | gate half]) */
  SDB_ACT_QUICK_GELU = 2, /* x * sigmoid(1.702 x): CLIP MLP (transformers CLIPMLP, quick_gelu) */
  SDB_ACT_SILU = 3        /* x * sigmoid(x): time_embed MLP, openaimodel.py:506-511 */
};

/*
 * Tensor-core GEMM / implicit-GEMM convolution (tcgen05 + TMA), fp16 operands, fp32 accumulate:
 *
 *   acc[m, n] = sum_k A[m, k] * B[n, k]
 *   v         = alpha * acc + bias[n] + film[m / rows_per_sample, n] + residual[m, n]
 *   out       = act(v)   written as fp16 and/or fp32, row stride ldo
 *
 * A is one to four NHWC fp16 tensors concatenated along channels: the UNet skip concat (openaimodel.py:736) folded
 * into the K loop, or the hi/lo fp16 halves of one fp32 activation ([A_hi | A_lo | A_hi] against [W_hi | W_hi | W_lo]
 * recovers ~fp32 operand precision for the few 1x1 convs that act on the raw residual stream). taps = 1: plain [rows, C] matrix (nn.Linear, 1x1 conv:
 * attention.py:161-168,233-248; openaimodel.py:241). taps = 9: 3x3 conv, stride 1, zero pad 1
 * (openaimodel.py:204,230,519,685; model.py:44-50,94-118) with B laid out [n, 9*(c0+c1)], k = tap*(c0+c1)+c.
 * All channel counts must be multiples of 64.
 */
typedef struct sdb_gemm_desc {
  const void* a0;        /* fp16 [nb, h, w, c0] */
  const void* a1;        /* fp16 [nb, h, w, c1] or NULL; further sources a2, a3 likewise (contiguous from a0) */
  const void* a2;
  const void* a3;
  int32_t c0, c1, c2, c3;
  int32_t nb, h, w;      /* rows M = nb*h*w */
  int32_t taps;          /* 1 or 9 */
  const void* b;         /* fp16 [n, taps*(c0+c1)] */
  int32_t n;
  float alpha;
  const float* bias;     /* [n] or NULL */
  const float* film;     /* [M / rows_per_sample, ldf] or NULL (timestep FiLM add, openaimodel.py:271-274) */
  int32_t ldf;           /* row stride of film (0 = n) */
  int32_t rows_per_sample;
  const float* residual; /* fp32 [M, ldr] or NULL */
  int32_t ldr;
  int32_t act;           /* SDB_ACT_* */
  void* out_f16;         /* fp16 [M, ldo] or NULL */
  void* out_f16_lo;      /* optional fp16 [M, ldo]: fp16(v - float(out_f16)), the low half of a hi/lo operand split */
  float* out_f32;        /* fp32 [M, ldo] or NULL */
  int32_t ldo;           /* 0 = dense (n, or n/2 for GEGLU) */
  int32_t block_n;       /* 0 = auto; else one of 32,64,128,160,256 */
  int32_t splits;        /* split-K factor: >1 explicit, 0/1 none, -1 auto (picked with block_n by the tile model,
                            bounded by workspace_floats); split-K needs workspace of splits*M*n floats */
  float* workspace;
  int64_t workspace_floats;
  void* stats_out;       /* optional fp32 [M / rows_per_sample, T, n / stats_group, 2]: per-tile partial {sum, sum of squares}
                            of the fp32 output per channel group, STORED by the epilogue of the tile that owns the slot
                            (no atomics, no zeroing, bit-reproducible) — the GroupNorm statistics of the tensor being
                            produced, so no separate reduction pass reads it again. T comes from sdb_gemm_plan; the
                            consumer (sdb_groupnorm) folds the T slots */
  int32_t b_dynamic;       /* non-zero: b is an activation produced by the preceding kernel (e.g. V^T = W_v . X^T swaps
                              the operand roles), so it must not be prefetched ahead of the programmatic-launch wait */
  int32_t conv_stride;     /* taps = 9 only. 0/1: stride 1. 2: stride-2 conv read straight from the NHWC input through
                              strided TMA boxes (no im2col): Downsample, openaimodel.py:149-153; model.py:72-76 */
  int32_t conv_shift;      /* input pixel of output o, tap t (per axis) = stride*o + t - 1 + conv_shift: 0 = zero pad 1
                              on every side (UNet), 1 = pad only right/bottom (the VAE's asymmetric F.pad, model.py:73) */
  int32_t in_h, in_w;      /* input height / width when they differ from the output's h / w (stride 2); 0 = h, w */
  int32_t pair;            /* 0 auto, 1 single CTAs, 2 CTA pairs: two CTAs of a cluster compute one 256 x block_n tile
                              with tcgen05.mma.cta_group::2, each loading half of the weight tile (block_n 128/160/256) */
  int32_t splitk_mode;     /* how split-K partials meet. 0 auto, 1 fp32 planes in `workspace` + a second kernel,
                              2 inside a thread-block cluster through distributed shared memory (2 or 4 slices, no
                              workspace traffic, fused epilogue in the same kernel) */
  int32_t stats_group;     /* channels per statistics entry (0/1 = per channel); must divide n and the tile width */
} sdb_gemm_desc;

int sdb_gemm(const sdb_gemm_desc* d, sdb_stream_t stream);
/* The tile configuration sdb_gemm would use for `d` (explicit requests honoured): out[0..4] = block_n, CTAs per tile
 * (1 | 2), split-K factor, split-K mode (0 none | 1 workspace | 2 cluster), statistics slots per sample T (0 when
 * stats_out is NULL). stats_out, when set, is written as fp32 [samples][T][n / stats_group][2]. */
int sdb_gemm_plan(const sdb_gemm_desc* d, int32_t* out);

/*
 * Fused multi-head attention (flash-style, S/P/O in TMEM), replaces CrossAttention.forward's
 * einsum -> scale -> softmax -> einsum (ldm/modules/attention.py:178-192) without materialising N x N.
 *   q  : fp16 [batch, nq,  heads*dpad]   (row stride ldq elements; head h at column h*dpad)
 *   k  : fp16 [batch, nkv, heads*dpad]   (row stride ldk)
 *   vt : fp16 [batch, heads*dpad, ldvt]  (V transposed: channel-major, nkv valid columns)
 *   out: fp16 [batch, nq, heads*d]       (row stride ldo; unpadded head dim d)
 * dpad in {64,128,192} (head dim zero-padded to a multiple of 64 by the projection weights: columns d .. dpad-1 of q / k
 * and rows d .. dpad-1 of each head of vt MUST be zero - the kernels only issue the tensor-core steps that hold real columns).
 * scale multiplies q.k before softmax (applied after the dot product, attention.py:180).
 * causal != 0 masks kv index > q index (CLIP text encoder).
 */
typedef struct sdb_attn_desc {
  const void* q;
  const void* k;
  const void* vt;
  void* out;
  int32_t batch, heads, nq, nkv, d, dpad;
  int32_t ldq, ldk, ldvt, ldo;
  int64_t q_batch_stride, k_batch_stride, vt_batch_stride, o_batch_stride; /* elements */
  float scale;
  int32_t causal;
} sdb_attn_desc;

int sdb_attention(const sdb_attn_desc* d, sdb_stream_t stream);

/*
 * GroupNorm(32) [+ SiLU] over NHWC fp32 input that may be the channel concat of two tensors
 * (ldm/modules/diffusionmodules/util.py:199-216 GroupNorm32 in fp32; attention.py:76-77 Normalize eps 1e-6;
 * model.py:38-39). Statistics: fp32 per-block partials, folded in fp64 by the last block of each sample. Writes the normalised fp16 operand
 * for the following conv and optionally a raw fp16 cast of the (concatenated) input for the 1x1 skip conv.
 */
int sdb_groupnorm(const float* x0, const float* x1, int32_t c0, int32_t c1, int32_t nb, int32_t hw, int32_t groups,
                  const float* gamma, const float* beta, float eps, int32_t silu, void* out_f16, void* raw_f16,
                  void* out_lo_f16 /* optional low half of the normalised output (hi/lo split) */,
                  void* raw_lo_f16 /* optional low half of the raw cast */,
                  void* stats_ws /* scratch: nb * (128*groups*2 + groups*2 + 1) * 4 bytes */,
                  const void* chan_stats0 /* optional fp32 [nb, stats_t0, c0 / stats_group, 2] from sdb_gemm.stats_out
                                             (skips the stats pass) */,
                  const void* chan_stats1 /* same for x1, [nb, stats_t1, c1 / stats_group, 2] */,
                  int32_t stats_t0, int32_t stats_t1 /* partial slots per sample (sdb_gemm_plan) */,
                  int32_t stats_group /* channels per entry; must divide c0, c1 and (c0 + c1) / groups */,
                  sdb_stream_t stream);

/* LayerNorm over the last dim of fp32 [rows, c] -> fp16 (attention.py:203-205, eps 1e-5). */
int sdb_layernorm(const float* x, int32_t rows, int32_t c, const float* gamma, const float* beta, float eps,
                  void* out_f16, float* out_f32 /* optional */, sdb_stream_t stream);

/* Row softmax of fp32 [rows, cols] * scale -> fp16 (VAE AttnBlock, model.py:191-194). */
int sdb_softmax_rows(const float* x, int32_t rows, int32_t cols, float scale, void* out_f16, sdb_stream_t stream);

/* ---- layout / elementwise helpers ---- */
/* NCHW fp32 -> NHWC fp32 (+ optional fp16 copy); NHWC fp32 -> NCHW fp32 */
int sdb_nchw_to_nhwc(const float* x, int32_t nb, int32_t c, int32_t hw, float* out_f32, void* out_f16,
                     sdb_stream_t stream);
int sdb_nhwc_to_nchw(const float* x, int32_t nb, int32_t c, int32_t hw, float* out, sdb_stream_t stream);
/* explicit im2col for the 3x3 convs whose C_in is not a multiple of 64, which the TMA path does not cover (UNet
 * conv_in, openaimodel.py:519; VAE conv_in, model.py:383,487): stride 1, zero pad 1, NHWC fp32 [nb, h, w, c] ->
 * fp16 [nb*h*w, kpad], k = (ky*3+kx)*c + ch, zero padded to kpad. */
int sdb_im2col3x3(const float* x, int32_t nb, int32_t h, int32_t w, int32_t c, int32_t kpad, void* out_f16,
                  sdb_stream_t stream);
/* nearest 2x upsample NHWC fp32 -> fp16 (openaimodel.py:116; model.py:54) */
int sdb_upsample2x(const float* x, int32_t nb, int32_t h, int32_t w, int32_t c, void* out_f16, sdb_stream_t stream);
/* fp32 -> fp16 cast, optional transpose of [rows, cols] per batch into [cols, ldo] */
int sdb_cast_f16(const float* x, int64_t n, void* out_f16, sdb_stream_t stream);
int sdb_transpose_f16(const void* x, int32_t batch, int32_t rows, int32_t cols, int32_t ldx, void* out,
                      int32_t ldo, sdb_stream_t stream);
/* sinusoidal timestep embedding [cos | sin] (util.py:151-171): t[n] -> fp32 [n, dim]; and the small-M
 * fp32-activation linear (time_embed MLP + all emb_layers, openaimodel.py:506-511,217-223):
 * out[m, j] = act(x[m, :] . w[j, :] + bias[j]), w fp16 [n, k], act NONE|SILU */
int sdb_timestep_embedding_f32(const float* t, int32_t n, int32_t dim, float max_period, float* out,
                               sdb_stream_t stream);
int sdb_linear_small(const float* x, int32_t m, int32_t k, const void* w_f16, int32_t n, const float* bias,
                     int32_t act, float* out_f32, void* out_f16, sdb_stream_t stream);

/*
 * One fused sampler update (classifier-free guidance + PLMS / DDIM step), replacing ~25 elementwise
 * launches per step (ldm/models/diffusion/plms.py:182-186,199-236; ddim.py:174-204).
 *   eps2   : fp32 [2, n] = [e_uncond; e_cond] (or [1, n] when guidance is off: scale==1)
 *   e_t    = e_uncond + scale * (e_cond - e_uncond)
 *   order 0: e' = e_t (DDIM / first PLMS half-step); 1..3: Adams-Bashforth with old eps h1,h2,h3
 *   order 4 (PLMS step 0 second half): e' = (e_t_old + e_t)/2 where e_t_old = h1
 *   pred_x0 = (x - sqrt(1-a_t) e') / sqrt(a_t);  x_prev = sqrt(a_prev) pred_x0 + sqrt(1-a_prev-sigma^2) e' + sigma*noise
 * coef = {a_t, a_prev, sigma_t, sqrt_one_minus_a_t}; e_t is written to e_out (for the multistep history).
 */
int sdb_sampler_step(const float* x, const float* eps2, const float* eps_cond /* NULL: eps2 + n. Otherwise the
                     conditional half lives elsewhere - e.g. in the peer GPU's buffer mapped over NVLink (CFG halves
                     evaluated on two GPUs, SURVEY 8f-2): the exchange is then the kernel's own peer loads */,
                     int32_t guided, float scale, int32_t order, const float* h1,
                     const float* h2, const float* h3, const float* noise, float a_t, float a_prev, float sigma_t,
                     float sqrt_one_minus_a_t, int64_t n, float* x_prev, float* x_prev2 /* optional second copy: the
                     cond half of the guidance-doubled latent batch */, float* pred_x0, float* e_out,
                     sdb_stream_t stream);

/*
 * DPM-Solver++ (multistep, order <= 2, data prediction) update fused with classifier-free guidance and the
 * noise -> x0 conversion: replaces model_wrapper.model_fn + DPM_Solver.data_prediction_fn +
 * dpm_solver_first_update / multistep_dpm_solver_second_update
 * (ldm/models/diffusion/dpm_solver/dpm_solver.py:321-346, 386-399, 504-533, 755-789).
 *   e   = e_uncond + scale (e_cond - e_uncond)            (eps2 as in sdb_sampler_step)
 *   m0  = (x - sigma_s e) / alpha_s                        -> m_out (the history entry for the next step)
 *   order 1: x_t = c_x x - c_m m0                          c_x = sigma_t / sigma_s, c_m = alpha_t * expm1(-h)
 *   order 2: x_t = c_x x - c_m m0 - (c_m / 2) inv_r0 (m0 - m_prev)      c_m = alpha_t * (exp(-h) - 1)
 * The host computes the scalars in fp32 exactly as the reference's schedule tensors do.
 */
int sdb_dpm_solver_step(const float* x, const float* eps2, const float* eps_cond /* as in sdb_sampler_step */,
                        int32_t guided, float scale, float sigma_s, float alpha_s,
                        int32_t order, const float* m_prev, float c_x, float c_m, float inv_r0, int64_t n,
                        float* m_out, float* x_out, float* x_out2 /* optional second copy */, sdb_stream_t stream);

/* Inpainting blend of the samplers' mask branch (plms.py:147-150, ddim.py:144-147), in place:
 * img = img_orig * mask + (1 - mask) * img; mask fp32 [nb, 1 or c, hw]; img2: optional second copy of the result. */
int sdb_mask_blend(const float* img_orig, const float* mask, int32_t mask_channels, int32_t nb, int32_t c, int64_t hw,
                   float* img, float* img2, sdb_stream_t stream);

/* VAE posterior sample + scale (distributions.py:24-37, ddpm.py:542-549): moments NHWC fp32 [rows, 8]
 * -> z NCHW. And image post-process clamp((x+1)/2,0,1)*255 -> uint8 NHWC (txt2img.py:314-324). */
int sdb_vae_sample(const float* moments, const float* noise_nchw, int32_t nb, int32_t hw, float scale_factor,
                   float* z_nchw, sdb_stream_t stream);
int sdb_to_uint8(const float* x_nhwc, int64_t n, uint8_t* out, sdb_stream_t stream);
/* out = a*x + b (latent scaling z/0.18215, ddpm.py:713) */
int sdb_axpby(const float* x, float a, float b, int64_t n, float* out, sdb_stream_t stream);
/* out = a*x + b*y (DDIMSampler.stochastic_encode, ddim.py:206-220; q_sample, ddpm.py:274-277) */
int sdb_axpby2(const float* x, const float* y, float a, float b, int64_t n, float* out, sdb_stream_t stream);

/* 1x1 conv with <= 16 channels in fp32 (post_quant_conv 4->4 with the 1/scale_factor folded in as alpha,
 * quant_conv 8->8; autoencoder.py:302-303,326,331): out[p, j] = sum_c (alpha x[p, c]) w[j, c] + b[j] */
int sdb_pointwise_small(const float* x, int64_t npix, int32_t cin, int32_t cout, const float* w, const float* b,
                        float alpha, float* out, sdb_stream_t stream);
/* CLIP token + position embedding gather (transformers CLIPTextEmbeddings): ids int64 [rows] -> fp32 [rows, dim] */
int sdb_embed_tokens(const int64_t* ids, int32_t rows, int32_t n_ctx, int32_t dim, int32_t vocab, const float* tok,
                     const float* pos, float* out, sdb_stream_t stream);

/* ---- post-processing of the decoded image: safety checker (scripts/txt2img.py:26-29, 88-95, 319) ----
 * The reference delegates to third-party code: transformers' CLIPFeatureExtractor (PIL bicubic resize of the shorter
 * side to 224, centre crop, 1/255, mean/std) and diffusers' StableDiffusionSafetyChecker (CLIP ViT-L/14 vision tower +
 * projection, cosine distance to 17 concept and 3 special-care embeddings). The vision tower runs on sdb_gemm /
 * sdb_attention / sdb_layernorm; these are the pieces around it. */
/* One pass of PIL's 8-bit ImagingResample over interleaved [n_img, H, W, 3] images: horizontal (vertical = 0: lines =
 * rows, in_size / out_size = widths) or vertical (vertical = 1: lines = columns, other_size_in = the row length W).
 * bounds int32 [out_size, 2] = {first source index, tap count}, coefs int32 [out_size, ksize] = 22-bit fixed-point
 * weights, both computed by the host exactly as PIL's precompute_coeffs / normalize_coeffs_8bpc. The source is uint8,
 * or fp32 in [0, 1] converted as numpy_to_pil does ((x * 255).round()). */
int sdb_resample_u8(const void* src_u8, const float* src_f32, int32_t n_img, int32_t lines, int32_t in_size,
                    int32_t out_size, int32_t ksize, const int32_t* bounds, const int32_t* coefs, int32_t vertical,
                    int32_t other_size_in, void* out_u8, sdb_stream_t stream);
/* centre crop to size x size, x / 255, (x - mean) / std: uint8 [nb, h, w, 3] -> fp32 NCHW [nb, 3, size, size] */
int sdb_clip_normalize(const void* img_u8, int32_t nb, int32_t h, int32_t w, int32_t size, float m0, float m1, float m2,
                       float s0, float s1, float s2, float* out_nchw, sdb_stream_t stream);
/* ViT patch extraction: NCHW fp32 [nb, 3, size, size] -> fp16 [nb * (size/patch)^2, kpad], k = (c * patch + py) * patch + px
 * (the flattening of CLIPVisionEmbeddings.patch_embedding.weight), zero-padded to kpad (multiple of 64) */
int sdb_patchify(const float* x_nchw, int32_t nb, int32_t size, int32_t patch, int32_t kpad, void* out_f16,
                 sdb_stream_t stream);
/* StableDiffusionSafetyChecker decision: scores fp32 [nb, n_special + n_concept] (rounded to 3 decimals as the
 * library does), flagged int32 [nb] */
int sdb_safety_scores(const float* image_embeds, int32_t nb, int32_t dim, const float* special_embeds,
                      const float* special_weights, int32_t n_special, const float* concept_embeds,
                      const float* concept_weights, int32_t n_concept, float* scores, int32_t* flagged,
                      sdb_stream_t stream);
/* images[i] = 0 for flagged images (fp32, per_image elements each) */
int sdb_blank_flagged(float* images, int64_t per_image, int32_t nb, const int32_t* flagged, sdb_stream_t stream);

/* Invisible watermark of scripts/txt2img.py:69-74, 261-264, 324 (third-party `invisible-watermark`: WatermarkEncoder
 * .encode(bgr, 'dwtDct') = EmbedMaxDct, scales [0, 36, 36], block 4) on uint8 RGB images [nb, h, w, 3]: cv2's 8-bit
 * RGB -> YUV, one watermark bit per 4x4 block of the Haar approximation band of U, YUV -> RGB. bits: uint8 [n_bits]
 * (0 / 1; "StableDiffusionV1" MSB first = 136 bits); yuv_scratch: nb*h*w*3 bytes. */
int sdb_watermark_dwtdct(const void* rgb_u8, int32_t nb, int32_t h, int32_t w, const void* bits_u8, int32_t n_bits,
                         float scale, void* yuv_scratch_u8, void* out_rgb_u8, sdb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Handle-level entry points: the engine, not just its kernels.
 *
 * A plan is the ordered list of sdb_* launches of one pass over the model, recorded (arguments copied by value) while
 * the host side walks the model once between sdb_plan_begin and sdb_plan_end - the calls still execute, so the
 * recording pass doubles as the warm-up. sdb_plan_launch replays it as ONE CUDA graph (captured on first use on a
 * private stream). Every pointer inside is a caller-owned static buffer (weights, workspaces, I/O) that must outlive
 * the plan. Recording is per host thread.
 */
typedef struct sdb_plan sdb_plan;
int sdb_plan_begin(sdb_plan** out);
int sdb_plan_end(sdb_plan* plan);
int sdb_plan_size(const sdb_plan* plan);                 /* recorded launches (-1: NULL) */
int sdb_plan_launch(sdb_plan* plan, sdb_stream_t stream); /* graph replay */
int sdb_plan_destroy(sdb_plan* plan);
int sdb_fill_f32(float* x, int64_t n, float value, sdb_stream_t stream);

/*
 * One guided UNet evaluation as a handle: replaces sampler -> LatentDiffusion.apply_model -> DiffusionWrapper.forward
 * -> UNetModel.forward (ldm/models/diffusion/ddpm.py:891-992,1393-1421; ldm/modules/diffusionmodules/openaimodel.py:
 * 710-742). `plan` was recorded over one evaluation whose first kernel reads x_static [n, c_in, h, w] (NCHW fp32) and
 * t_static [n] and whose last kernel writes eps_static [n, c_out, h, w]; the cross-attention context is baked into the
 * plan (its K / V buffers are static: re-fill them to change the prompt). sdb_unet_forward copies x / t in when they
 * are not the static buffers themselves (NULL = already in place), launches the graph and copies eps out (NULL = leave
 * it in eps_static).
 */
typedef struct sdb_unet sdb_unet;
int sdb_unet_create(sdb_plan* plan, float* x_static, float* t_static, float* eps_static, int32_t n, int32_t c_in,
                    int32_t c_out, int32_t h, int32_t w, sdb_unet** out);
int sdb_unet_forward(sdb_unet* unet, const float* x, const float* t, float* eps, sdb_stream_t stream);
int sdb_unet_destroy(sdb_unet* unet);

/*
 * A whole PLMS trajectory (ldm/models/diffusion/plms.py:98-236, eta = 0) on the device: per step one sdb_unet_forward
 * (two on the first step: pseudo improved Euler) and one fused sdb_sampler_step. The schedule is passed as host arrays
 * indexed like the reference's ddim_* arrays (index 0 = the LAST step taken); timesteps are the ddim_timesteps as
 * floats. `unet` evaluates 2 * batch samples when guided ([uncond; cond] halves of the latent), else batch.
 */
typedef struct sdb_plms_desc {
  sdb_unet* unet;
  const float* x;          /* x_T, fp32 [batch, c, h, w] (device) */
  float* x_out;            /* final latent [batch, c, h, w] (device; may alias x) */
  float* pred_x0_out;      /* optional: last predicted x0 */
  float* work;             /* device scratch: (5 + 2 * rep) * batch*c*h*w floats, rep = guided ? 2 : 1 */
  int32_t batch, n_steps, guided;
  float scale;             /* unconditional_guidance_scale */
  const float* timesteps;  /* host [n_steps] */
  const float* alphas;     /* host [n_steps] ddim_alphas */
  const float* alphas_prev;
  const float* sqrt_one_minus_alphas;
  const float* sigmas;     /* host [n_steps] or NULL (eta = 0) */
} sdb_plms_desc;
int sdb_sample_plms(const sdb_plms_desc* d, sdb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SDB200_H */
