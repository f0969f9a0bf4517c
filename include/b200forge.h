/* b200forge.h — C ABI of libb200forge.so, the sm_100a kernel library that sits under
 * stable-diffusion-webui-forge's backend/ plug points (SURVEY.md §8b).
 *
 * Conventions
 *   - The caller owns every buffer (PyTorch allocates); the library allocates nothing persistent.
 *   - Every call enqueues on the given cudaStream_t (pass torch.cuda.current_stream().cuda_stream);
 *     no hidden synchronisation, safe under CUDA-graph capture.
 *   - Return 0 on success or a negative B200_E* code; never throws, never exits.
 *     b200_last_error() returns a thread-local human-readable message for the last failure.
 *   - dtype: B200_F16 or B200_BF16 for activations/weights; statistics and sampler state are fp32.
 *   - Activations inside the UNet are channels-last: an NHWC tensor is the row-major matrix
 *     [N*H*W, C]; a token tensor [b, L, C] is the same thing.
 *
 * Each entry point names the reference call site it replaces (paths relative to the reference tree).
 */
#ifndef B200FORGE_H
#define B200FORGE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* b200_stream_t; /* cudaStream_t */

enum { B200_OK = 0, B200_EINVAL = -1, B200_EUNSUPPORTED = -2, B200_ECUDA = -3, B200_ENODEVICE = -4 };
enum { B200_F16 = 0, B200_BF16 = 1 };
enum {
  B200_EPI_NONE = 0,
  B200_EPI_SILU = 1,  /* y = silu(acc + bias) */
  B200_EPI_GEGLU = 2, /* weight rows pre-interleaved per BN tile: y[:, j] = (x_j + b) * gelu_erf(gate_j + b) */
  B200_EPI_GELU = 3,  /* y = gelu_erf(acc + bias) */
  B200_EPI_GELU_TANH = 4 /* y = gelu_tanh(acc + bias)  (nn.GELU(approximate="tanh"), backend/nn/flux.py:193,202,280) */
};

int b200_version(void);
const char* b200_last_error(void);
/* 0 when a CUDA device of compute capability 10.x is visible, else B200_ENODEVICE. */
int b200_device_ok(void);
int b200_num_sms(void);

/* ---------------------------------------------------------------------------------------------
 * GEMM  C[M,N] = epi( A[M,K] @ B[N,K]^T + bias + rowvec + residual )       (tcgen05 + TMA + TMEM)
 * replaces: torch.nn.functional.linear via backend/operations.py:149-156 (ForgeOperations.Linear),
 *           1x1 Conv2d via backend/operations.py:169-176, GEGLU backend/nn/unet.py:104-111.
 * A may be the channel concatenation [A1 | A2] (torch.cat skip, backend/nn/unet.py:741) without a copy.
 */
typedef struct {
  int M, N, K;        /* K = K1 + K2 when A2 is given; K1 % 64 == 0 in that case            */
  int lda, ldb, ldc;  /* leading dimensions in elements (multiples of 8)                    */
  int dtype;
  int epilogue;       /* B200_EPI_*; GEGLU: N is the interleaved width (2x the output width) */
  int block_n;        /* 0 = choose; else multiple of 32, <= 256                              */
  const void* bias;   /* [N] (or [M] when bias_along_m), same dtype; may be NULL             */
  int bias_along_m;
  const void* residual; /* [M, N_out] added after the activation; may be NULL                */
  int ldr;
  const void* rowvec; /* [M / rows_per_vec, N] added before the activation (time-embedding)  */
  int ld_rowvec;
  int rows_per_vec;
  const void* A2;     /* second A source or NULL */
  int lda2;
  int K1;
  /* LayerNorm folded into the GEMM (replaces F.layer_norm + F.linear, backend/nn/unet.py:171-175 with operations.py:323-329):
   * A holds the un-normalised rows, B = W.diag(gamma); y = rstd_m*(acc - mean_m*ln_c[n]) + ln_d[n] with
   * ln_c = rowsum(B) and ln_d = W.beta (+ bias), both fp32 [N]; ln_stats [ln_stats_parts, M, 4] fp32 = partial row
   * statistics (count, mean, sum of squared deviations, 0) of each A row as a producer GEMM's row_stats_out wrote them;
   * the epilogue merges the partials with the parallel-variance formula (no sumsq/K - mean^2 cancellation). */
  const float* ln_stats;
  int ln_stats_parts;
  const float* ln_c;
  const float* ln_d;
  float ln_eps;
  /* when set, the epilogue writes partial statistics of every output row into row_stats_out
   * [b200_gemm_row_stats_parts(N, epilogue, block_n), M, 4] fp32 (part-major) — the ln_stats of the next GEMM, so no separate
   * LayerNorm pass touches HBM.  Each partial is written exactly once (no atomics, nothing to zero, bit-reproducible).
   * N must be a multiple of 32; not available with the GEGLU epilogue. */
  float* row_stats_out;
  /* Two row segments with their own weights — Flux DoubleStreamBlock (backend/nn/flux.py:206-264) keeps txt and img
   * tokens in one joint [B, L_txt + L_img, C] activation: rows with (m % seg_period) < seg_split use B / bias / rowvec,
   * the others B2 / bias2 / rowvec2 (same shapes and leading dimensions).  seg_period, seg_split multiples of 256.
   * B2 = NULL: one weight set (all other fields of this block ignored). */
  const void* B2;
  const void* bias2;
  const void* rowvec2;
  int seg_period, seg_split;
  int rowvec_mul; /* rowvec multiplies instead of adds: y = residual + rowvec * (acc + bias)  (modulation gate, flux.py:252-258,300) */
  int act_col0;   /* the activation applies to output columns >= act_col0 (multiple of block_n); SingleStreamBlock.linear1
                     = [qkv | mlp] with GELU on the mlp part only (flux.py:289-298) */
  float alpha;    /* 0 or 1: off; else the fp32 accumulators are multiplied by alpha first: C = epi(alpha * A B^T + ...).
                     The GEMM-softmax-GEMM attention paths put Dh^-1/2 here so that the stored logits are the SCALED ones
                     (unscaled fp16 logits can overflow; the reference scales q or the fp32 product, backend/attention.py:64-70) */
  /* K-split of the last, partly filled wave of output tiles (the persistent kernel walks T tiles on U = SMs [/ 2] units; the
   * T mod U tail tiles otherwise keep a few units busy for a whole tile time while the rest idle — 4.3 waves cost 5): the
   * tail tiles are cut along K into shares run by the idle units, which exchange fp32 partial accumulators through this
   * caller-owned scratch buffer: b200_gemm_workspace_bytes() bytes, 16-byte aligned, ZEROED ONCE by the caller (the kernel
   * leaves its flags zeroed), not shared by launches that may run concurrently (one buffer per stream).  NULL: no split.
   * Results do not depend on timing (fixed summation order), but differ in the last fp32 rounding from the unsplit sum. */
  void* workspace;
} b200_gemm_desc;

size_t b200_gemm_workspace_bytes(void);
int b200_gemm(const void* A, const void* B, void* C, const b200_gemm_desc* d, b200_stream_t s);
/* number of float4 partials per row that a b200_gemm with this N / epilogue / block_n writes to row_stats_out */
int b200_gemm_row_stats_parts(int N, int epilogue, int block_n);

/* ---------------------------------------------------------------------------------------------
 * 3x3 stride-1 pad-1 convolution on NHWC as an implicit GEMM (A tiles fetched by 4-D TMA boxes per
 * filter tap, zero fill = padding).  y[N,H,W,Cout] = epi(conv(x) + bias + temb[n, :] + residual)
 * replaces: torch.nn.Conv2d._conv_forward via backend/operations.py:169-176 inside
 *           ResBlock (backend/nn/unet.py:433-478), Upsample (:330-355), VAE ResnetBlock (backend/nn/vae.py:77-115).
 * Weights are packed [Cout, 9*(C1+C2)] with k = (ky*3+kx)*(C1+C2) + c.  C1, C2 multiples of 64.
 */
typedef struct {
  int N, H, W;
  int C1, C2; /* input = concat(x1[..., C1], x2[..., C2]); C2 = 0 for a single source */
  int Cout;
  int dtype;
  int epilogue;
  int block_n;
  const void* bias;     /* [Cout] */
  const void* residual; /* [N*H*W, Cout] */
  int ldr;
  const void* temb;     /* [N, ld_temb] row n added to every pixel of image n (ResBlock emb_layers) */
  int ld_temb;
  void* workspace;      /* K-split scratch, see b200_gemm_desc.workspace; NULL: no split */
} b200_conv3x3_desc;

int b200_conv3x3(const void* x1, const void* x2, const void* w_packed, void* y, const b200_conv3x3_desc* d,
                 b200_stream_t s);

/* Nearest-neighbour x2 upsample FOLDED into the following 3x3 convolution:
 *   y[N,2H,2W,Cout] = epi(conv3x3(upsample2x(x[N,H,W,C])) + bias (+ temb + residual, indexed on the 2H x 2W grid))
 * replaces: F.interpolate(scale_factor=2, mode="nearest") + self.conv in Upsample.forward (backend/nn/unet.py:330-355)
 *           and the VAE decoder's Upsample (backend/nn/vae.py:38-58) — without materialising the 4x tensor.
 * On the upsampled image every output pixel of parity (py, px) = (Y % 2, X % 2) sees only a 2x2 neighbourhood of the LOW-RES
 * image (rows y + py - 1, y + py; columns x + px - 1, x + px), so the 3x3 filter collapses to four 2x2 filters whose taps are
 * sums of the original ones (rows {0 | 1+2} for py = 0, {0+1 | 2} for py = 1; same for columns): 16 instead of 36
 * multiply-adds per output pixel and channel pair.  w_packed4 is [4*Cout, 4*(C1+C2)]: row (py*2+px)*Cout + co,
 * k = (ty*2+tx)*(C1+C2) + c, sums taken in fp32 and rounded once to the operand type (pack_conv3x3_up2x in ops.py).
 * The descriptor carries the LOW-RES N, H, W; any H, W (generic tiling, masked stores).
 */
int b200_conv3x3_up2x(const void* x1, const void* x2, const void* w_packed4, void* y, const b200_conv3x3_desc* d,
                      b200_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * Multi-head attention forward  O = softmax(Q K^T * scale) V   (FlashAttention-style, S and O tiles in
 * TMEM, K/V tiles by TMA, online softmax in registers).  No mask, no dropout, non-causal.
 * replaces: backend/attention.py:280-321 (attention_xformers) / :324-339 (attention_pytorch).
 * q/k/v/o point at head 0 of each operand; element (b, l, h, d) lives at
 *   ptr + b*stride_b + l*stride_l + h*Dh + d     (strides in elements, multiples of 8).
 * This lets q,k,v alias one fused QKV projection output without copies.  Dh must be 64 or 128.
 */
typedef struct {
  int B, H, Lq, Lk, Dh;
  long long q_stride_b, q_stride_l;
  long long k_stride_b, k_stride_l;
  long long v_stride_b, v_stride_l;
  long long o_stride_b, o_stride_l;
  float scale;
  int dtype;
} b200_attn_desc;

int b200_attention(const void* q, const void* k, const void* v, void* o, const b200_attn_desc* d, b200_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * GroupNorm on NHWC, split in a statistics pass and a fused apply(+SiLU)(+concat) pass.
 * replaces: torch.nn.functional.group_norm via backend/operations.py:304-310 and the following
 *           nn.SiLU (backend/nn/unet.py:395-396,418-419,691; backend/nn/vae.py:12-13,85).
 */
typedef struct {
  int N, HW;
  int C1, C2; /* channels of the two concatenated sources (C2 = 0: single source) */
  int groups;
  float eps;
  int silu;
  int dtype;
} b200_gn_desc;

/* Two launches share a caller-owned workspace `ws` of b200_groupnorm_ws_bytes(d) bytes (16-byte aligned): _stats reduces
 * each (sample, group) deterministically (fixed-order tree, sums shifted by a per-group pivot so that a large mean does not
 * cancel) and leaves (mean, rstd) in it, _apply normalises.  The first 4*N bytes of `ws` (ticket counters) must be zero
 * before the FIRST use; the kernel resets them, so one zero-initialised workspace serves any number of stream-ordered calls. */
size_t b200_groupnorm_ws_bytes(const b200_gn_desc* d);
int b200_groupnorm_stats(const void* x1, const void* x2, void* ws, const b200_gn_desc* d, b200_stream_t s);
int b200_groupnorm_apply(const void* x1, const void* x2, const void* ws, const void* gamma, const void* beta,
                         void* y, const b200_gn_desc* d, b200_stream_t s);

/* LayerNorm over the last dimension of [rows, C]; gamma/beta may be NULL (Flux: no affine).
 * replaces: torch.nn.functional.layer_norm via backend/operations.py:323-329. */
int b200_layernorm(const void* x, const void* gamma, const void* beta, void* y, int rows, int C, float eps,
                   int dtype, b200_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * Layout / gather helpers (HBM-bound).
 */
int b200_fill_zero(void* p, size_t bytes, b200_stream_t s);
/* nearest-neighbour x2 upsample on NHWC (F.interpolate(mode="nearest"), backend/nn/unet.py:352). */
int b200_upsample2x(const void* x, void* y, int N, int H, int W, int C, int dtype, b200_stream_t s);
/* im2col for 3x3 convs that the TMA path does not cover (C not a multiple of 64, stride 2):
 * out[(n,ho,wo), (ky*3+kx)*C + c] zero padded to ldo columns.  pad_lo is the top/left zero padding
 * (1 for the UNet convs; 0 for the VAE encoder's asymmetric (0,1,0,1) pad). */
int b200_im2col3x3(const void* x, void* out, int N, int H, int W, int C, int stride, int pad_lo, int Ho, int Wo,
                   int ldo, int dtype, b200_stream_t s);
/* y[(n,h,w), c] = x[n,c,h,w] * scale for c < C, 0 for C <= c < ldy (channel padding for the TMA/GEMM paths);
 * x is fp32 when in_is_f32 else dtype.  Used at the UNet/VAE entry (NCHW latents). */
int b200_nchw_to_nhwc(const void* x, void* y, int N, int C, int H, int W, int ldy, float scale, int in_is_f32,
                      int dtype, b200_stream_t s);
int b200_nhwc_to_nchw(const void* x, void* y, int N, int C, int H, int W, int ldx, int out_is_f32, int dtype,
                      b200_stream_t s);
/* y = silu(x) elementwise (SiLU in front of ResBlock.emb_layers, backend/nn/unet.py:412). */
int b200_silu(const void* x, void* y, size_t n, int dtype, b200_stream_t s);
/* Row softmax in place on [rows, cols] with scale; columns >= valid_cols are treated as masked and written as 0
 * (VAE single-head attention, backend/nn/vae.py:118-137; generic head dims with padded key counts). */
int b200_softmax_rows(void* x, int rows, int cols, int valid_cols, int ld, float scale, int dtype, b200_stream_t s);
/* Block-diagonal variant: row r attends to columns (r / block_rows) * block_cols + [0, valid_in_block) only and every other
 * column is written as 0.  S = Q_h K_h^T over a whole batch [B*Lq, B*Lk] followed by this softmax and P V_h is per-sample
 * attention for one head in three launches — the path for head dims the flash kernels do not cover (SD1.5's 160,
 * backend/nn/unet.py:133-155 with num_heads = 8 at 1280 channels). */
int b200_softmax_rows_blockdiag(void* x, int rows, int cols, int ld, float scale, int block_rows, int block_cols,
                                int valid_in_block, int dtype, b200_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * UNet entry: sinusoidal timestep embedding (backend/nn/unet.py:55-67) -> [B, dim] in dtype,
 * [cos | sin] order, freqs = exp(-ln(max_period) * i / half).
 */
int b200_timestep_embedding(const float* t, void* out, int B, int dim, float max_period, int dtype, b200_stream_t s);

/* KModel input scaling + layout + im2col for conv_in in one pass
 * (backend/modules/k_model.py:27,34; backend/modules/k_prediction.py:74-79; conv_in backend/nn/unet.py:553):
 * x fp32 NCHW [B, C, H, W], sigma fp32 [B]  ->  cols[(b,h,w), (ky*3+kx)*C + c] = x / sqrt(sigma^2 + 1), zero padded to ldo.
 * The batch is written `reps` times (cond/uncond batching, backend/sampling/sampling_function.py:234). */
int b200_unet_input_im2col(const float* x, const float* sigma, void* cols, int B, int C, int H, int W, int ldo,
                           int reps, int dtype, b200_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * Fused denoise epilogue + CFG + sampler update, one launch per step.
 * replaces: KModel.apply_model tail (backend/modules/k_model.py:45-46, k_prediction.py:81-92),
 *           the CFG combine (backend/sampling/sampling_function.py:276-289,312) and the per-step
 *           update of k_diffusion/sampling.py:119-137 (euler), :140-159 (euler ancestral), :648-671 (dpm++ 2m).
 * eps: UNet output, NHWC [(2 or 1)*B, H, W, ld_eps] in dtype; rows [0,B) = uncond, [B,2B) = cond
 *      (the reference batches [uncond, cond], sampling_function.py:186-188); has_uncond = 0 -> cond only.
 * x (fp32 NCHW [B,C,H,W]) is updated in place; denoised (fp32 NCHW) is written every step
 * (callback 'denoised'); old_denoised is read+written for DPM++ 2M.
 * All sigma-dependent scalars are precomputed on the host for the whole schedule (no device->host syncs):
 *   euler / euler_a : x += (x - D)/sigma * dt  [+ noise * noise_scale]
 *   dpmpp_2m        : x = c_x * x + c_d * D + c_old * D_old
 */
enum {
  B200_STEP_EULER = 0,
  B200_STEP_DPMPP_2M = 1,
  /* b200_sampler_update only: x = c_x*x + c_d*denoised + c_old*old_denoised + noise_scale*noise, all operands read-only
   * (the second stage of Heun / DPM2 / DPM++ 2S steps, k_diffusion/sampling.py:188-290, 573-603) */
  B200_STEP_LINEAR = 2
};
typedef struct {
  int kind;
  int B, C, H, W;
  int ld_eps;
  int has_uncond;
  int prediction; /* 0 = epsilon (D = x - eps*sigma), 1 = v_prediction, 2 = const/flow (D = x - v*sigma) */
  float sigma;    /* sigma_i (sigma_hat) */
  float cfg_scale;
  float dt;          /* euler: sigma_down - sigma_i */
  float noise_scale; /* euler ancestral: s_noise * sigma_up (0: no noise read) */
  float c_x, c_d, c_old; /* dpm++ 2m coefficients */
  int eps_dtype;
} b200_step_desc;

int b200_sampler_step(float* x, const void* eps, const float* noise, float* denoised, float* old_denoised,
                      const b200_step_desc* d, b200_stream_t s);

/* The update alone, for samplers installed under an unmodified CFGDenoiser (plug point P4): `denoised` is what
 * the model callable returned (fp32 NCHW).  Same scalars as b200_sampler_step; eps-related fields are ignored. */
int b200_sampler_update(float* x, const float* denoised, const float* noise, float* old_denoised,
                        const b200_step_desc* d, b200_stream_t s);

/* KModel.apply_model tail for the model_function_wrapper plug point (backend/modules/k_model.py:45-46,
 * backend/modules/k_prediction.py:81-92): denoised[n,c,h,w] = x - eps*sigma_n from the channels-last UNet output. */
int b200_eps_to_denoised(const float* x, const void* eps, const float* sigma, float* out, int N, int C, int H, int W,
                         int ld_eps, int prediction, int eps_dtype, b200_stream_t s);

/* VAE post-decode: clamp((x+1)/2, 0, 1) NHWC (dtype) -> fp32 NHWC [B,H,W,3]
 * (backend/patcher/vae.py:142,147).  ldx = channel stride of x (the padded conv_out width). */
int b200_vae_postprocess(const void* x, float* out, size_t pixels, int ldx, int dtype, b200_stream_t s);

/* Tiled VAE decode (backend/patcher/vae.py:11-49 tiled_scale_multidim, :104-115 decode_tiled_): a decoded tile NHWC
 * [th, tw, ld >= 3] (dtype) is accumulated into acc [H, W, 4] fp32 = (sum of (tile + bias) * mask for r, g, b; sum of mask) at
 * (y0, x0), mask = linear ramps over the first / last `feather` rows and columns.  _resolve writes (or adds, `accumulate`)
 * acc.rgb / acc.mask into out [H, W, 3] fp32 and, on the last pass (`finalize`), scales and clamps to [0, 1]. */
int b200_tile_blend(const void* tile, float* acc, int H, int W, int y0, int x0, int th, int tw, int ld, float bias,
                    int feather, int dtype, b200_stream_t s);
int b200_tile_resolve(const float* acc, float* out, size_t pixels, int accumulate, float final_scale, int finalize,
                      b200_stream_t s);

/* fp32 images in [0, 1] -> uint8, the conversion modules/processing.py:1039-1040 does on the host after the D2H copy
 * (255 * x, astype(uint8): truncation); doing it on the device quarters the bytes that leave the GPU.  n % 4 == 0. */
int b200_images_to_u8(const float* x, unsigned char* out, size_t n, b200_stream_t s);

/* Control residual, in place: h NHWC [N, H, W, C] (dtype) += ctrl, with ctrl NCHW [ctrl_batch, C, H, W] or, when ctrl_nhwc,
 * NHWC [ctrl_batch, H, W, C] (16-byte aligned); dtype, or fp32 when ctrl_is_f32.  ctrl_batch is N or 1: a batch-1 residual
 * is added to every image, as torch's broadcasting `h += ctrl` does (backend/nn/unet.py:44-52 apply_control on the
 * input / middle / output-skip activations, T2I-Adapter residuals of one hint image; backend/nn/cnets/cldm.py:259-262
 * `h += guided_hint`).  C multiple of 8. */
int b200_add_control(void* h, const void* ctrl, int N, int C, int H, int W, int ctrl_batch, int ctrl_nhwc, int ctrl_is_f32,
                     int dtype, b200_stream_t s);
/* b200_add_control with an NCHW residual of batch N. */
int b200_add_nchw(void* h, const void* ctrl, int N, int C, int H, int W, int ctrl_is_f32, int dtype, b200_stream_t s);

/* VAE encode entry: pixels NHWC fp32 [pixels, 3] in [0, 1] -> [pixels, 8] in dtype, channels 0-2 = 2x - 1, 3-7 = 0
 * (backend/patcher/vae.py:177: `(2. * pixel_samples - 1.).to(vae_dtype)`; padded to 8 channels for the conv_in im2col). */
int b200_vae_preprocess(const float* x, void* out, size_t pixels, int dtype, b200_stream_t s);

/* DiagonalGaussianDistribution.sample() / .mode() (backend/nn/vae.py:16-32) on channels-last moments [N, H*W, ld]
 * (mean = channels [0, C), logvar = [C, 2C)):  out NCHW fp32 [N, C, H*W] = (mean + exp(0.5*clamp(logvar,-30,20))*noise)*scale;
 * noise (fp32, NCHW like out) may be NULL -> the mode.  scale = 1 for VAE.encode, the latent scaling factor for
 * process_in (backend/nn/vae.py:312-313). */
int b200_vae_posterior(const void* moments, const float* noise, float* out, int N, int C, int HW, int ld, float scale,
                       int dtype, b200_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * Flux (DiT) path — backend/nn/flux.py.  Token activations are [rows, C]; a joint activation holds, for every
 * sample, `seg_split` txt rows followed by img rows (`seg_period` rows per sample); segment 0 = txt, 1 = img.
 */

/* Modulated LayerNorm: y = (1 + scale_g[b]) * LayerNorm(x, no affine, eps) + shift_g[b]
 * (flux.py:211-212,232-233,255,259 DoubleStreamBlock; :287 SingleStreamBlock; :319 LastLayer).
 * shift/scale: row b of a [B, ld_mod] matrix (the Modulation output chunk).  shift1 = NULL: one parameter set. */
int b200_adaln(const void* x, void* y, int rows, int C, float eps, const void* shift0, const void* scale0,
               const void* shift1, const void* scale1, int ld_mod, int seg_period, int seg_split, int dtype,
               b200_stream_t s);

/* QKNorm + rotary embedding, in place on the q and k thirds of a fused QKV projection row [3, H, Dh] (row stride ld):
 * t = rms_norm(x, eps) * scale, then rotation of adjacent pairs by (cos, sin)[row % seg_period]
 * (flux.py:128-139 QKNorm; :15-18, :45-51 apply_rope).  cos_t / sin_t: fp32 [seg_period, Dh/2] (EmbedND, :75-89).
 * Dh = 128 only (else B200_EUNSUPPORTED). */
int b200_qk_norm_rope(void* qkv, int rows, int H, int Dh, int ld, const void* q_scale0, const void* k_scale0,
                      const void* q_scale1, const void* k_scale1, const float* cos_t, const float* sin_t, int seg_period,
                      int seg_split, float eps, int dtype, b200_stream_t s);

/* RMSNorm over the rows of [rows, C]: y = x * rsqrt(mean(x^2) + eps) * scale[C]  (backend/nn/flux.py:115-126 RMSNorm as the
 * Chroma Approximator applies it to hidden-wide rows, backend/nn/chroma.py:14-28).  Added after the round's GPU budget was
 * spent: compiled and reviewed, exercised so far only through the CPU emulation of the Chroma engine's launch sequence. */
int b200_rmsnorm_rows(const void* x, const void* scale, void* y, int rows, int C, float eps, int dtype, b200_stream_t s);

/* 2x2 patchify: x NCHW [B, C, H, W] (fp32 if in_is_f32 else dtype) -> tokens [B*(H/2)*(W/2), ld], feature c*4 + ph*2 + pw
 * (flux.py:398-399; even H, W only: the circular-pad branch returns B200_EUNSUPPORTED). */
int b200_flux_patchify(const void* x, void* tokens, int B, int C, int H, int W, int ld, int in_is_f32, int dtype,
                       b200_stream_t s);
/* inverse (flux.py:412): tokens -> NCHW fp32 [B, C, H, W] if out_nchw_f32 else NHWC [B, H, W, C] in dtype
 * (the layout b200_sampler_step reads). */
int b200_flux_unpatchify(const void* tokens, void* out, int B, int C, int H, int W, int ld, int out_nchw_f32, int dtype,
                         b200_stream_t s);

#ifdef __cplusplus
}
#endif
#endif /* B200FORGE_H */
