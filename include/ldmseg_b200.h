/*
 * ldmseg_b200.h -- C ABI of the B200-native LDMSeg sampler hot path (libldmseg_b200.so).
 *
 * The reference (weentiaan/Video-latent-diffusion-panoptic-segmentation) is pure Python and has no FFI; its
 * seam for this path is four Python call signatures (SURVEY.md section 8b).  The Python mirror classes under
 * video_latent_diffusion_panoptic_segmentation_b200/ldmseg/ keep those signatures and bind the entry points
 * below through ctypes.  Each entry point cites the reference code whose arithmetic it replaces.
 *
 * Conventions (all entry points):
 *   - raw device pointers + explicit shapes in POD structs; the CALLER owns all memory (no allocation inside);
 *   - asynchronous on the given CUDA stream, no device synchronisation, no global mutable state;
 *   - return 0 on success, negative ldm_status on error; ldm_last_error() returns a thread-local message;
 *   - activations are NHWC ("channels last"): [B, H, W, C]; bf16 = __nv_bfloat16 bit pattern; f32 = IEEE float;
 *   - built only for sm_100a: ldm_check_device() refuses any other device.
 */
#ifndef LDMSEG_B200_H_
#define LDMSEG_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* ldm_stream_t; /* cudaStream_t */

enum ldm_status {
  LDM_OK = 0,
  LDM_ERR_BAD_ARG = -1,
  LDM_ERR_BAD_SHAPE = -2,
  LDM_ERR_ALIGNMENT = -3,
  LDM_ERR_ARCH = -4,
  LDM_ERR_CUDA = -5,
  LDM_ERR_DRIVER = -6
};

int ldm_abi_version(void); /* 4 since the LayerNorm-fold fields of ldm_gemm_desc (3: splitk_ws; 2: qkv_part0 / ldm_attn_desc.kv_seq) */
const char* ldm_last_error(void);
/* 0 when the current device is compute capability 10.0 (B200); LDM_ERR_ARCH otherwise. */
int ldm_check_device(void);
/* number of kernels this library has launched in the calling process (bench.py "gpu_launches"). */
long long ldm_launch_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * Tensor-core contraction: plain GEMM (Linear / conv1x1) and implicit-GEMM conv3x3 (stride 1, pad 1).
 * Replaces: diffusers Conv2d/Linear inside ResnetBlock2D / Transformer2DModel / BasicTransformerBlock
 * (SURVEY.md App. A; call sites ldmseg/models/unet.py:357-431) and the seg-AE decoder convs
 * (ldmseg/models/vae.py:134-173).
 *   out[b,y,x,n] = epilogue( sum_{tap,c} A[b, y+dy(tap), x+dx(tap), c] * W[n, tap*(c1+c2) + c] )
 * A is the channel concatenation of source a1 (c1 channels) and optional a2 (c2 channels); c1, c2 % 64 == 0
 * for taps == 9 (any multiple of 8 for taps == 1 with a2 == NULL).
 * ---------------------------------------------------------------------------------------------------------- */
enum ldm_gemm_flags {
  LDM_GEMM_OUT_F32 = 1 << 0,   /* out is f32 [rows, N] (default bf16)                                         */
  LDM_GEMM_GEGLU = 1 << 1,     /* weights/bias pre-interleaved in blocks of 16 (value | gate);                 */
                               /* out[rows, N/2] = value * gelu_erf(gate)   (diffusers GEGLU)                  */
  LDM_GEMM_QKV_SPLIT = 1 << 2, /* N = 3*heads*head_dim; scatter to q/k [B*heads, seq, dpad], vt [B*heads, d, seq_pad] */
  LDM_GEMM_SILU = 1 << 3,      /* out = silu(acc + bias ...)                                                   */
  LDM_GEMM_OUT_NCHW_F32 = 1 << 5, /* out is planar f32 [B, n_store, H, W] (UNet conv_out, unet.py:431): only the first
                                     n_store (<= N) output channels are stored; weights may be zero-padded to N % 8 == 0 */
  LDM_GEMM_CONVT_LN_SILU = 1 << 4 /* N = 4*Cout: ConvTranspose2d(k2,s2) pixel-shuffle + LayerNorm2d + SiLU
                                     (vae.py:156-158,310-323); block_n must equal Cout (<= 256)               */
};

typedef struct ldm_gemm_desc {
  const void* a1;       /* bf16 NHWC [B,H,W,c1]                                                  */
  const void* a2;       /* bf16 NHWC [B,H,W,c2] or NULL                                          */
  const void* w;        /* bf16 [N, taps*(c1+c2)] (tap-major, channel-minor)                     */
  const float* bias;    /* f32 [N] or NULL                                                       */
  const float* rowbias; /* f32 [B, N] or NULL: per-image bias (time-embedding projection)         */
  const void* residual; /* bf16 [B*H*W, N] or NULL, added after bias                             */
  void* out;            /* bf16/f32 [B*H*W, N] (GEGLU: N/2 columns; CONVT: bf16 [B,2H,2W,N/4])   */
  void* q;              /* QKV_SPLIT outputs                                                     */
  void* k;
  void* vt;
  const float* ln_gamma; /* CONVT_LN_SILU: LayerNorm2d weight/bias f32 [Cout], eps                */
  const float* ln_beta;
  float ln_eps;
  int32_t B, H, W;      /* output (= input) spatial extents; a plain GEMM uses B=1,H=1,W=rows    */
  int32_t c1, c2;
  int32_t N;
  int32_t taps;         /* 1 or 9                                                                */
  int32_t block_n;      /* 0 = choose; else multiple of 32 in [32,256]                           */
  int32_t flags;
  int32_t heads, head_dim, dpad, seq, seq_pad; /* QKV_SPLIT geometry (seq = tokens per image)    */
  int32_t vt_rows;      /* rows per head of vt (ldm_attn_vt_rows(head_dim)); 0 = head_dim         */
  int32_t n_store;      /* OUT_NCHW_F32: channels stored (0 = N)                                 */
  int32_t qkv_part0;    /* QKV_SPLIT: the N = nparts*heads*head_dim columns hold parts qkv_part0 .. of (q, k, v): 0 with
                           N = 3C is the fused self-attention projection; 0 with N = C writes q only (cross-attention
                           to_q); 1 with N = 2C writes k and vt from the context rows (to_k | to_v). Buffers of parts
                           that are not written may be NULL.                                                    */
  const void* identity; /* optional bf16 [256,256] identity matrix (caller-owned, may be shared by all calls). When
                           given, a short-K pointwise GEMM adds `residual` on the tensor core: the residual rows
                           are streamed by TMA as extra K blocks against identity weights instead of being read
                           row by row in the epilogue. NULL: always the epilogue path.                    */
  void* splitk_ws;      /* optional split-K workspace (caller-owned device memory, 16-byte aligned, no initial
                           contents needed, may be shared by all calls of one stream). When given, launches with
                           few tiles and a long K (small M: the 6x20 level, or one frame per GPU) cut every tile's K
                           range into work items that run on different SMs and leave fp32 partial tiles here; a
                           second small launch adds them in a fixed order (bit-reproducible run to run) and applies
                           the epilogue. NULL: never split.                                                    */
  int64_t splitk_ws_bytes;
  /* LayerNorm folded into the GEMMs around it (diffusers BasicTransformerBlock.norm1 / norm2 / norm3 in front of
     to_q|k|v and ff.net.0, SURVEY.md App. A) -- no normalisation pass and no normalised copy of the activations:
       LN(x) W^T + b = rstd_m (x (gamma o W)^T - mean_m g) + (b + W beta),   g[n] = sum_c (gamma o W)[n, c].
     The GEMM that WRITES x (plain bf16 epilogue) also writes, per 32-column chunk and row, the sum and the sum of
     squares of its bf16 outputs into row_stats_out (f32 [ceil(N / 32), rows, 2]: part-major, so that a warp's 32 rows
     are 256 contiguous bytes on both sides). The GEMM that READS x (QKV_SPLIT or GEGLU, pointwise) runs on the raw x
     with w = gamma o W, bias = b + W beta, ln_colsum = g, and applies the row's mean / rstd in its epilogue from
     ln_stats (the producer's row_stats_out; ln_parts = ceil(c1 / 32) partials per row, added in index order:
     bit-reproducible).                                                                                         */
  void* row_stats_out;
  const void* ln_stats;
  const float* ln_colsum;
  float ln_fold_eps;
  int32_t ln_parts;
  /* Strided and sub-pixel convolutions without a gather pass: the tensor maps carry element strides of 2 in the pixel
     dimensions, so the TMA unit reads / writes every other pixel (tools/microbench/tma_stride_test.cu).
     a_stride = 2 (taps = 9): Conv2d(3x3, stride 2) -- diffusers Downsample2D (SURVEY.md App. A). B, H, W are the OUTPUT
       extents, a1 (and a2) are [B, a_H, a_W, c]; output pixel (y, x) reads input (2y + ky - a_pad, 2x + kx - a_pad), zero
       outside (a_pad = 1: padding 1; a_pad = 0: F.pad(x, (0, 1, 0, 1)) + padding 0). a_stride = 0 / 1: dense.
     up2 = 1 (taps = 4, N = 4 * cout): F.interpolate(scale 2, nearest) followed by Conv2d(3x3, padding 1) -- diffusers
       Upsample2D -- as four 2x2 convolutions of the LOW-resolution input, one per output parity class
       cls = 2 * (row & 1) + (col & 1): 4/9 of the multiply-adds and no up-sampled copy. w rows [cls * cout, (cls + 1) *
       cout) hold that class's kernel, tap (i, j) = 2 i + j reads input (y + i - 1 + (cls >> 1), x + j - 1 + (cls & 1));
       bias is [4 * cout] (the conv bias four times). B, H, W are the INPUT extents, out is the dense
       [B, out_H, out_W, cout] tensor with out_H = 2H, out_W = 2W exactly. (The nearest resize to an ODD size that
       diffusers does for a skip connection -- 20 -> 39 columns -- keeps the gather pass: its last column sees the zero
       padding where the collapsed kernel would see a pixel.) Plain bf16 epilogue only (bias, SiLU). */
  int32_t a_stride, a_pad, a_H, a_W;
  int32_t up2, out_H, out_W;
} ldm_gemm_desc;

int ldm_gemm_bf16(const ldm_gemm_desc* d, ldm_stream_t stream);
/* The tiling the calling thread's last ldm_gemm_bf16 launch chose (tests and profiling tools): N tile width, 1 for the
 * CTA-pair kernel, work items per tile (1 = no split-K). Any pointer may be NULL. */
int ldm_gemm_last_config(int32_t* block_n, int32_t* pair, int32_t* split_k);

/* ------------------------------------------------------------------------------------------------------------
 * Fused flash-style self-attention, softmax(Q K^T * scale) V, per (image, head).
 * Replaces: diffusers Attention / AttnProcessor2_0 (F.scaled_dot_product_attention) in BasicTransformerBlock.attn1
 * (SURVEY.md App. A; cross-attention removed by ldmseg/models/unet.py:83-105).
 *   q, k : bf16 [B*heads, seq, dpad]   (dpad = 64*ceil(d/64), columns >= d are zero; k has kv_seq rows when kv_seq > 0)
 *   vt   : bf16 [B*heads, vt_rows, seq_pad]  (V transposed; seq_pad % 8 == 0; vt_rows = ldm_attn_vt_rows(d) =
 *          16*ceil(d/16); when d % 16 != 0 row d of every head must hold 1.0 for the valid keys and rows > d zero:
 *          the P.V MMA then also yields the softmax row sums)
 *   out  : bf16 [B*seq, heads*d]
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct ldm_attn_desc {
  const void* q;
  const void* k;
  const void* vt;
  void* out;
  int32_t B, heads, seq, head_dim, dpad, seq_pad, vt_rows;
  float scale;    /* head_dim^-0.5 */
  int32_t kv_seq; /* keys / values per (image, head); 0 = seq (self-attention). Cross-attention (BasicTransformerBlock
                     .attn2 against encoder_hidden_states, unet.py:319-323 / SURVEY 8f rank 4): q [B*heads, seq, dpad],
                     k [B*heads, kv_seq, dpad], vt [B*heads, vt_rows, seq_pad] with seq_pad >= kv_seq.               */
} ldm_attn_desc;

int ldm_attn_vt_rows(int head_dim);

int ldm_flash_attn_fwd(const ldm_attn_desc* d, ldm_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * GroupNorm (+ optional SiLU) over the channel concatenation of x1 (c1) and x2 (c2), NHWC bf16.
 * Replaces: torch.nn.GroupNorm + SiLU in ResnetBlock2D.norm1/norm2, Transformer2DModel.norm,
 * UNet.conv_norm_out (unet.py:428-430), seg-AE decoder GroupNorm (vae.py:163-164).
 * stats: caller-provided scratch of ldm_groupnorm_scratch_bytes(B, groups) bytes (per-chunk partial moments; the
 * reduction order is fixed, so results are bit-reproducible run to run) followed by the barrier counters of the
 * one-launch path. The scratch must be ZERO before its first use; every call leaves the counters zero. One scratch
 * must not be shared by GroupNorms running concurrently on different streams.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct ldm_groupnorm_desc {
  const void* x1;
  const void* x2; /* or NULL */
  const float* gamma;
  const float* beta;
  void* out;     /* bf16 [B, HW, c1+c2] */
  void* stats;   /* scratch, ldm_groupnorm_scratch_bytes(B, groups) bytes */
  int32_t B, HW, c1, c2, groups;
  float eps;
  int32_t silu;
} ldm_groupnorm_desc;

size_t ldm_groupnorm_scratch_bytes(int32_t B, int32_t groups);
int ldm_groupnorm_silu(const ldm_groupnorm_desc* d, ldm_stream_t stream);

/* LayerNorm over the last dim of bf16 [rows, C] (BasicTransformerBlock.norm1 / norm3). */
int ldm_layernorm(const void* x, const float* gamma, const float* beta, void* out, int32_t rows, int32_t C,
                  float eps, ldm_stream_t stream);

/* Timestep embedding pieces (unet.py:301-307 + diffusers Timesteps / TimestepEmbedding; the timestep is one
 * 0-dim tensor expanded over the batch, unet.py:302-303, so the embedding is a single vector).
 *   ldm_timestep_sinusoid: out[0:half] = cos(t*freqs), out[half:2*half] = sin(t*freqs)  (flip_sin_to_cos, shift 0),
 *   t = timesteps[*t_index] (int64 device array; t_index on device so a captured CUDA graph replays every step).
 *   ldm_gemv_bf16: out[n] = act(bias[n] + bias2[n] + sum_k w[n,k]*x[k]); w bf16 [N,K]; x,out f32; act = SiLU if
 *   silu_out. Used for linear_1 (+SiLU), linear_2 (+SiLU, the resnets' nonlinearity(temb)) and for ALL
 *   time_emb_proj layers in one launch (bias2 = the conv1 biases, so the result is conv1's epilogue bias). */
int ldm_timestep_sinusoid(const int64_t* timesteps, const int32_t* t_index, const float* freqs, float* out,
                          int32_t half, ldm_stream_t stream);
int ldm_gemv_bf16(const void* w, const float* bias, const float* bias2, const float* x, float* out, int32_t N,
                  int32_t K, int32_t silu_out, ldm_stream_t stream);

/* 3x3 conv (pad 1) with few input channels, fused with the latent concat + cast + scale:
 *   conv_in of the UNet: cat([x_t, rgb_latents(, condition)], 1) (trainers_ldm_cond.py:1131-1141) -> unet.py:357
 *   seg-AE decoder[0]  : z * (1/scaling_factor) (trainers_ldm_cond.py:423) -> vae.py:134
 * s0..s2: f32 NCHW [B,cps,h,w] sources (nsrc of them), scaled by `scale`; w f32 [nsrc*cps, 3, 3, cout] (the reference's
 * [cout, cin, 3, 3] permuted so that the output channel is innermost: coalesced weight reads); out bf16 NHWC [B,h,w,cout]. */
int ldm_conv3x3_small_cin(const float* s0, const float* s1, const float* s2, int32_t nsrc, int32_t cps, float scale,
                          const float* w, const float* bias, void* out, int32_t B, int32_t h, int32_t wd,
                          int32_t cout, ldm_stream_t stream);
/* the same with an optional SiLU on the result: seg-AE encoder[0..1] (Conv2d + SiLU on the bit planes, vae.py:191-195) */
int ldm_conv3x3_small_cin_act(const float* s0, const float* s1, const float* s2, int32_t nsrc, int32_t cps, float scale,
                              const float* w, const float* bias, void* out, int32_t B, int32_t h, int32_t wd,
                              int32_t cout, int32_t silu, ldm_stream_t stream);

/* the same with an affine map of the input samples, v = x * scale + shift (two roundings): conv_in of the RGB VAE encoder
 * fused with `images = 2. * images - 1.` (trainers_ldm_cond.py:372 -> diffusers Encoder.conv_in; SURVEY 8f rank 1).
 * The conv's zero padding is applied after the map, as in the reference. */
int ldm_conv3x3_small_cin_affine(const float* s0, const float* s1, const float* s2, int32_t nsrc, int32_t cps,
                                 float scale, float shift, const float* w, const float* bias, void* out, int32_t B,
                                 int32_t h, int32_t wd, int32_t cout, int32_t silu, ldm_stream_t stream);

/* conv_out: bf16 NHWC [B,h,w,Cin] (already GroupNorm+SiLU'ed) -> conv3x3 -> f32 NCHW [B,Cout,h,w] (Cout <= 8).
 * w f32 [Cout,Cin,3,3] (unet.py:431). */
int ldm_conv_out(const void* x, const float* w, const float* bias, float* out, int32_t B, int32_t h, int32_t wd,
                 int32_t cin, int32_t cout, ldm_stream_t stream);

/* DDIM update (ddim_scheduler.py:218-269, epsilon prediction, no clipping), fp32, bit-exact with the reference's
 * op order:  x0 = (x - sqrt(1-a_t)*eps) / sqrt(a_t);  prev = sqrt(a_prev)*x0 + sqrt(1-a_prev)*eps.
 * coef: device f32 [T,4] = {sqrt(1-a_t), sqrt(a_t), sqrt(a_prev), sqrt(1-a_prev)} rows selected by *t_index.
 * prev_sample / pred_x0 may be NULL.  */
int ldm_ddim_step(const float* eps, const float* sample, const float* coef, const int32_t* t_index,
                  float* prev_sample, float* pred_x0, int64_t n, ldm_stream_t stream);

/* The same with classifier-free guidance in front (trainers_ldm_cond.py:1147-1149, `noise_pred_uncond + guidance_scale *
 * (noise_pred_text - noise_pred_uncond)`, fp32, the reference's three roundings): eps_uncond / eps_text are the two
 * halves of the doubled batch's UNet output; eps_text == NULL is ldm_ddim_step. */
int ldm_ddim_step_cfg(const float* eps_uncond, const float* eps_text, float guidance_scale, const float* sample,
                      const float* coef, const int32_t* t_index, float* prev_sample, float* pred_x0, int64_t n,
                      ldm_stream_t stream);

/* The same with the scheduler's clip_sample / use_clipped_model_output (ddim_scheduler.py:253-261): clip_sample_range
 * > 0 clamps pred_original_sample to [-range, range] before prev_sample is formed (0: no clipping); with
 * use_clipped_model_output the noise is re-derived from the clamped x0, `(sample - sqrt(a_t) * x0) / sqrt(1 - a_t)`.
 * The reference's constructor default is clip_sample=True; base.yaml:55 turns it off for this path. */
int ldm_ddim_step_clip(const float* eps_uncond, const float* eps_text, float guidance_scale, const float* sample,
                       const float* coef, const int32_t* t_index, float* prev_sample, float* pred_x0, int64_t n,
                       float clip_sample_range, int32_t use_clipped_model_output, ldm_stream_t stream);

/* DPM-Solver++ multistep update (algorithm_type "dpmsolver++", solver_type "midpoint", epsilon prediction, solver
 * order 1 or 2), fp32, bit-exact with the same formulas in torch eager on the CPU (round-to-nearest, this op order):
 *   x0   = (sample - sig_i * eps) / alpha_i
 *   prev = A * sample - Bc * x0                                  (order 1)
 *   prev = (A * sample - Bc * x0) - hb * (c * (x0 - x0_prev))    (order 2)
 * with A = sig_{i+1} / sig_i, Bc = alpha_{i+1} * (exp(-h) - 1), h = lam_{i+1} - lam_i, c = 1 / r0,
 * r0 = (lam_i - lam_{i-1}) / h, hb = 0.5 * Bc, and per sigma alpha = 1 / sqrt(sigma^2 + 1), sig = sigma * alpha,
 * lam = log(alpha) - log(sig). The host builds these scalars: coef is a device f32 [steps, 8] table, row i =
 * {sig_i, alpha_i, A, Bc, c, hb, order (1.0 or 2.0), 0}, selected by the DEVICE int32 *step_index (no host sync).
 * eps_text != NULL: eps = eps_uncond + guidance_scale * (eps_text - eps_uncond) first, as ldm_ddim_step_cfg.
 * x0 is written to x0_prev in place (read first when order == 2); prev_sample may alias sample. No argument but
 * eps_text may be NULL. */
int ldm_dpmpp_step(const float* eps_uncond, const float* eps_text, float guidance_scale, const float* sample,
                   const float* coef, const int32_t* step_index, float* prev_sample, float* x0_prev, int64_t n,
                   ldm_stream_t stream);

/* UniPC multistep update (predict_x0, solver_type "bh2", epsilon prediction, solver order 1, 2 or 3): the corrector
 * UniC of the previous step's result and the predictor UniP to the next sigma in one launch, fp32, bit-exact with the
 * same formulas in torch eager on the CPU (round-to-nearest, this op order; oracle/unipc_oracle.py states it in full):
 *   m    = (sample - sig_i * eps) / alpha_i
 *   S    = rho_m * (m - m1)                                                           (corrector order 1)
 *   S    = ((rho_1 * ((m2 - m1) / r_1)) [+ rho_2 * ((m3 - m1) / r_2)]) + rho_m * (m - m1)     (order 2 [3])
 *   xc   = (A * last - Phi * m1) - Bh * S                          (xc = sample when the corrector is off)
 *   prev = A' * xc - Phi' * m                                                         (predictor order 1)
 *   prev = (A' * xc - Phi' * m) - Bh' * ((rho'_1 * ((m1 - m) / r'_1)) [+ rho'_2 * ((m2 - m) / r'_2)])  (order 2 [3])
 *   last <- xc;  m3 <- m2, m2 <- m1, m1 <- m
 * Per sigma alpha = 1 / sqrt(sigma^2 + 1), sig = sigma * alpha, lam = log(alpha) - log(sig); an update from index a to
 * t at order q has h = lam_t - lam_a, phi = B = expm1(-h), A = sig_t / sig_a, Phi = alpha_t * phi, Bh = alpha_t * B,
 * r_k = (lam_{a-k} - lam_a) / h, and rho from the UniPC linear system (0.5 at predictor order 2 and corrector order 1).
 * The corrector of step i updates a = i - 1 -> t = i; the predictor a = i -> t = i + 1. The host builds the scalars:
 * coef is a device f32 [steps, 20] table, row i = {sig_i, alpha_i, p, q, A', Phi', Bh', r'_1, r'_2, rho'_1, rho'_2,
 * A, Phi, Bh, r_1, r_2, rho_1, rho_2, rho_m, 0} with p the predictor order (1..3) and q the corrector order (0: off),
 * selected by the DEVICE int32 *step_index (no host sync). eps_text != NULL: eps = eps_uncond + guidance_scale *
 * (eps_text - eps_uncond) first, as ldm_ddim_step_cfg. m1 .. m_order are the previous x0 predictions (m1 the newest),
 * updated in place; m_k with k > solver_order is not touched and may be NULL. prev_sample may alias sample; last,
 * m1, m2, m3 alias nothing. Every element is read before it is written by the same thread. */
int ldm_unipc_step(const float* eps_uncond, const float* eps_text, float guidance_scale, const float* sample,
                   const float* coef, const int32_t* step_index, float* prev_sample, float* last, float* m1, float* m2,
                   float* m3, int32_t solver_order, int64_t n, ldm_stream_t stream);

/* Per-image timesteps (the streaming sampler: every image of a batch at its own step of its own trajectory). Each
 * output element takes exactly the arithmetic of the single-timestep entry point above it, so image b's slice is bit
 * for bit what that entry point gives for image b's timestep or row.
 *   ldm_timestep_sinusoid_rows: out [B, 2*half], row b from t = timesteps[b] (int64 device [B]).
 *   ldm_gemv_bf16_rows: x f32 [B, K] -> out[b][n] = act(bias[n] + bias2[n] + w[n,:] . x[b]), as ldm_gemv_bf16. With
 *     seg_offs == NULL out is [B, N]; otherwise seg_offs is a device int32 [nseg + 1] of ascending column offsets from
 *     0 to N, and out is segment-major: segment s (columns [o_s, o_{s+1})) is a contiguous [B, o_{s+1} - o_s] block at
 *     float offset o_s * B -- the rowbias (ldm_gemm_desc.rowbias) of every resnet's conv1 from one launch.
 *   ldm_ddim_step_rows / ldm_dpmpp_step_rows / ldm_unipc_step_rows: the updates of ldm_ddim_step / ldm_dpmpp_step /
 *     ldm_unipc_step without guidance, element i reading coefficient row rows[i / elems_per_image] (device int32, one
 *     entry per image; DDIM: the timestep value, as *t_index; DPM-Solver++ and UniPC: the step index).
 *     elems_per_image is a positive multiple of 4; n need not be a multiple of it (the last image may be partial). */
int ldm_timestep_sinusoid_rows(const int64_t* timesteps, const float* freqs, float* out, int32_t half, int32_t B,
                               ldm_stream_t stream);
int ldm_gemv_bf16_rows(const void* w, const float* bias, const float* bias2, const float* x, float* out, int32_t N,
                       int32_t K, int32_t B, const int32_t* seg_offs, int32_t nseg, int32_t silu_out,
                       ldm_stream_t stream);
int ldm_ddim_step_rows(const float* eps, const float* sample, const float* coef, const int32_t* rows,
                       float* prev_sample, float* pred_x0, int64_t n, int64_t elems_per_image, ldm_stream_t stream);
int ldm_dpmpp_step_rows(const float* eps, const float* sample, const float* coef, const int32_t* rows,
                        float* prev_sample, float* x0_prev, int64_t n, int64_t elems_per_image, ldm_stream_t stream);
int ldm_unipc_step_rows(const float* eps, const float* sample, const float* coef, const int32_t* rows,
                        float* prev_sample, float* last, float* m1, float* m2, float* m3, int32_t solver_order,
                        int64_t n, int64_t elems_per_image, ldm_stream_t stream);

/* Layout helpers (NHWC bf16). */
int ldm_upsample_nearest(const void* x, void* out, int32_t B, int32_t h, int32_t w, int32_t C, int32_t oh,
                         int32_t ow, ldm_stream_t stream); /* F.interpolate(mode="nearest") */
int ldm_im2col3x3_s2(const void* x, void* out, int32_t B, int32_t h, int32_t w, int32_t C, int32_t oh, int32_t ow,
                     ldm_stream_t stream); /* Downsample2D conv (stride 2, pad 1) -> [B*oh*ow, 9*C] */

/* im2col of a 3x3 stride-2 conv with pad_lo (0 or 1) zero rows / columns in front of the image and one after it:
 * pad_lo = 1 is ldm_im2col3x3_s2; pad_lo = 0 is diffusers Downsample2D(padding=0) of the RGB VAE encoder
 * (F.pad(x, (0, 1, 0, 1)) then Conv2d(stride 2, padding 0)). out [B*oh*ow, 9*C], oh = (h + pad_lo - 2) / 2 + 1. */
int ldm_im2col3x3_s2_pad(const void* x, void* out, int32_t B, int32_t h, int32_t w, int32_t C, int32_t oh, int32_t ow,
                         int32_t pad_lo, ldm_stream_t stream);

/* Row softmax of an unfused attention: p[r, c] = softmax_c(scale * s[r, c]) for c < cols, fp32 math, bf16 result.
 * s f32 [rows, ld_s]; p bf16 [rows, ld_p] (columns >= cols are not written). Replaces the softmax of diffusers
 * Attention in the RGB VAE mid block (one head of 512 channels: too wide for the fused flash kernels, whose O
 * accumulator lives in TMEM), between two ldm_gemm_bf16 calls (Q K^T with LDM_GEMM_OUT_F32, then P V). */
int ldm_softmax_rows(const float* s, void* p, int64_t rows, int32_t cols, int64_t ld_s, int64_t ld_p, float scale,
                     ldm_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Integer tail.
 * ---------------------------------------------------------------------------------------------------------- */
/* argmax + softmax-max threshold (trainers_ldm_cond.py:1287-1295) on NHWC f32 logits [B,h,w,C] upsampled
 * bilinearly (align_corners=False) by `up` (1 or 2) on the fly (vae.py:271 / trainers_ldm_cond.py:1264-1269).
 * ids: int32 [B, up*h, up*w] (argmax, or ignore_label where max softmax prob < mask_th)
 * Also accumulates, per image, count[c] = #pixels with id == c and over[c] = #pixels with sigmoid(logit_c) >= mask_th
 * (the two sums of the merge, :1307-1315).  counts: int32 [B, 2, C], zeroed by the call. */
int ldm_logits_to_ids(const float* logits, int32_t* ids, int32_t* counts, int32_t B, int32_t h, int32_t w,
                      int32_t C, int32_t up, float mask_th, int32_t ignore_label, ldm_stream_t stream);
/* Materialising variant of the bilinear x`up` resize: NHWC f32 [B,h,w,C] -> NCHW f32 [B,C,up*h,up*w]. */
int ldm_bilinear_up_nchw(const float* logits, float* out, int32_t B, int32_t h, int32_t w, int32_t C, int32_t up,
                         ldm_stream_t stream);
/* General bilinear resize, F.interpolate(size=(oh,ow), mode="bilinear", align_corners=False), of the crop window
 * [y0, y0+ch) x [x0, x0+cw) of NHWC f32 [B,h,w,C] (C % 4 == 0) into NHWC f32 [B,oh,ow,C]: the resize to the RGB size
 * (trainers_ldm_cond.py:1264-1269), crop_padding (:1175-1181,1276) and the resize to meta.im_size (:1279-1284). */
int ldm_resize_bilinear_nhwc(const float* in, float* out, int32_t B, int32_t h, int32_t w, int32_t C, int32_t y0,
                             int32_t x0, int32_t ch, int32_t cw, int32_t oh, int32_t ow, ldm_stream_t stream);
/* The same arithmetic on planar f32 maps [P, h, w] -> [P, oh, ow] (NCHW tensors with P = B*C): the image / latent
 * resizes of encode_inputs (trainers_ldm_cond.py:368-369,382-393). */
int ldm_resize_bilinear_planar(const float* in, float* out, int32_t P, int32_t h, int32_t w, int32_t oh, int32_t ow,
                               ldm_stream_t stream);
/* Panoptic merge (trainers_ldm_cond.py:1303-1325): for every class c, keep[c] = count[c] >= count_th and
 * c != ignore_label and not (count[c] / over[c] < overlap_th) (float64 ratio as numpy computes it); then
 * cleaned[i] = keep[ids[i]] ? ids[i] : -1.  counts is the [B,2,C] array written by ldm_logits_to_ids. */
int ldm_segment_filter(const int32_t* ids, const int32_t* counts, int32_t* cleaned, int32_t B, int64_t hw,
                       int32_t C, int32_t count_th, double overlap_th, int32_t ignore_label, ldm_stream_t stream);
/* decode_bitmap (ldmseg/data/cityscapes.py:263-270, kitti.py:299-306; coco.py:385-391 has no ==31 line):
 * x f32 [B,n,H,W] -> int32 [B,H,W], id = sum_i (x_i > 0) << i; id == 31 -> 0 when quirk31. n <= 24. */
int ldm_decode_bitmap(const float* x, int32_t* ids, int32_t B, int32_t nbits, int64_t hw, int32_t quirk31,
                      ldm_stream_t stream);
/* encode_bitmap (cityscapes.py:256-261): ids int32 [B,H,W] -> f32 [B,n,H,W]; pixels == ignore_label -> fill. */
int ldm_encode_bitmap(const int32_t* ids, float* x, int32_t B, int32_t nbits, int64_t hw, int32_t ignore_label,
                      float fill, ldm_stream_t stream);
/* 4-connected component labelling with scipy.ndimage.label numbering (components numbered in raster order of
 * their first pixel) of the binary mask (sem == target), per image: labels int32 [B,H,W] (0 = background),
 * ncomp int32 [B]. scratch: ldm_ccl_scratch_bytes(B,H,W) bytes. (cityscapes_pap_eval.py:76-84,96-101) */
size_t ldm_ccl_scratch_bytes(int32_t B, int32_t H, int32_t W);
int ldm_ccl_label4(const int32_t* sem, int32_t target, int32_t* labels, int32_t* ncomp, int32_t* scratch, int32_t B,
                   int32_t H, int32_t W, ldm_stream_t stream);
/* Joint histogram of id pairs (a[i], b[i]) -- the np.unique(gt*offset + pred, return_counts=True) of vpq_eval
 * (eval/eval_dvpq.py:39-49) and the mask intersections of CityscapesPanopticEvaluator.add_image
 * (cityscapes_pap_eval.py:113-146) -- as an open-addressing hash table in caller memory:
 * keys[slot] = ((uint64)(uint32)a << 32) | (uint32)b, or 0x8000000000000000 when empty; counts[slot] = pixels.
 * capacity: power of two >= 64; *overflow is set to 1 if the table filled up. The call clears the table first. */
int ldm_joint_hist(const int32_t* a, const int32_t* b, int64_t n, unsigned long long* keys, int32_t* counts,
                   int32_t capacity, int32_t* overflow, ldm_stream_t stream);

/* Batched front half of CityscapesPanopticEvaluator.add_image (cityscapes_pap_eval.py:66-110) for B images in ONE
 * sequence of launches: pred_seg int32 [B,H,W] (-1 = void -> ignore_label), gt_sem int32 [B,H,W] ->
 *   gt_pan  : thing pixels -> sem * max_ins + component (4-connected, scipy numbering per class), ignore_label -> -1
 *   pred_pan: ignore_label -> 0, thing pixels -> label * max_ins + component, then -1 where gt or pred is ignore_label
 * thing_slots: int8 [2][256] in device memory, row 0 for the prediction, row 1 for the ground truth: slot index
 * (0 .. n_things-1) of a thing label, -1 otherwise (labels outside [0, 256) are never things). n_things <= 32.
 * scratch: ldm_city_pan_scratch_bytes(B,H,W,n_things) bytes. */
size_t ldm_city_pan_scratch_bytes(int32_t B, int32_t H, int32_t W, int32_t n_things);
int ldm_city_pan_maps(const int32_t* pred_seg, const int32_t* gt_sem, int32_t* pred_pan, int32_t* gt_pan,
                      const int8_t* thing_slots, int32_t n_things, int32_t ignore_label, int32_t max_ins,
                      int32_t* scratch, int32_t B, int32_t H, int32_t W, ldm_stream_t stream);
/* n_tables joint histograms in one launch (all images of a batch, or all sliding windows of eval/eval_dvpq.py:153-184):
 * table t counts the pairs (a[t*stride + j], b[t*stride + j]), j < n_per_table (windows of k frames over frame-major
 * maps: stride = H*W, n_per_table = k*H*W), into keys/counts[t*capacity ...] laid out as in ldm_joint_hist;
 * overflow[t] is set when table t filled up. */
int ldm_joint_hist_batch(const int32_t* a, const int32_t* b, int64_t n_per_table, int64_t stride, int32_t n_tables,
                         unsigned long long* keys, int32_t* counts, int32_t capacity, int32_t* overflow,
                         ldm_stream_t stream);

/* id-map helpers of CityscapesPanopticEvaluator.add_image (cityscapes_pap_eval.py:66-110):
 *   ldm_pan_insert: pan[i] = target*max_ins + labels[i] where sem[i] == target   (thing -> sem*max_ins + instance)
 *   ldm_id_mask   : x[i] = fill where a[i] == va or (b != NULL and b[i] == vb)     (ignore regions -> -1)        */
int ldm_pan_insert(const int32_t* sem, const int32_t* labels, int32_t target, int32_t max_ins, int32_t* pan,
                   int64_t n, ldm_stream_t stream);
int ldm_id_mask(int32_t* x, const int32_t* a, int32_t va, const int32_t* b, int32_t vb, int32_t fill, int64_t n,
                ldm_stream_t stream);

/* pan[i] = cat[i] * max_ins + ins[i]: the panoptic id of eval/eval_dvpq.py:108-121 (`pan = cat * max_ins + ins` for the
 * prediction and the ground truth of a window) on device-resident id maps. Values must fit int32 (cat <= 255,
 * max_ins = 2^20 in the reference). */
int ldm_pan_combine(const int32_t* cat, const int32_t* ins, int32_t max_ins, int32_t* pan, int64_t n,
                    ldm_stream_t stream);

/* Depth-aware masking of a DVPQ window (eval/eval_dvpq.py:123-145: `depth_mask = depth_gts > 0`, abs-rel error,
 * `pred_in_depth_mask[ignored_pred_mask] = 19 * max_ins`). For every pixel of the [H, Wd] depth maps with depth_gt > 0:
 *   rel = |depth_pred - depth_gt| / depth_gt in float64, with numpy's arithmetic of the PNG sample type -- elem_bits 8 / 16:
 *   unsigned subtraction modulo 2^bits (np.abs is then the identity), 32: signed int32; pred[y, x] = fill where rel > thres.
 * pred: int32 [H, pred_stride] (the window's id map, pred_stride >= Wd: only its first Wd columns are touched).
 * depth_pred / depth_gt: the samples widened to int32 by the caller. partial_sum / partial_cnt [nblocks]: per-CTA sum of
 * rel and number of valid pixels, added by the caller in index order (abs_rel = sum / count; the reference's np.mean is a
 * pairwise sum -- agreement to ~1e-15 relative, not bitwise; the masking itself is exact). */
int ldm_depth_mask_pred(int32_t* pred, int32_t pred_stride, const int32_t* depth_pred, const int32_t* depth_gt, int32_t H,
                        int32_t Wd, int32_t elem_bits, double thres, int32_t fill, double* partial_sum,
                        unsigned long long* partial_cnt, int32_t nblocks, ldm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LDMSEG_B200_H_ */
