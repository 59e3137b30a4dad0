/* tango_b200.h — C ABI of libtango_b200.so (B200 / sm_100a kernels for the Tango inference hot path).
 *
 * The reference (declare-lab/tango) is pure Python on stock PyTorch ops: it has no FFI layer of its own.
 * Each entry point below therefore replaces a *library op call site* of the reference hot path (SURVEY.md §2.1,
 * §8a); the file:line cited is the reference code whose arithmetic the kernel reproduces. The Python host
 * (tango_b200/*.py) binds these with ctypes and mirrors the reference's module interface on top.
 *
 * Conventions: plain pointers (device memory unless stated), explicit sizes/strides, `stream` is a
 * cudaStream_t passed as void*. Every function returns 0 on success and a negative TNG_E* code on error;
 * tng_last_error() gives a message. Nothing is allocated or retained by the library. No CPU fallback exists:
 * without a CUDA device every compute entry point fails with TNG_ECUDA.
 *
 * Activations are channels-last ("NHWC", rows = pixels / tokens / time positions, channels contiguous).
 */
#ifndef TANGO_B200_H
#define TANGO_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define TNG_OK 0
#define TNG_EINVAL (-1) /* bad argument / unsupported shape */
#define TNG_ECUDA (-2)  /* CUDA runtime / driver error (incl. no device) */

#define TNG_ACT_NONE 0
#define TNG_ACT_SILU 1
#define TNG_ACT_LRELU 2 /* slope = act_param */
#define TNG_ACT_GEGLU 3 /* out[j] = acc[j] * gelu_erf(acc[j + BN/2]) within each N tile (weights pre-interleaved) */
#define TNG_ACT_GEGLU_TANH 4 /* same pairing with the tanh-form GELU ("gelu_new": T5 v1.1 gated feed-forward) */

#define TNG_DT_F32 0
#define TNG_DT_BF16 1

#define TNG_MAX_AVIEWS 4
#define TNG_MAX_KGROUPS 40

int tng_version(void);
const char* tng_last_error(void);
/* Number of kernels this library has launched since load (bench.py's `gpu_launches`). */
uint64_t tng_launch_count(void);

/* ---------------------------------------------------------------------------------------------------------
 * tng_conv_gemm — tcgen05 implicit-GEMM convolution / linear layer (one persistent warp-specialised kernel).
 * Replaces: nn.Conv2d in ResnetBlock2D / Down/Upsample2D / conv_in / conv_out
 *             (mustango/diffusers/src/diffusers/models/resnet.py:570,590,157,206; unet_2d_condition.py:626,702),
 *           nn.Linear in Transformer2DModel / Attention / GEGLU FeedForward
 *             (transformer_2d.py:255-263,282-290; attention_processor.py:500-540; attention.py:384-387,431-433),
 *           VAE decoder Conv2d (audioldm/variational_autoencoder/modules.py:155-175,658-680),
 *           HiFi-GAN Conv1d / ConvTranspose1d-as-GEMM (audioldm/hifigan/models.py:96-103,124-135,149-165).
 *
 * D[row, n] = sum_g sum_{k<64*nkb_g} A_{view_g}[pixel(row) + (dw_g, dh_g), a_c0_g + k] * B[n, b_k0_g + k]
 *   rows enumerate the output pixel grid (img, h, w), w fastest; A views are bf16 channels-last 4-D tensors
 *   read through TMA with zero fill outside [0,W)x[0,H)x[0,NB) (this is the conv zero padding);
 *   B is a bf16 row-major [Ncols, Ktot] matrix (K contiguous).
 * Epilogue: x = (acc + bias[n] + rowvec[img, n] + res[row, n]) * alpha (+ out_f32[row, n] if accumulate);
 *   out_f32[row, n] = x (optional); out_bf16[row, n] = act(x) (optional; with `split_off > 0` the bf16
 *   rounding residual is also written at column n + split_off — "hi/lo" operand for the 3-term split GEMM).
 */
typedef struct {
  const void* ptr;      /* bf16, element (img, h, w, c) at ptr + img*s_n + h*s_h + w*s_w + c (strides in elements) */
  int64_t C, W, H, NB;  /* extents */
  int64_t s_w, s_h, s_n;
} tng_aview;

typedef struct {
  int32_t view;  /* index into a[] */
  int32_t a_c0;  /* first channel of A */
  int32_t dw, dh; /* tap offset added to the output pixel coordinate */
  int32_t b_k0;  /* first K column of B */
  int32_t nkb;   /* number of 64-wide K blocks */
} tng_kgroup;

typedef struct {
  tng_aview a[TNG_MAX_AVIEWS];
  int32_t n_aviews;
  const void* b; /* bf16 [Ncols, Ktot], row stride ldb elements */
  int64_t Ncols, Ktot;
  int64_t ldb;         /* 0 = Ktot */
  int32_t W, H, NB; /* output pixel grid */
  tng_kgroup g[TNG_MAX_KGROUPS];
  int32_t n_groups;
  /* epilogue */
  const float* bias;   /* [Ncols] or NULL */
  const float* rowvec; /* [NB, rowvec_ld] per-image vector (first Ncols entries used) or NULL */
  int64_t rowvec_ld;   /* 0 = Ncols */
  const void* res;     /* [rows, ldr] residual or NULL */
  int32_t res_dtype;   /* TNG_DT_* */
  int64_t ldr;
  float alpha;
  int32_t accumulate;  /* out_f32 += x */
  float* out_f32;      /* or NULL */
  int64_t ld_f32;
  void* out_bf16;      /* or NULL */
  int64_t ld_bf16;
  int32_t act;         /* TNG_ACT_* applied to the bf16 output only */
  float act_param;
  int32_t split_off;   /* 0 = off */
  int32_t block_n;     /* N tile: 0 = auto; one of 32, 64, 128, 160, 256 */
  /* GroupNorm statistics of the output for the norm that consumes it (resnet.py:555,581; transformer_2d.py:253):
   * gn_stats[(img * Ncols + n) * 2 + {0, 1}] += sum / sum of squares of x[:, n] (the fp32 epilogue value, before any
   * rounding; a plain bf16 output without an fp32 one is allowed) over the stats_hw rows of image
   * img = row / stats_hw (fp64 accumulators the caller zeroes; per CHANNEL, so that any grouping - also across the
   * channel concat of a skip connection - is a sum of entries). Emitted from the epilogue of the producing GEMM when
   * every tile is full, otherwise by a pass over the output that follows it in the stream. NULL = off. */
  double* gn_stats;
  int64_t stats_hw;
} tng_gemm_desc;

int tng_conv_gemm(const tng_gemm_desc* d, void* stream);
/* What tng_conv_gemm would do with this descriptor, without launching: the N tile, the launch mode (1 = one CTA per SM,
 * 4 = CTA pair on a 256 x 2 block_n tile, 2 / 3 = experiment modes) and the split-K factor. Used by bench.py to label
 * its per-kernel timings with the instantiation that actually runs. Any output pointer may be NULL. */
int tng_gemm_plan(const tng_gemm_desc* d, int32_t* block_n, int32_t* mode, int32_t* ksplit);

/* ---------------------------------------------------------------------------------------------------------
 * tng_attention — tcgen05 flash attention, head width 64, fp32 online softmax.
 * Replaces: Attention + AttnProcessor(2_0) core  softmax(q k^T * scale + bias) v
 *           (mustango/diffusers/src/diffusers/models/attention_processor.py:232-261,263-299,500-540)
 *           and the additive mask bias of unet_2d_condition.py:575-579.
 * q: bf16 rows = batch*Lq tokens, head h at columns q_col0 + 64*h; k, v likewise with Lk tokens per batch.
 * kbias: optional fp32 [batch, Lk] additive bias (already (1-mask)*-10000). out: bf16 [batch*Lq, ld_o],
 * head h at columns 64*h (hi) and, if split_off > 0, the rounding residual at + split_off.
 * nsplit = 1: plain bf16 operands. nsplit = 2: every operand also carries its bf16 rounding residual ("lo") at
 * column + *_lo_off, and the kernel evaluates the 3-term split products hi*hi + lo*hi + hi*lo (parity mode).
 */
typedef struct {
  const void* q; int64_t ld_q; int32_t q_col0; int32_t q_lo_off;
  const void* k; int64_t ld_k; int32_t k_col0; int32_t k_lo_off;
  const void* v; int64_t ld_v; int32_t v_col0; int32_t v_lo_off;
  const float* kbias;
  void* out; int64_t ld_o; int32_t split_off;
  int32_t batch, heads, Lq, Lk;
  float scale;
  int32_t nsplit;
} tng_attn_desc;

int tng_attention(const tng_attn_desc* d, void* stream);

/* tng_attention_wide — tcgen05 flash attention for ONE head of width `dim` = 512, Lq = Lk = L, no mask: the AudioLDM VAE
 * AttnBlock  softmax(q k^T * scale) v  over the H*W positions of each image
 * (audioldm/variational_autoencoder/modules.py:204-230). q / k / v: bf16 rows = batch*L positions, the operand at columns
 * [col0, col0 + dim) of a row-major matrix with leading dimension ld (elements); out: bf16 [batch*L, ld_o], columns
 * [0, dim). The [L, L] score matrix stays on the SM (S, P and O live in tensor memory). L must be a multiple of 128. */
int tng_attention_wide(const void* q, int64_t ld_q, int32_t q_col0, const void* k, int64_t ld_k, int32_t k_col0,
                       const void* v, int64_t ld_v, int32_t v_col0, void* out, int64_t ld_o, int32_t batch, int32_t L,
                       int32_t dim, float scale, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * GroupNorm (+SiLU) over channels-last input that may be the channel concat of two tensors (skip connection).
 * Replaces: nn.GroupNorm + SiLU in ResnetBlock2D (resnet.py:555-557,581-587), conv_norm_out
 *           (unet_2d_condition.py:699-701), Transformer2DModel.norm (transformer_2d.py:253),
 *           torch.cat skip (unet_2d_blocks.py:2210,2495), VAE Normalize+swish (modules.py:37-41,155-175).
 * Statistics are kept PER CHANNEL: col_stats fp64 [NB, C, 2] (sum, sum of squares over the HW pixels of an image). They
 * normally come out of the producing tng_conv_gemm (gn_stats above); tng_groupnorm_stats is the stand-alone pass for
 * tensors no GEMM produced (it ADDS to col_stats: the caller zeroes them).
 */
int tng_groupnorm_stats(const void* x, int32_t dt, int64_t C, int64_t ld, int64_t NB, int64_t HW, double* col_stats,
                        void* stream);
/* y = act((x - mean) * rstd * gamma + beta) -> bf16 [NB*HW, ld_y] (+ lo half at split_off if > 0) for x = [x0 | x1]
 * (x1 / stats1 may be NULL); mean / rstd of group g over its (C0 + C1) / groups consecutive channels of the concat, from
 * stats0 [NB, C0, 2] and stats1 [NB, C1, 2]; optional bf16 copy of the *raw* concat input to raw_bf16 (the operand of
 * the fused 1x1 shortcut conv). */
int tng_groupnorm_apply(const void* x0, int32_t dt0, int64_t C0, const double* stats0, const void* x1, int32_t dt1,
                        int64_t C1, const double* stats1, int64_t NB, int64_t HW, int32_t groups, const float* gamma,
                        const float* beta, float eps, int32_t act, void* y, int64_t ld_y, int32_t split_off,
                        void* raw_bf16, int64_t ld_raw, int32_t raw_split_off, void* stream);

/* LayerNorm over the last dim of fp32 [rows, C] -> bf16 (attention.py:259,267,274). */
int tng_layernorm(const float* x, int64_t rows, int64_t C, const float* gamma, const float* beta, float eps,
                  void* y, int64_t ld_y, int32_t split_off, void* stream);

/* ---- text-conditioning front-end (SURVEY.md section 8(f).1): FLAN-T5 encoder as called from models.py:98-100 (T5EncoderModel),
 * models.py:129-147 (encode_text) and models.py:266-305 (encode_text_classifier_free). The arithmetic lives in the pip
 * dependency `transformers` (models/t5/modeling_t5.py: T5LayerNorm, T5Attention, T5DenseGatedActDense, T5Stack), which is
 * not under /root/reference; the entry points below replace those modules, the projections run through tng_conv_gemm. */

/* T5LayerNorm: y = x * rsqrt(mean(x^2) + eps) * gamma over the last dim of fp32 [rows, C] -> bf16 y (+ lo half) and/or a
 * dense fp32 copy y_f32 [rows, C] (the final_layer_norm output handed to the UNet); either output may be NULL. */
int tng_rmsnorm(const float* x, int64_t rows, int64_t C, const float* gamma, float eps, void* y, int64_t ld_y,
                int32_t split_off, float* y_f32, void* stream);
/* nn.Embedding lookup (T5Stack.embed_tokens): out[r, :] = table[ids[r], :], fp32 [rows, C]; ids are int64 and must lie in
 * [0, n_table_rows) (checked by the caller, as nn.Embedding's own index check is host-side on CPU). */
int tng_gather_rows(const float* table, int64_t n_table_rows, const int64_t* ids, int64_t rows, int64_t C, float* out,
                    void* stream);
/* T5Attention.forward core for head width 64: softmax(q k^T + relbias[h, key - query] + kbias[b, key]) v, no score
 * scaling. qkv: fp32 [batch*L, ld] with the q / k / v blocks of `heads*64` columns at q_col0 / k_col0 / v_col0;
 * relbias: fp32 [heads, 2L-1] (index key - query + L - 1; the bucketed relative_attention_bias of block 0, shared by all
 * blocks); kbias: fp32 [batch, L] additive key mask (0 or finfo.min, as get_extended_attention_mask builds it) or NULL;
 * out: bf16 [batch*L, ld_o] (+ lo half at split_off). */
int tng_rel_attention(const float* qkv, int64_t ld, int32_t q_col0, int32_t k_col0, int32_t v_col0, int32_t batch,
                      int32_t heads, int32_t L, const float* relbias, const float* kbias, void* out, int64_t ld_o,
                      int32_t split_off, void* stream);

/* fp32 [rows, C] -> bf16 [rows, ld_y] with optional activation, optional hi/lo split, optional nearest x2
 * upsample of an (NB, H, W) grid (resnet.py:146; modules.py:53-57) — the cast in front of a conv that consumes
 * the residual stream directly (conv_in, Downsample2D, Upsample2D, HiFi-GAN leaky_relu -> conv). */
int tng_cast_act(const float* x, int64_t NB, int64_t H, int64_t W, int64_t C, int64_t ld_x, int32_t upsample2x,
                 int32_t act, float act_param, void* y, int64_t ld_y, int32_t split_off, void* stream);

/* Row softmax of fp32 [rows, L] * scale -> bf16 [rows, ld_y] (VAE AttnBlock, modules.py:211-214). */
int tng_softmax_rows(const float* x, int64_t rows, int64_t L, int64_t ld_x, float scale, void* y, int64_t ld_y,
                     int32_t split_off, void* stream);

/* bf16 [B, R, C] -> bf16 [B, C, R] (per-batch transpose; builds K-major V^T for the VAE attention PV GEMM). */
int tng_transpose_bf16(const void* x, int64_t B, int64_t R, int64_t C, int64_t ld_x, void* y, int64_t ld_y,
                       void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Fused classifier-free guidance + scheduler update (one HBM pass).
 * Replaces: models.py:244-249 (chunk, uncond + g*(text-uncond)) and DDPMScheduler.step
 *           (scheduling_ddpm.py:290-344) / DDIMScheduler.step eta=0 (scheduling_ddim.py:292-354).
 * coef = float[10] {c_x0_sample, c_x0_model, c_prev_x0, c_prev_sample, c_noise, c_eps_sample, c_eps_model,
 *         c_prev_eps, clip (0 = off), c_x0_div}: fp32 scalars computed on the host with the reference's own fp32
 *         op order (device pointer, so a step can be replayed from a CUDA graph with updated coefficients).
 *   x0   = (c_x0_sample * sample + c_x0_model * v) / c_x0_div   (clamped to +-clip if clip > 0)
 *   eps  = c_eps_sample * sample + c_eps_model * v
 *   prev = c_prev_x0 * x0 + c_prev_sample * sample + c_prev_eps * eps + c_noise * noise
 * model_out: fp32 channels-last [(2)B, HW, C] (uncond half first when cfg); sample/noise/prev: fp32 NCHW
 * [B, C, HW] (the reference's latent layout); also writes next_in: the channels-last bf16 UNet input
 * [(2)B, HW, ld_in] for the next step (latents duplicated for the two CFG halves, hi/lo split optional).
 */
int tng_sched_step(const float* model_out, int64_t ld_mo, int32_t cfg, float guidance, const float* sample,
                   const float* noise, const float* coef, float* prev, void* next_in, int64_t ld_in,
                   int32_t split_off, int64_t B, int64_t C, int64_t HW, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Fused classifier-free guidance + multistep DPM-Solver / DPM-Solver++ update (one HBM pass).
 * Replaces: models.py:244-249 and DPMSolverMultistepScheduler.step (scheduling_dpmsolver_multistep.py:
 *           convert_model_output + the first / second / third order updates).
 * coef = float[11] {c_s, c_m, c_div, k_s, k0, k1, k2, a1, a2, a3, a4}: fp32 scalars computed on the host with the
 *        reference's fp32 op order (device pointer). The reference's subtractions are folded into negative
 *        coefficients (exact in IEEE arithmetic). Every operation below is rounded on its own (no fma contraction):
 *   v  = u + guidance * (t - u)      (cfg; else v = model_out)
 *   m0 = (c_s * sample + c_m * v) / c_div                              -> written to m0 (this step's history entry)
 *   order 1: prev = k_s * sample + k0 * m0
 *   order 2: D1 = a1 * (m0 - m1);  prev = (k_s * sample + k0 * m0) + k1 * D1
 *   order 3: E0 = a1 * (m0 - m1);  E1 = a2 * (m1 - m2);  D1 = E0 + a3 * (E0 - E1);  D2 = a4 * (E0 - E1)
 *            prev = ((k_s * sample + k0 * m0) + k1 * D1) + k2 * D2
 * model_out: fp32 channels-last [(2)B, HW, ld_mo] (uncond half first when cfg); sample, m1, m2 (the converted outputs
 * of the previous two steps; read only when `order` needs them), m0, prev: fp32 NCHW [B, C, HW]; prev may alias
 * sample, m0 may not alias sample, m1 or m2. prev and next_in are optional (at least one). next_in: the channels-last
 * bf16 UNet input of the next step, exactly as tng_sched_step writes it.
 */
int tng_sched_multistep(const float* model_out, int64_t ld_mo, int32_t cfg, float guidance, const float* sample,
                        const float* m1, const float* m2, const float* coef, int32_t order, float* m0, float* prev,
                        void* next_in, int64_t ld_in, int32_t split_off, int64_t B, int64_t C, int64_t HW,
                        void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Small exact-fp32 pieces.
 * tng_timestep_embedding: get_timestep_embedding (embeddings.py:22-62), flip_sin_to_cos / freq_shift configurable.
 * tng_linear_f32: y = act(x) @ W^T + b for tiny M (TimestepEmbedding, resnet time_emb_proj; embeddings.py:200-212,
 *                 resnet.py:572-573). pre_act is applied to x on load, post_act to y.
 */
int tng_timestep_embedding(const float* t, int64_t n, int32_t dim, int32_t flip_sin_to_cos, float freq_shift,
                           float* out, void* stream);
int tng_linear_f32(const float* x, int64_t M, int64_t K, const float* w, const float* b, int64_t N,
                   int32_t pre_act, int32_t post_act, float* y, void* stream);

/* HiFi-GAN ConvTranspose1d overlap-add: y[b, l, co] = bias[co] + sum_{q,t: q*stride + t - pad = l} Y[b, q, t*Cout + co]
 * (audioldm/hifigan/models.py:124-135,153), Y being the tng_conv_gemm output [B, Lin, ktaps*Cout] fp32. */
int tng_convt_gather(const float* Y, int64_t B, int64_t Lin, int32_t ktaps, int64_t Cout, int32_t stride, int32_t pad,
                     int64_t Lout, const float* bias, float* y, void* stream);

/* Final waveform: tanh then the host-side `(x * 32768).astype(int16)` of hifigan/utilities.py:81
 * (C-style truncation toward zero; the +1.0 wrap-around of the reference is reproduced). */
int tng_tanh_to_i16(const float* x, int64_t n, int64_t ld_x, float* wave_f32, int16_t* wave_i16, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * TacotronSTFT mel front-end (SURVEY.md section 8(f).2): audioldm/audio/stft.py:52-83 (STFT.transform: reflect pad,
 * strided conv1d with the windowed Fourier basis, magnitude), :161-186 (mel_spectrogram), audio_processing.py:85-91
 * (log of the value clamped at 1e-5). The two contractions (basis, mel filter bank) run through tng_conv_gemm.
 * tng_stft_frames: y fp32 [B, T] -> reflect-padded by `pad` on both sides, split into bf16 hi / lo planes [B, ld]
 *   (ld >= T + 2 pad, zero beyond): frame f of batch b is the OVERLAPPING window [f hop, f hop + filter_length) of a plane,
 *   i.e. a tng_aview with s_w = hop — the conv1d needs no im2col buffer.
 * tng_stft_magnitude: F fp32 [rows, ldF] = (real | imag) halves of `bins` columns -> mag = sqrt(re^2 + im^2) as the bf16
 *   operand of the mel GEMM (hi at column b, lo at split_off + b; may be NULL), log_mag fp32 [rows, bins] =
 *   log(max(mag, floor)) (may be NULL), energy fp32 [rows] = ||mag||_2 (may be NULL).
 * tng_log_clamp: y = log(max(x, floor)). */
int tng_stft_frames(const float* y, int64_t B, int64_t T, int32_t pad, void* hi, void* lo, int64_t ld, void* stream);
int tng_stft_magnitude(const float* F, int64_t rows, int32_t bins, int64_t ldF, void* mag_op, int64_t ld_op,
                       int32_t split_off, float* log_mag, float* energy, float floor_v, void* stream);
int tng_log_clamp(const float* x, int64_t n, float floor_v, float* y, void* stream);

#ifdef __cplusplus
}
#endif
#endif
