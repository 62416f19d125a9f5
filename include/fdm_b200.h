/*
 * fdm_b200.h — C ABI of libfdm_b200.so: the sm_100a kernels behind the LG-LDM sampling hot path
 * of wangxuanx/Face-Diffusion-Model (SURVEY.md §8).
 *
 * Conventions (all entry points):
 *   - plain device pointers + explicit sizes/strides (element units unless stated), no torch types;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - every call is asynchronous on `stream`, never allocates or frees caller memory;
 *   - return 0 on success, non-zero on error; fdm_last_error() returns a thread-local message;
 *   - dtype codes: FDM_F32 = 0, FDM_BF16 = 1.
 *
 * The reference has no FFI layer (it is pure PyTorch); each entry point cites the reference
 * Python call site it replaces (paths relative to the reference checkout).
 */
#ifndef FDM_B200_H
#define FDM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FDM_F32 0
#define FDM_BF16 1

/* activation codes for the GEMM / norm epilogues */
#define FDM_ACT_NONE 0
#define FDM_ACT_RELU 1       /* nn.TransformerDecoderLayer FFN (models/fdm_vocaset.py:45) */
#define FDM_ACT_MISH 2       /* nn.Mish in audio_extract / latent_encoder / time_embedd (models/fdm_vocaset.py:20-39) */
#define FDM_ACT_GELU_ERF 3   /* HF HuBERT "gelu" (transformers/models/hubert/modeling_hubert.py) */
#define FDM_ACT_GELU_TANH 4  /* models/utils/base_model_util.py:81-94 */
#define FDM_ACT_LEAKY02 5    /* nn.LeakyReLU(0.2) in the VQ decoder expander (models/vq_vae_vocaset.py:197) */

/* ---- library / device ------------------------------------------------------------------- */
const char* fdm_last_error(void);
/* Fills SM count and compute capability of the current device; fails unless it is sm_100. */
int fdm_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);
int fdm_abi_version(void);

/* ---- dense layers (SURVEY K1) ----------------------------------------------------------- *
 * C[M,N] = act(A[M,K] * W[N,K]^T + bias[N]) + residual[M,N]
 * replaces every nn.Linear / Conv1d call on the path (models/fdm_vocaset.py:20-51,
 * models/lib/base_models.py:71-174, models/vq_vae_vocaset.py:194-258, HF HuBERT convs/linears).
 *
 * Implicit 1-D convolution: with taps > 1, K = taps * tap_k and
 *   A(m, tap*tap_k + c) = A[(m + tap*tap_row_shift) * lda + c],
 * i.e. the k-th filter tap reads the activation row shifted by tap*tap_row_shift; strided convs
 * use a plain GEMM with lda = stride * C_in (rows overlap). a_rows = number of addressable rows
 * of A (bounds for the TMA descriptor; >= M + (taps-1)*tap_row_shift).
 */
typedef struct fdm_gemm_args {
  const void* A;          /* bf16 (fdm_gemm_bf16) or f32 (fdm_gemm_f32), row-major, K contiguous */
  int64_t lda;            /* row stride of A in elements */
  int64_t a_rows;
  const void* W;          /* same dtype as A, [N, K] row-major (nn.Linear.weight layout) */
  int64_t ldw;
  const float* bias;      /* [N] f32 or NULL */
  const void* residual;   /* [M, N] or NULL; added after the activation */
  int64_t ldr;
  int32_t res_dtype;      /* FDM_F32 / FDM_BF16 */
  int32_t out_dtype;      /* FDM_F32 / FDM_BF16 */
  void* C;
  int64_t ldc;
  int64_t M, N, K;
  int32_t act;
  int32_t taps;           /* 1 = plain GEMM */
  int64_t tap_k;
  int64_t tap_row_shift;
  /* ---- LayerNorm folding (fdm_gemm_bf16 only; every pointer NULL = plain GEMM) -------------------------------------
   * A post-norm layer ends in y = LN(u; gamma, beta). Instead of materialising y, the GEMM that produces u also writes
   * per-row partial statistics (stats_out), fdm_ln_stats_finalize turns them into (mean, rstd) per row, and
   *  - a consumer y W^T is computed from u with pre-scaled weights W' = W diag(gamma):
   *        C = rstd (u W'^T - mean * w_colsum) + bias',   w_colsum[n] = sum_k W'[n,k],  bias' = bias + W beta   (a_ln)
   *  - a residual  "+ y"  is rebuilt element-wise from u:  (u - mean) rstd res_gamma + res_beta                 (res_ln)
   * This removes the LayerNorm kernel between two GEMMs (one read and one write of the activation). */
  const float* a_ln;       /* [M][2] (mean, rstd) of the rows of A, or NULL */
  const float* w_colsum;   /* [N], required with a_ln */
  const float* res_ln;     /* [M][2] (mean, rstd) of the rows of `residual`, or NULL (needs the bf16-in / bf16-out TMA path) */
  const float* res_gamma;  /* [N] */
  const float* res_beta;   /* [N] */
  float* stats_out;        /* [M][N/64][2]: per 64-column group, sum and sum of squares of the fp32 OUTPUT row values;
                              needs the bf16 residual TMA path and N % 64 == 0, or NULL */
  /* ---- split-bf16 ("bf16x3") operands (fdm_gemm_bf16 only; both NULL = plain bf16 GEMM) ------------------------------
   * fp32-grade products on the tensor cores: with x = x_hi + x_lo (fdm_split_bf16x2) the kernel accumulates, in ONE
   * fp32 TMEM accumulator,  A_lo W^T + A W_lo^T + A W^T  (A / W hold the hi parts; the lo.lo term, 2^-18 relative, is
   * dropped), i.e. three passes over K inside the same tile. A_lo / W_lo have exactly the layout of A / W (same lda /
   * a_rows / taps, same ldw). Used by the high-precision steps of the sampler and the once-per-clip audio encoder. */
  const void* A_lo;
  const void* W_lo;
  /* ---- grouped (block-diagonal) mode, fdm_gemm_bf16 only; 0 = off ------------------------------------------------------
   * A grouped Conv1d (HF HubertPositionalConvEmbedding: 16 groups of 64 channels, k = 128) as ONE launch: output columns
   * [64 g, 64 g + 64) are computed from the columns [g * a_group_cols, (g + 1) * a_group_cols) of A (per tap) and rows
   * [64 g, 64 g + 64) of W, whose K index runs over that group's taps x channels only. Needs N % 64 == 0 and
   * a_group_cols == tap_k (taps > 1) or == K, a multiple of 64. */
  int64_t a_group_cols;
  /* ---- tail split-K workspace (fdm_gemm_bf16 only; NULL = off) ---------------------------------------------------------
   * When the static tile schedule leaves the last wave at most half full, the tiles of that wave are cut along K into
   * slices that run on the otherwise idle SMs; the slices exchange fp32 partial tiles through this DEVICE buffer
   * (deterministic: fixed summation order). The first 4096 bytes hold counters and must be ZERO before the first use;
   * the kernel leaves them zero. 256-byte aligned; 20 MB covers every shape (4096 + (SMs / 4) * 8 * 256 KB is the
   * maximum); a launch whose plan does not fit simply runs without the split. One workspace must not be shared by
   * launches that may run CONCURRENTLY (different streams); launches ordered on a stream or in a graph can share it. */
  void* splitk_ws;
  int64_t splitk_ws_bytes;
} fdm_gemm_args;

/* Kernel-selection switches of fdm_gemm_bf16 (process-wide; results are identical up to fp32 summation order):
 *   "resmma" = 1: a bf16 residual of a GEMM without activation is accumulated by the tensor core (identity k-blocks appended
 *                 to the K loop) instead of being added in the epilogue; 0 (default, or env FDM_B200_GEMM_RESMMA) = epilogue. */
int fdm_gemm_set_option(const char* name, int32_t value);
/* TMA-fed tcgen05/TMEM GEMM, bf16 operands, fp32 accumulation. */
int fdm_gemm_bf16(const fdm_gemm_args* args, void* stream);
/* fp32 FFMA GEMM (deterministic k order) — the "fp32 mode" used for the 1e-4 parity runs. */
int fdm_gemm_f32(const fdm_gemm_args* args, void* stream);
/* (mean, rstd) per row from the partial statistics a GEMM wrote through stats_out: partials [M][parts][2] (sum, sum
 * of squares per column group), d = number of columns they cover; mean_rstd [M][2]. Deterministic (fixed order). */
int fdm_ln_stats_finalize(const float* partials, int64_t M, int64_t parts, int64_t d, float eps, float* mean_rstd,
                          void* stream);

/* ---- normalisation (SURVEY K4, K9) ------------------------------------------------------- *
 * Row LayerNorm with fused residual adds; replaces norm1/2/3 of nn.TransformerDecoderLayer
 * (post-norm, eps 1e-5), base_models.Norm (models/lib/base_models.py:37-52) and HF HuBERT LNs.
 *   y = x + r1 (if r1)            ; y = LN(y; g1, b1)  (if g1)  ; y = act1(y)
 *   if g2: y = y + r2[row % r2_rows] (if r2) + vec2[vec_index * d .. ] (if vec2) ; y = LN(y; g2, b2)
 *          (r2_rows = 0 means r2 has one row per input row; otherwise r2 is shared by row blocks, e.g. by the
 *           conditional and unconditional guidance passes)
 * out (out_dtype) and optional out2 (the other dtype) receive y.
 * vec_index is read on the device from *vec_index_dev (the denoising step t) when vec2 != NULL.
 */
typedef struct fdm_norm_args {
  const void* x; int64_t ldx; int32_t x_dtype;
  const void* r1; int64_t ldr1; int32_t r1_dtype;
  const float* g1; const float* b1;
  int32_t act1;
  const void* r2; int64_t ldr2; int32_t r2_dtype; int64_t r2_rows;
  const float* vec2; const int32_t* vec_index_dev;
  const float* g2; const float* b2;
  void* out; int64_t ldo; int32_t out_dtype;
  void* out2; int64_t ldo2; int32_t out2_dtype;
  int64_t rows; int64_t d;
  float eps;
} fdm_norm_args;
int fdm_layernorm(const fdm_norm_args* args, void* stream);

/* y = post_act( InstanceNorm_over_time( leaky_relu(x, slope) ) * gamma + beta ) on a [B, T (t_stride rows per
 * clip), C] activation, written with out_t_stride rows per clip (this also compacts a padded conv output).
 * slope = 0.2, gamma = beta = NULL, post_act = NONE: LeakyReLU + InstanceNorm1d(affine=False) of the VQ decoder
 * expander (models/vq_vae_vocaset.py:194-199). slope = 1, gamma/beta, post_act = GELU: the per-channel GroupNorm +
 * GELU after the first conv of the wav2vec2-base feature encoder (HF Wav2Vec2GroupNormConvLayer, behind
 * models/wav2vec.py:88). Statistics are biased (divide by T), fp32. */
int fdm_leaky_instnorm(const void* x, int32_t x_dtype, void* out, int32_t out_dtype,
                       int64_t B, int64_t T, int64_t t_stride, int64_t out_t_stride, int64_t C,
                       float slope, float eps, const float* gamma, const float* beta, int32_t post_act,
                       void* stream);

/* ---- attention (SURVEY K2) ---------------------------------------------------------------- *
 * O[b,t,h,:] = softmax_j( scale * Q[b,t,h,:].K[b,j,h,:] + bias(h,t,j) ) V[b,j,h,:]
 * bias_mode 0: none (VQ decoder, models/lib/base_models.py:150-174; HuBERT encoder)
 * bias_mode 1: FaceFormer-style periodic ALiBi + causal mask computed in-kernel,
 *              bias = -slopes[h] * floor((t-j)/period) for j<=t, -inf for j>t
 *              (models/fdm_vocaset.py:94-115 init_biased_mask; never materialised here).
 * Row of (b,t) = b*t_stride + t; head h at column h*dh of each of Q/K/V; ld* in elements.
 */
typedef struct fdm_attn_args {
  const void* Q; const void* K; const void* V; int64_t ldq; int64_t ldk; int64_t ldv;
  void* O; int64_t ldo;
  int32_t dtype;          /* dtype of Q/K/V/O */
  int64_t B, T, t_stride, H, dh;
  float scale;
  int32_t bias_mode; int32_t period; const float* slopes;
} fdm_attn_args;
int fdm_self_attention(const fdm_attn_args* args, void* stream);

/* ---- diffusion step (SURVEY K7: S4 + S5 + C1) --------------------------------------------- *
 * One fused, vectorised kernel per denoising step:
 *   x0   = x0_uncond + guidance * (x0_cond - x0_uncond)      (utiles/classifierfree.py:20-21; skipped if x0_uncond == NULL)
 *   mean = c1[t]*x0 + c2[t]*x_t                              (diffusion_BIWI_encoder_decoder.py:632-639)
 *   out  = mean + sigma[t]*noise   (no noise when t == 0)    (diffusion_BIWI_encoder_decoder.py:650-656)
 * t comes from t_per_clip[b] (int64, p_sample API) or, if NULL, from *t_dev (device-resident step
 * counter: CUDA-graph replay without host sync). noise == NULL selects the in-kernel Philox4x32-10 +
 * Box-Muller generator keyed by (seed, clip_index0 + b, t, element). Products and sums are
 * individually rounded (no FMA contraction) to match the PyTorch expression bit for bit.
 * out_bf16 (optional) receives a bf16 copy of out for the next step's first GEMM.
 */
typedef struct fdm_ddpm_args {
  const float* x0_cond; const float* x0_uncond; float guidance;
  const float* x_t; const float* noise;
  float* out; void* out_bf16;
  const float* c1; const float* c2; const float* sigma;    /* [num_timesteps] tables */
  const int64_t* t_per_clip; const int32_t* t_dev;
  int64_t B; int64_t elems_per_clip;
  uint64_t seed; int64_t clip_index0;
  const uint64_t* seed_dev;  /* optional: the Philox seed is read from device memory instead of `seed`, so a captured
                                step graph can be replayed with a fresh seed per sampling call */
} fdm_ddpm_args;
int fdm_ddpm_step(const fdm_ddpm_args* args, void* stream);
/* DDIM update (eta = 0), reference diffusion_BIWI_encoder_decoder.py:675-710, fused with the optional CFG combine:
 *   eps = (a_recip[i] * x_t - x0) / a_recipm1[i] ;  out = x0 * sqrt_an[i] + c[i] * eps
 * where i = *index_dev indexes per-step coefficient tables prepared on the host with the reference's fp32 torch
 * expressions (a_recip = sqrt_recip_alphas_cumprod[t], a_recipm1 = sqrt_recipm1_alphas_cumprod[t],
 * sqrt_an = sqrt(alphas_cumprod[t_next]), c = sqrt(1 - alphas_cumprod[t_next])). Each operation is rounded
 * separately, as in the PyTorch expression. */
typedef struct fdm_ddim_args {
  const float* x0_cond; const float* x0_uncond; float guidance;
  const float* x_t; float* out; void* out_bf16;
  const float* a_recip; const float* a_recipm1; const float* sqrt_an; const float* c;
  const int32_t* index_dev;
  int64_t n;               /* total elements */
} fdm_ddim_args;
int fdm_ddim_step(const fdm_ddim_args* args, void* stream);

/* Known frames (latent inpainting / continuation): for every row r = b*T + f (sequence b, frame f, d elements) whose
 * mask[r] is non-zero, with i = *index_dev + offset:
 *   x = ka[i] * known + kb[i] * z      (each product rounded, then added: the reference's q_sample expression)
 *   x = ka[i] * known                  (when kb[i] == 0; no draw)
 * Rows whose mask is zero are not touched. z is noise[...] (noise may alias x: the start state reuses x_T's own value),
 * or, when noise == NULL, the Philox normal fdm_ddpm_step draws for (seed = *seed_dev, clip_index0 + b, t = *t_dev,
 * element) - bit-identical to fdm_philox_normal at that key. x_bf16 (optional) receives the bf16 copy of the rows
 * written. ka / kb are per-call tables (entry 0: the start state, entry s + 1: the state after step s). */
typedef struct fdm_known_args {
  float* x; void* x_bf16;
  const float* known; const uint8_t* mask;
  const float* noise;
  const float* ka; const float* kb;
  const int32_t* index_dev; int32_t offset;
  const uint64_t* seed_dev; const int32_t* t_dev; int64_t clip_index0;
  int64_t B; int64_t T; int64_t d;   /* B sequences of T rows of d elements; x / known / noise hold B*T*d floats */
} fdm_known_args;
int fdm_known_frames(const fdm_known_args* args, void* stream);

/* End of a graph-replayed step: cursor[0] += 1; t_dev[0] = t_sched[min(cursor[0], n_sched-1)]. */
int fdm_advance_cursor(int32_t* cursor_dev, const int32_t* t_sched, int32_t n_sched, int32_t* t_dev, void* stream);
/* Fill out[B*elems_per_clip] with the same Philox normals the fused step would draw for step t. */
int fdm_philox_normal(float* out, int64_t B, int64_t elems_per_clip, uint64_t seed,
                      int64_t clip_index0, int32_t t, void* stream);

/* ---- VQ quantiser (SURVEY K8 / Q1) --------------------------------------------------------- *
 * For each row z (D floats): d_j = (sum z^2 + sum e_j^2) - 2*(z . e_j), all fp32, each sum a
 * sequential fmaf chain over k = 0..D-1 starting from 0.0f; index = argmin_j d_j, lowest j on
 * ties (models/lib/quantizer.py:35-64, models/vq_vae_emotion.py:221-252).
 * code_offset[b] (optional) selects the per-clip codebook slice [off, off+n_codes) (emotion).
 * Writes indices (int64, local to the slice) and z_q in the reference's permuted layout
 * z_q[b, k, l] (B, D, L) and/or row layout z_q_rows[b, l, k].
 */
int fdm_vq_quantize(const float* z, const float* codebook, const int64_t* code_offset,
                    int64_t B, int64_t L, int64_t D, int64_t n_codes,
                    int64_t* indices, float* zq_bdl, float* zq_rows, void* stream);
/* Same contract with an explicit algorithm. FDM_VQ_FFMA evaluates every chain on the fp32 pipes (any D in {32,64,128}).
 * FDM_VQ_TENSOR (D = 64 or 128) ranks the codes with a bf16x3 tcgen05 distance GEMM, proves all but a window of near-minimal
 * codes cannot win, and evaluates the exact chains for the survivors only: identical indices, HBM-bound instead of
 * FFMA-bound. FDM_VQ_AUTO picks FDM_VQ_TENSOR when D = 64 / 128. recheck_rows (optional, device, caller-zeroed) counts the rows
 * that needed the exact pass; dbg_acc (optional, device, [B*L, n_codes] f32) receives the tensor-core dot products. */
#define FDM_VQ_AUTO 0
#define FDM_VQ_FFMA 1
#define FDM_VQ_TENSOR 2
int fdm_vq_quantize_ex(const float* z, const float* codebook, const int64_t* code_offset,
                       int64_t B, int64_t L, int64_t D, int64_t n_codes,
                       int64_t* indices, float* zq_bdl, float* zq_rows, int32_t algo,
                       uint64_t* recheck_rows, float* dbg_acc, void* stream);
/* By-products of VectorQuantizer.forward (models/lib/quantizer.py:52-61, models/vq_vae_emotion.py:240-250) from the chosen
 * indices in one pass over z: sqerr_partials[n_partials] = per-block partial sums of (e_idx - z)^2 over all elements (the
 * caller adds them; loss = (1 + beta) * sum / (rows * D)), hist[n_codes] += code usage counts (caller zero-fills; perplexity
 * = exp(-sum p log(p + 1e-10))). code_offset as in fdm_vq_quantize (per-clip slice; indices are slice-local). */
int fdm_vq_stats(const float* z, const float* codebook, const int64_t* code_offset, const int64_t* indices, int64_t B,
                 int64_t L, int64_t D, int64_t n_codes, float* sqerr_partials, int64_t n_partials, int64_t* hist,
                 void* stream);

/* ---- small data-movement kernels ------------------------------------------------------------ */
/* hi = bf16(x), lo = bf16(x - hi): the operand pair of the split-bf16 GEMM (fdm_gemm_args.A_lo / W_lo). n elements. */
int fdm_split_bf16x2(const float* src, void* hi, void* lo, int64_t n, void* stream);
int fdm_cast(const void* src, int32_t src_dtype, void* dst, int32_t dst_dtype, int64_t n, void* stream);
/* dst[b, l, c] = src[b, c, l] (+ cast); used for VQAutoEncoder.decode's (B,D,L) input. */
int fdm_transpose_bcl_to_blc(const float* src, void* dst, int32_t dst_dtype,
                             int64_t B, int64_t C, int64_t L, void* stream);
/* Copy [B, T, C] rows into a per-clip padded buffer [B, pad_l + T + pad_r, C]; padding rows are
 * replicated edge rows (mode 1, Conv1d padding_mode='replicate') or zeros (mode 0). */
int fdm_pad_time(const void* src, int64_t src_t_stride, void* dst, int32_t dtype, int64_t B, int64_t T,
                 int64_t C, int64_t pad_l, int64_t pad_r, int32_t mode, void* stream);
/* dst[r, :] = cast(src[r, 0:cols]) then zeros up to ld_dst: gives activations whose row length is not a multiple of
 * 8 (in_dim = 15069 / 70110 of the EVQ-VAE encoder's first Linear) the 16-byte row pitch the TMA-fed GEMM needs. */
int fdm_cast_rows(const float* src, int64_t ld_src, void* dst, int32_t dst_dtype, int64_t ld_dst,
                  int64_t rows, int64_t cols, void* stream);
/* Audio front-end of the demos (demo/demo_3d_mead.py:85-97): Wav2Vec2Processor's zero-mean / unit-variance
 * normalisation per clip ((x - mean) / sqrt(var + eps), population variance, eps = 1e-7) followed by Lout - L zero
 * samples (the demos append one second). audio [B, L] f32 -> out [B, Lout] f32. */
int fdm_audio_normalize_pad(const float* audio, int64_t B, int64_t L, float* out, int64_t Lout, float eps,
                            void* stream);
/* Polyphase FIR resampling with scipy.signal.resample_poly semantics, B clips of L_in samples -> L_out samples:
 * out[m] = sum_k taps[k] * xup[(m + pre) * down - k], xup = input zero-stuffed by `up`. The taps (low-pass design, already
 * scaled by `up` and front-padded) and `pre` come from the host (fdm_b200/frontend.py: resample). The demo path's
 * librosa.load(path, sr=16000) step (demo/demo_3d_mead.py:83), SURVEY section 8(f) item 2. */
int fdm_resample_poly(const float* audio, int64_t B, int64_t L_in, float* out, int64_t L_out, const float* taps,
                      int64_t n_taps, int64_t up, int64_t down, int64_t pre, void* stream);
/* Vertex-error metrics of metric/metric.py:115-138 on device: for every frame, reduce over the vertices
 * vertex_idx[0..n_idx) (NULL: all V vertices) the squared L2 distance between pred and gt ([frames, V, 3] f32;
 * gt == NULL compares against zeros): mode 0 = max (LVE / FVE / all-vertex error), mode 1 = mean (EME).
 * out_per_frame [frames] f32; the metric is its mean over frames. */
int fdm_vertex_error(const float* pred, const float* gt, int64_t frames, int64_t V, const int64_t* vertex_idx,
                     int64_t n_idx, int32_t mode, float* out_per_frame, void* stream);
/* Audio feature-encoder layer 0: Conv1d(1, C, k=10, stride=5, optional bias) on raw audio, then
 * LayerNorm(C) + GELU (ln_g != NULL: hubert-large "layer" variant) or nothing (ln_g == NULL: wav2vec2-base "group"
 * variant, normalised over time afterwards by fdm_leaky_instnorm).
 * audio [B, L] f32 -> out [B, out_t_stride, C] (rows >= Lout zero-filled). */
int fdm_hubert_conv0(const float* audio, int64_t B, int64_t L, const float* w, const float* bias,
                     const float* ln_g, const float* ln_b, void* out, int32_t out_dtype,
                     int64_t Lout, int64_t out_t_stride, int64_t C, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FDM_B200_H */
