/* b200sd -- C-ABI of the Blackwell-native Stable Diffusion hot path.
 *
 * Drop-in boundary.  The reference (apple/ml-stable-diffusion) is pure Python; its device
 * boundary is `CoreMLModel.__call__(**np.ndarray) -> dict` (python_coreml_stable_diffusion/
 * coreml_model.py:118-120) which hands the whole UNet / VAE graph to Core ML.  The
 * replacement for that opaque runtime is this library: the graph of the reference network
 * definitions (unet.py:975-1048 etc.) is issued op-by-op through the entry points below by
 * the Python host mirror (`b200sd.model.B200Model`, same `expected_inputs` / `__call__`
 * contract), captured once into a CUDA graph and replayed per denoising step.
 *
 * Conventions
 *   - plain pointers + sizes, no torch types; all pointers are DEVICE pointers unless noted;
 *   - activations are fp16, channels-last: images NHWC, token matrices [rows, channels];
 *   - weights fp16, bias / statistics / scheduler scalars fp32;
 *   - every function returns 0 on success, non-zero on failure with the message available
 *     from b200sd_last_error(); nothing falls back to a CPU path;
 *   - `stream` is a cudaStream_t passed as void*.
 *
 * Each entry point cites the reference code it replaces.
 */
#ifndef B200SD_H
#define B200SD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* b200sd_last_error(void);
int b200sd_version(void);
/* Programmatic dependent launch on/off (default off; env B200SD_PDL=1 enables): lets each kernel's
 * prologue overlap the previous kernel's tail inside the captured CUDA graph. */
void b200sd_set_pdl(int enabled);
/* Measurement aid: only entry points whose class bit is set launch (others return 0 at once): 1 GEMM / convolution,
 * 2 attention, 4 normalisation, 8 elementwise; default 0xF.  bench.py captures one CUDA graph per class over the same
 * buffers to attribute the step time per kernel class. */
void b200sd_set_launch_classes(uint32_t mask);
/* number of kernels launched by this library since load (bench.py's gpu_launches) */
uint64_t b200sd_launch_count(void);

/* ---- tensor-core GEMM / implicit-GEMM convolution --------------------------------------
 * out[M, N] = epilogue( A[M, K] * W[N, K]^T ),  fp16 operands, fp32 accumulate (tcgen05.mma
 * kind::f16, accumulators in TMEM, operands TMA-staged with 128B swizzle).
 *
 *   mode 0  "linear"  : every nn.Conv2d(k=1) of the reference (unet.py:74-84 q/k/v/out,
 *                       :533-551 proj_in/out, :613 GEGLU proj, :601 FF out, :464 conv_shortcut,
 *                       :642-658 TimestepEmbedding).  A = a0 [M, c0] (optionally ++ a1 [M, c1]
 *                       along K: the concat-free form of torch.cat, unet.py:215,270).
 *   mode 1  "conv3x3" : 3x3 pad-1 convolution as an im2col-free implicit GEMM
 *                       (ResnetBlock2D.conv1/conv2 unet.py:435-456, conv_in/out :853,970,
 *                       Downsample2D :507 with stride 2, Upsample2D conv :499).  A = NHWC image
 *                       a0 [n_img, h, w, c0] (optionally ++ a1 with c1 channels); the 9 taps are
 *                       9 shifted TMA boxes with hardware zero fill at the borders.
 *                       W is [N, 9 * (c0 + c1)] with k = (ky*3 + kx) * C + c  (OHWI).
 *   epilogue: + bias[(row / bias_rows) * bias_stride + col] (bias_rows = rows sharing one bias vector;
 *             0 = one vector for all rows; h*w adds the per-image time embedding, unet.py:476-478)
 *             ; GEGLU a*gelu_erf(g) on interleaved column pairs (unet.py:616-617), output N/2 cols
 *             ; + residual[row, col] (unet.py:484-487, :563, :587-589)
 *             ; store fp16 or fp32.
 *   split_k > 1: the k-splits of a tile run as one thread-block cluster (2 / 4 / 8 CTAs) and reduce their fp32
 *   tiles through distributed shared memory; other split counts accumulate fp32 partials in `workspace` and
 *   finish with a reduce kernel (b200sd_gemm_workspace_bytes() says how much scratch a call needs, 0 = none).
 */
typedef struct {
    int32_t mode;          /* 0 linear, 1 conv3x3 */
    int32_t m;             /* rows (linear); ignored for conv (= n_img*h_out*w_out) */
    int32_t n;             /* output channels (before GEGLU halving) */
    int32_t c0, c1;        /* input channels from a0 / a1 (c1 = 0: single source) */
    int32_t n_img, h, w;   /* conv: INPUT image geometry */
    int32_t stride;        /* conv: 1 or 2 */
    int32_t geglu;         /* 1: GEGLU epilogue */
    int32_t out_f32;       /* 1: store fp32 */
    int32_t bias_rows;     /* see above */
    int32_t bias_stride;   /* elements between consecutive bias vectors (0 = n) */
    int32_t split_k;       /* 0 = auto */
    int32_t block_n;       /* 0 = auto; else multiple of 16 in [16, 256] */
    int32_t act;           /* after the bias: 0 none; 1 SiLU (ControlNet conditioning embedder, controlnet.py:36-44);
                              2 GELU (erf) / 3 quick-GELU x*sigmoid(1.702x): the CLIP text encoders' MLP */
    int32_t wgt_tiled;     /* 1: `wgt` is pre-tiled [n_tiles][k_blocks][block_n][64] (block_n must be given): every
                              weight tile is one contiguous block_n*128-byte burst instead of block_n strided rows */
    int32_t pad_after_only; /* conv, stride 2: zero-pad one pixel after the last row / column only, i.e. diffusers'
                               Downsample2D(padding=0) = F.pad(x, (0, 1, 0, 1)) + conv (VAE encoder); 0 = pad 1 all round */
    const void* a0;
    const void* a1;
    const void* wgt;
    const float* bias;     /* or NULL */
    const void* residual;  /* fp16 [M, N_out] or NULL */
    void* out;             /* [M, N_out] fp16 / fp32 */
    float* workspace;      /* split-K scratch (may be NULL when b200sd_gemm_workspace_bytes() == 0) */
    size_t workspace_bytes;
    /* ---- fused normalisation (all optional; zero / NULL = off) ---------------------------------------------------
     * GroupNorm -> SiLU -> conv (unet.py:470-489, 1044-1046) and LayerNormANE -> linear (layer_norm.py:66-78,
     * unet.py:575-590) run without a normalisation launch: the PRODUCER of a tensor leaves its statistics behind
     * (per-channel sums for GroupNorm, per-row sums for LayerNorm) and the CONSUMER applies them -- in the operand
     * path of the halo convolution (GroupNorm + SiLU, applied once per activation patch in shared memory) or as a
     * row scale in the epilogue (LayerNorm folded into the weights). */
    int32_t halo;          /* mode 1, stride 1, pad 1: halo-reuse kernel: one (rows + 2) x (w + 1) activation patch per
                              64-channel chunk in shared memory, the nine taps are row-shifted MMA descriptors; `wgt`
                              must be pre-tiled chunk-major: k-block = chunk * 9 + tap.  1: loader warps fill the patch
                              (GroupNorm / SiLU / upsample on the way in, statistics outputs); 2: plain convolution, the
                              patch is one TMA box per chunk (no gn_*, upsample2x, cs_*; fp16 output, block_n % 32 == 0) */
    int32_t upsample2x;    /* halo: a0 is [n_img, h/2, w/2, c0] and is read nearest-x2 upsampled (Upsample2D, unet.py:499) */
    int32_t gn_groups;     /* halo: > 0 = y = silu?(groupnorm(a0 ++ a1)) feeds the convolution */
    int32_t gn_silu;
    float gn_eps;
    const float* gn_chan0; /* [n_img][c0][2] (sum, sum of squares) per channel of a0 over its h*w pixels */
    const float* gn_chan1; /* same for a1 */
    const float* gn_gamma; /* [c0 + c1] */
    const float* gn_beta;
    /* statistics of THIS call's fp16 output (from the rounded values, deterministic; needs split_k == 1):
     * per-channel sums for a consumer GroupNorm: cs_partial [n_img][slots][n][2] scratch (slots from
     * b200sd_gemm_plan_ex), cs_chan [n_img][n][2] result, cs_tickets [n_img][n_tiles] zero-initialised counters
     * (self-resetting); cs_hw = output rows per image.  rs_out [n_tiles][m][2]: per-row sums for a consumer
     * LayerNorm (mode 0). */
    float* cs_partial;
    float* cs_chan;
    uint32_t* cs_tickets;
    int32_t cs_hw;
    float* rs_out;
    /* LayerNorm folded into this GEMM (mode 0): `wgt` holds gamma (.) W, `bias` holds W beta + b, ln_wg[j] = sum_k
     * of the packed row j, ln_stat [ln_parts][m][2] are the producer's rs_out partials:
     * out = rstd_r * (acc - mu_r * ln_wg) + bias. */
    const float* ln_stat;
    const float* ln_wg;
    int32_t ln_parts;
    float ln_eps;
    /* ResNet shortcut folded into conv2 (mode 1, stride 1; ResnetBlock2D: out = conv2(h) + conv_shortcut(x),
     * unet.py:483-489): a 1x1 convolution over a2 ++ a3 ([n_img, h, w, c2] / [.., c3], c3 may be 0) accumulated into the
     * same output tile as extra k-blocks that read the centre tap only.  `wgt` then holds [n, 9 * (c0 + c1) + c2 + c3]
     * (the shortcut's [n, c2 + c3] matrix appended along K; pre-tiled in that order) and `bias` the sum of both biases. */
    const void* a2;
    const void* a3;
    int32_t c2, c3;
} b200sd_gemm_args;

int b200sd_gemm(const b200sd_gemm_args* args, void* stream);
/* host-only: block_n / split count / k-block count the launcher would choose: out[0..3] = block_n, splits,
 * kb_total, n_tiles */
int b200sd_gemm_plan(const b200sd_gemm_args* args, int32_t* out4);
/* host-only: out[0..7] = block_n, splits, kb_total, n_tiles, statistics slots per image (0: this plan cannot emit
 * column statistics), staged epilogue (0/1), pipeline stages, m_tiles */
int b200sd_gemm_plan_ex(const b200sd_gemm_args* args, int32_t* out8);
/* host-only: human-readable tiling plan (tile shape, split-K, pipeline depth) the launcher would use */
int b200sd_gemm_describe_plan(const b200sd_gemm_args* args, char* buf, size_t buf_size);
/* bytes of fp32 scratch b200sd_gemm would need for these args (0 if no split-K) */
size_t b200sd_gemm_workspace_bytes(const b200sd_gemm_args* args);

/* small-M linear on CUDA cores (weight-bandwidth bound): out[m, n] = act_in(x[m, :]) . W[n, :] + b[n]
 * for the time-embedding MLPs (unet.py:665-682) and the per-ResNet time_emb_proj(silu(emb))
 * (unet.py:442, 476-478).  x, out fp32; W fp16 [n, k]; act_in: 0 none, 1 SiLU on the input;
 * act_out: 0 none, 1 SiLU on the output; add: fp32 [n] added to every row (conv bias fold) or NULL. */
int b200sd_linear_small(const float* x, const void* wgt, const float* bias, const float* add, float* out,
                        int32_t m, int32_t n, int32_t k, int32_t act_in, int32_t act_out, void* stream);

/* sinusoidal timestep embedding (unet.py:703-728; flip_sin_to_cos: cos first): out fp32 [m, dim] */
int b200sd_timestep_embedding(const float* timesteps, float* out, int32_t m, int32_t dim,
                              int32_t flip_sin_to_cos, float freq_shift, void* stream);

/* ---- normalisation ------------------------------------------------------------------------
 * GroupNorm (torch.nn.GroupNorm, unet.py:430,448,528,966) on NHWC fp16, fp32 statistics, optional
 * fused SiLU (unet.py:472-473,480-481), reading one or two channel-concatenated sources and writing
 * the concatenated normalised tensor (the torch.cat of unet.py:215,270 never materialises raw).
 * One launch on thread-block clusters: a cluster owns one (image, channel chunk), keeps its pixels in shared
 * memory, computes exact two-pass statistics exchanged through DSMEM and normalises from the slab.  Tensors too
 * large for that (slab > 200 KB per CTA) take two launches (chunk partials in `stats_ws`, then apply). */
int b200sd_group_norm(const void* x0, const void* x1, int32_t c0, int32_t c1, int32_t n_img, int32_t hw,
                      int32_t groups, float eps, const float* gamma, const float* beta, int32_t silu,
                      void* out, float* stats_ws, size_t stats_ws_bytes, void* stream);
size_t b200sd_group_norm_workspace_bytes(int32_t n_img, int32_t hw, int32_t c, int32_t groups);
/* GroupNorm (+SiLU, + concat) from PRODUCER-SIDE statistics: chan0 / chan1 are the per-channel (sum, sum of squares)
 * [n_img][c][2] a b200sd_gemm call left behind (cs_chan); no statistics pass, one read + one write of the tensor.  Used
 * where the consumer is not the halo convolution (which applies the normalisation in its own operand path). */
int b200sd_group_norm_apply(const void* x0, const void* x1, int32_t c0, int32_t c1, int32_t n_img, int32_t hw,
                            int32_t groups, float eps, const float* chan0, const float* chan1, const float* gamma,
                            const float* beta, int32_t silu, void* out, void* stream);

/* LayerNorm over channels of a token matrix [rows, c] (LayerNormANE, layer_norm.py:51-80, in the
 * x_hat*w+b convention of the checkpoint, cf. unet.py:132-138). */
int b200sd_layer_norm(const void* x, const float* gamma, const float* beta, void* out, int32_t rows,
                      int32_t c, float eps, void* stream);

/* row softmax of fp32 scores [rows, cols] -> fp16 probabilities, exp2 domain; used only for the VAE
 * decoder's single-head d=512 mid-block attention (diffusers AutoencoderKL via torch2coreml.py:584-594),
 * whose Q K^T and P V products run on b200sd_gemm. */
int b200sd_softmax_rows(const float* in, void* out, int32_t rows, int32_t cols, float scale, void* stream);

/* ---- attention ------------------------------------------------------------------------------
 * softmax(q k^T / sqrt(d) [+ mask]) v per (batch, head): attention.py:24-168 (all three
 * AttentionImplementations compute this function) via Einsum (unet.py:45-59).
 * q [batch, sq, ldq] / k,v [batch, sk, ldk] fp16 token-major with head h in columns
 * [h*d, (h+1)*d) of the given base pointers; out [batch, sq, ldo].  d must be 64.
 * mask: optional fp32 additive [batch, sk] (unet.py:99-114) or NULL.
 * impl: 0 ORIGINAL, 1 SPLIT_EINSUM, 2 SPLIT_EINSUM_V2 (tile policy only; same result);
 *       | 0x100 adds the causal mask of the CLIP text encoder (key j visible to query i iff j <= i). */
int b200sd_attention(const void* q, const void* k, const void* v, void* out, const float* mask,
                     int32_t batch, int32_t heads, int32_t sq, int32_t sk, int32_t d,
                     int32_t ldq, int32_t ldk, int32_t ldv, int32_t ldo, float scale, int32_t impl,
                     void* stream);
/* The same with a caller-provided device workspace of b200sd_attention_workspace_bytes() bytes, which lets the launch
 * cut the (query tile x K/V tile) work into equal per-CTA ranges ("stream-K") when whole query tiles would fill the GPU
 * badly (S = 4096: 320 tiles on 296 CTA slots).  Pieces of a split tile meet in the workspace and are merged in a fixed
 * order, so results are reproducible.  The workspace must be zero-filled once before its first use (the kernel leaves its
 * counters at zero) and must not be shared with a concurrently running attention launch. */
size_t b200sd_attention_workspace_bytes(void);
int b200sd_attention_ws(const void* q, const void* k, const void* v, void* out, const float* mask,
                        int32_t batch, int32_t heads, int32_t sq, int32_t sk, int32_t d,
                        int32_t ldq, int32_t ldk, int32_t ldv, int32_t ldo, float scale, int32_t impl,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- layout / elementwise ----------------------------------------------------------------- */
/* NCHW (fp16 or fp32) -> NHWC fp16 with channel padding to c_pad (zeros) */
int b200sd_nchw_to_nhwc(const void* in, int32_t in_f32, void* out, int32_t n, int32_t c, int32_t h,
                        int32_t w, int32_t c_pad, void* stream);
/* NHWC fp32/fp16 [n,h,w,c_pad] -> NCHW fp32 [n,c,h,w] (first c channels) */
int b200sd_nhwc_to_nchw_f32(const void* in, int32_t in_f32, float* out, int32_t n, int32_t c, int32_t h,
                            int32_t w, int32_t c_pad, void* stream);
/* nearest x2 upsample NHWC fp16 (F.interpolate, unet.py:499) */
int b200sd_upsample2x(const void* in, void* out, int32_t n, int32_t h, int32_t w, int32_t c, void* stream);
/* out = a + b (fp16; ControlNet residual injection unet.py:1009-1022) */
int b200sd_add(const void* a, const void* b, void* out, size_t numel, void* stream);
/* BC1S fp16/fp32 context (B, D, 1, S) -> token-major fp16 [B*S, D] */
int b200sd_ctx_to_tokens(const void* in, int32_t in_f32, void* out, int32_t b, int32_t d, int32_t s,
                         void* stream);

/* CLIP text-encoder input embeddings (transformers CLIPTextEmbeddings as called through pipeline.py:151-175):
 * out[b*s + t, :] = token_embedding[ids[b, t]] + position_embedding[t]; ids float32 [batch, s]; tables fp16 */
int b200sd_embed_tokens(const float* ids, const void* token_embedding, const void* position_embedding, void* out,
                        int32_t batch, int32_t s, int32_t d, int32_t vocab, void* stream);

/* ---- CFG + scheduler step (single fused elementwise kernel) -------------------------------
 * eps = eps_u + g (eps_c - eps_u)           (pipeline.py:559-562; performGuidance
 *                                            StableDiffusionPipeline.swift:469-483)
 * then one scheduler update written as a linear combination
 *     x_prev = cx * x + ce * eps' + sum_i ch[i] * hist[i]
 *     x0     = x0_cx * x + x0_ce * eps' + sum_i x0_ch[i] * hist[i]     (denoised estimate)
 * whose fp32 coefficients the host derives per step for DDIM (eta=0), DPM-Solver++(2M) and
 * PNDM/PLMS (Scheduler.swift:218-343, DPMSolverMultistepScheduler.swift:135-244).  `hist` is a
 * 4-slot ring of latent-sized fp32 buffers holding past eps' (PLMS `ets`), past x0
 * (DPM `modelOutputs`) or a saved sample (PLMS `currentSample`); all history reads of a step happen
 * before its pushes.  noise_pred: fp32 NCHW [2*n, c, h, w] (uncond batch first); latents fp32
 * [n, c, h, w] updated in place; `unet_in` (fp16 NHWC [2n, h, w, c_pad], may be NULL) receives the
 * duplicated next UNet input (pipeline.py:502: np.concatenate([latents] * 2)). */
typedef struct {
    float guidance;
    float cx, ce;
    float ch[4];
    float x0_cx, x0_ce;
    float x0_ch[4];
    int32_t n_hist;          /* history slots read this step (0..4) */
    int32_t push_eps_slot;   /* >= 0: hist[slot] = eps'  */
    int32_t push_x0_slot;    /* >= 0: hist[slot] = x0    */
    int32_t push_x_slot;     /* >= 0: hist[slot] = x (sample before this update) */
    int32_t noise_pred_nhwc; /* 1: noise_pred is NHWC fp32 [2*n, h, w, c] (the UNet's conv_out epilogue output, no
                                layout kernel in between); 0: NCHW */
} b200sd_step_coeffs;

int b200sd_cfg_scheduler_step(const float* noise_pred, float* latents, float* hist /* [4][numel] */,
                              float* denoised /* x0 out or NULL */, void* unet_in, int32_t c_pad,
                              int32_t n, int32_t c, int32_t h, int32_t w,
                              const b200sd_step_coeffs* coeffs /* host */, void* stream);

/* ---- sampler step: the CFG + scheduler step above, extended for the sigma-space and stochastic samplers ----
 * (EulerDiscrete, EulerAncestralDiscrete, LMSDiscrete, DDIM with eta > 0; pipeline.py:504-508 scale_model_input)
 *     x_prev  = <the linear update of b200sd_step_coeffs> + noise_scale * z
 *     unet_in = fp16(in_scale * x_prev)     (in_scale: the NEXT step's c_in = 1 / sqrt(sigma^2 + 1))
 * z is a standard normal from Philox-4x32-10 keyed by rng_key[0..1] (device memory, so a new seed needs no graph
 * recapture), counter (noise_draw + b, 0, element index within image b, 0), Box-Muller on the first two words in
 * double precision rounded once to fp32: the stream of the Swift pipeline's nvidiaRNG (rng.py NvRandomSource), so
 * draw d of this kernel equals the d-th normal_array() call of a NvRandomSource with the same seed.
 * noise_pred == NULL selects the input-only mode: unet_in = fp16(in_scale * latents), nothing else is read or written
 * (the first UNet input of a loop).  With in_scale == 1 and noise_scale == 0 the arithmetic is that of
 * b200sd_cfg_scheduler_step, bit for bit.  rng_key may be NULL when noise_scale == 0. */
typedef struct {
    b200sd_step_coeffs step;
    float in_scale;          /* multiplies the value written to unet_in */
    float noise_scale;       /* 0: no noise term */
    uint32_t noise_draw;     /* Philox counter word 0 of image 0; image b uses noise_draw + b */
} b200sd_sampler_coeffs;

int b200sd_sampler_step(const float* noise_pred /* or NULL: input-only mode */, float* latents,
                        float* hist /* [4][numel] */, float* denoised /* x0 out or NULL */, void* unet_in,
                        int32_t c_pad, int32_t n, int32_t c, int32_t h, int32_t w,
                        const b200sd_sampler_coeffs* coeffs /* host */, const uint32_t* rng_key /* device, 2 words */,
                        void* stream);

/* VAE decoder input: out = post_quant_conv(z * inv_scale) as NHWC fp16 padded to c_pad channels
 * (pipeline.py:313-316 `z / 0.18215`; torch2coreml.py:590-594 post_quant_conv); z fp32 NCHW, c <= 8,
 * w fp32 [c, c], b fp32 [c]. */
int b200sd_latent_prep(const float* z, const float* w, const float* b, float inv_scale, void* out, int32_t n,
                       int32_t c, int32_t h, int32_t wd, int32_t c_pad, void* stream);

/* VAE post-process: clip(x/2+0.5,0,1) (pipeline.py:317) NHWC fp16/32 -> NHWC fp32 [n,h,w,3] and/or u8 */
int b200sd_image_postprocess(const void* in, int32_t in_f32, int32_t c_pad, float* out_f32, uint8_t* out_u8,
                             int32_t n, int32_t h, int32_t w, int32_t c, void* stream);

/* ================================================================================================================
 * Model-level handles: one "predict" per model, like the reference's device boundary.
 *
 * The op-level entry points above are what the hot path is made of; a host that is not Python should not have to
 * re-implement the launch graph.  A handle owns the packed weights (given once, in the reference's own parameter names
 * and layouts: the diffusers UNet2DConditionModel state dict the reference loads unchanged, unet.py:121-146 /
 * torch2coreml.py:915-918), the activation arena, the statistics buffers and the launch sequence; per call only device
 * pointers go in.  Replaces `CoreMLModel.__call__` for the unet (coreml_model.py:118-120, tensor names
 * pipeline.py:531-536) and `Unet.predictNoise` (swift/StableDiffusion/pipeline/Unet.swift:90-144).
 * Not thread-safe: one handle per stream / thread (the reference serialises per model, ManagedMLModel.swift:23-66). */
typedef struct b200sd_unet b200sd_unet;

typedef struct {
    const char* name;     /* diffusers key, e.g. "down_blocks.0.resnets.0.conv1.weight" */
    const void* data;     /* HOST pointer, row-major */
    int32_t dtype;        /* 0 = fp16, 1 = fp32 */
    int32_t ndim;         /* 1..4; linear weights may be [out, in] or [out, in, 1, 1] */
    int64_t shape[4];
} b200sd_weight;

typedef struct {
    /* architecture (the keys of the reference's UNet config, unet.py:733-800) */
    int32_t in_channels, out_channels, layers_per_block, norm_num_groups, cross_attention_dim;
    float norm_eps;
    int32_t n_blocks;                 /* len(block_out_channels) */
    int32_t block_out_channels[8];
    int32_t attention_heads[8];       /* `attention_head_dim` of the reference = number of heads (unet.py:929) */
    int32_t transformer_layers[8];    /* transformer_layers_per_block, per down block */
    int32_t mid_transformer_layers;
    int32_t down_cross_attn[8];       /* 1: CrossAttnDownBlock2D, 0: DownBlock2D */
    int32_t up_cross_attn[8];         /* 1: CrossAttnUpBlock2D, 0: UpBlock2D (in up-block order) */
    int32_t flip_sin_to_cos;
    float freq_shift;
    int32_t addition_embed_text_time; /* SDXL `text_time` conditioning (unet.py:1051-1152) */
    int32_t addition_time_embed_dim, projection_class_embeddings_input_dim;
    int32_t num_time_ids;             /* 6 (SDXL base), 5 (refiner); 0 = 6 */
    int32_t support_controlnet;       /* forward accepts additional_residuals (unet.py:1009-1022) */
    /* geometry the handle is built for */
    int32_t batch, height, width, seq_len;   /* UNet batch (2 x images), latent height / width, text tokens */
} b200sd_unet_config;

/* Packs the weights (fp16, tiled per call site, LayerNorm folded into its consumer GEMMs), runs one sizing pass and
 * allocates the activation arena.  `stream`: the stream the sizing pass runs on. */
int b200sd_unet_create(const b200sd_unet_config* cfg, const b200sd_weight* weights, int32_t n_weights, void* stream,
                       b200sd_unet** out);
/* Optional per-prompt prologue: cross-attention K / V of every block from encoder_hidden_states (fp16 device
 * (batch, cross_attention_dim, 1, seq_len)); later forwards may then pass encoder_hidden_states = NULL. */
int b200sd_unet_prepare_prompt(b200sd_unet* h, const void* encoder_hidden_states, void* stream);
/* noise_pred = UNet(sample, timestep, encoder_hidden_states [, time_ids, text_embeds][, additional_residual_i]).
 * All pointers are DEVICE pointers: sample NCHW fp16 (or fp32 with sample_f32) (batch, in_channels, h, w); timesteps
 * fp32 [batch]; encoder_hidden_states fp16 BC1S or NULL after b200sd_unet_prepare_prompt; time_ids fp32 (batch,
 * num_time_ids) and text_embeds fp32 (batch, pooled) for SDXL, else NULL; additional_residuals: NULL or an array (host)
 * of device pointers to the fp16 NCHW ControlNet residuals in controlnet.py:218-229 order; noise_pred fp32 NCHW. */
int b200sd_unet_forward(b200sd_unet* h, const void* sample, int32_t sample_f32, const float* timesteps,
                        const void* encoder_hidden_states, const float* time_ids, const float* text_embeds,
                        const void* const* additional_residuals, float* noise_pred, void* stream);
/* the reference's attention switch (unet.py:33-39): 0 ORIGINAL, 1 SPLIT_EINSUM, 2 SPLIT_EINSUM_V2 (same result) */
int b200sd_unet_set_attention_impl(b200sd_unet* h, int32_t impl);
/* bytes of activation arena + scratch the handle holds (weights excluded) */
size_t b200sd_unet_device_bytes(const b200sd_unet* h);
void b200sd_destroy(b200sd_unet* h);

#ifdef __cplusplus
}
#endif
#endif /* B200SD_H */
