/* dreamlab_b200 — C-ABI of the B200-native LCM denoise + VAE-decode hot path.
 *
 * This is the drop-in boundary below the `b200` worker (backends/b200_worker.py), which itself
 * implements the reference's `PipelineWorker` protocol (reference `backends/base.py:29-39`).
 * The reference has NO native interface for this path: its CUDA worker makes one call into the
 * third-party diffusers pipeline (reference `backends/cuda_worker.py:221-229`), which in turn
 * dispatches to cuDNN/cuBLAS/SDPA through torch.  Each entry point below therefore cites the
 * diffusers module / reference line whose arithmetic it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless noted;
 *   - activations are NHWC bf16, statistics / time embeddings / latents fp32;
 *   - every function enqueues on `stream` (a cudaStream_t passed as void*) and returns
 *     0 on success; non-zero -> text in dl_last_error().  Nothing allocates or synchronises,
 *     so every call is CUDA-graph capturable;
 *   - there is no CPU fallback: without a CUDA device / sm_100a every call fails.
 */
#ifndef DREAMLAB_B200_H
#define DREAMLAB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DL_ABI_VERSION 3

/* ---- library ---------------------------------------------------------------------------- */
int dl_abi_version(void);
const char* dl_last_error(void);           /* thread-local text of the last failure          */
int dl_device_sm_count(void);              /* SM count of the current device (148 on B200)   */

/* ---- implicit-GEMM conv / linear (tcgen05 + TMEM + TMA) ---------------------------------- *
 * Replaces torch.nn.Conv2d(3x3,s1,p1 | 1x1) and torch.nn.Linear inside diffusers'
 * ResnetBlock2D / Transformer2DModel / Attention projections / FeedForward(GEGLU) /
 * Upsample2D / AutoencoderKL decoder convs, reached from reference
 * `backends/cuda_worker.py:222` (UNet call mirrored at `backends/rknnlcm.py:588-593`,
 * VAE decode at `backends/rknnlcm.py:618`).                                                  */
enum {
  DL_EPI_BF16 = 0,      /* out bf16 [pixels, ldo]: acc*alpha + bias + rowadd + residual      */
  DL_EPI_GEGLU = 1,     /* weights interleaved (value,gate): out[:, j] = v_j * gelu(g_j)      */
  DL_EPI_F32 = 2,       /* out fp32 [pixels, ldo] (UNet conv_out -> noise_pred)               */
  DL_EPI_U8_IMAGE = 3,  /* VaeImageProcessor tail fused: clamp(x/2+.5,0,1)*255 -> u8 NHWC
                           (reference `backends/rknnlcm.py:220-235`)                          */
  DL_EPI_BF16_RELU = 4  /* as DL_EPI_BF16, then max(0, .) on the fp32 value before the bf16 store
                           (AutoencoderTiny decoder convs).  No gn_partial, row_stats_out, ln_*,
                           strided output or peer outputs.                                    */
};

typedef struct dl_igemm_desc {
  const void* a0;            /* source 0: NHWC bf16, channels [0,c0)                          */
  long long a0_pix_stride;   /* elements between consecutive pixels of a0 (>= c0)             */
  int c0;                    /* multiple of 64                                                */
  const void* a1;            /* optional source 1 (skip-concat partner), channels [c0,c0+c1)  */
  long long a1_pix_stride;
  int c1;                    /* 0 or multiple of 64                                           */
  int nimg, h, w;            /* activation extent; Linear over M rows: nimg=1, h=1, w=M       */
  int taps;                  /* 9: conv3x3 stride 1 pad 1;  1: conv1x1 / Linear;  4: one phase of
                                the nearest-2x-upsample+conv3x3 fold (see tap_phase)           */
  int tap_phase;             /* taps == 4: phase 2a+b -> output pixel (2y+a, 2x+b); else -1   */
  const void* wgt;           /* bf16 [n, taps*(c0+c1)], K index = tap*(c0+c1) + channel       */
  long long ldw;             /* weight row stride in elements; 0 = dense                      */
  int n;                     /* output channels                                               */
  void* out;
  long long ldo;             /* output row stride in elements                                 */
  long long out_x_stride;    /* optional strided output view (elements): between x neighbours, */
  long long out_y_stride;    /*   between rows, between images; 0 = dense (ldo, ldo*w, ldo*w*h) */
  long long out_img_stride;
  const float* bias;         /* [n] or NULL                                                   */
  const float* rowadd;       /* [nimg, ld_rowadd] per-image channel add (time emb) or NULL    */
  int ld_rowadd;
  const void* residual;      /* bf16 [pixels, ldr] or NULL (DL_EPI_BF16 only)                 */
  long long ldr;
  const void* identity;      /* 256x256 bf16 identity (dl_fill_identity); needed with residual:
                                the add runs on the tensor core as out += R . I                */
  int mode;                  /* DL_EPI_*                                                      */
  float alpha;               /* accumulator scale (0 -> 1)                                    */
  int bn;                    /* N tile (multiple of 16, <=256); 0 = auto                      */
  float* gn_partial;         /* optional: GroupNorm (sum, sumsq) records of the bf16 OUTPUT, fp32        */
  int gn_cpg;                /*   [nimg, gn_slots, n/gn_cpg, 2]; one slot per M tile of an image, written */
  int gn_slots, gn_slot0;    /*   at gn_slot0 + tile (folded-upsample phases use disjoint slot ranges);   */
  int gn_rows_per_img;       /*   channels per group 4/8/16/32.  Token-row GEMMs (nimg=1,h=1) give the
                                rows per image (multiple of 128); 0 for NHWC convs.  The records feed
                                dl_groupnorm_finalize: the consumer norm then reads its input once.   */
  void* peer_out[7];         /* all-gather fused into the GEMM (SDXL patch parallel, §8e X2): every output  */
  int n_peer_out;            /*   tile is ALSO TMA-stored into these peer-mapped buffers (same layout and
                                strides as `out`, which already points at this rank's row block); the caller
                                follows the launch with a dl_peer_allgather(nbytes = 0) barrier             */
  int in_rows;               /* halo-padded row strips (SDXL patch parallel, SURVEY.md §8e X1): a0/a1 */
  int in_row0;               /*   hold in_rows >= h rows per image and output row y reads input rows
                                y + dy + in_row0; 0/0 = dense (in_rows = h)                    */
  /* LayerNorm folded into the GEMMs around it (BasicTransformerBlock norm1/2/3, SURVEY.md K8): no LayerNorm pass.
     PRODUCER (the GEMM whose bf16 output is the LayerNorm input, DL_EPI_BF16): row_stats_out fp32
     [rows, row_stats_slots, 2] receives per-row (sum, sum of squares) partials of the output, one slot per
     (N tile, epilogue half): row_stats_slots = 2 * ceil(n / dl_igemm_plan_bn(desc)).
     CONSUMER (the GEMM that reads LayerNorm(x): weights pre-multiplied by gamma, W'[j,k] = W[j,k] gamma[k]):
     ln_stats = the producer's records of its A rows (ln_slots slots), ln_colsum[j] = sum_k W'[j,k],
     bias[j] = b[j] + sum_k beta[k] W[j,k]; the epilogue computes
       out = rstd_r * (acc - mean_r * ln_colsum[j]) + bias[j],  mean / rstd over the ln_c = K channels.   */
  float* row_stats_out;
  int row_stats_slots;
  const float* ln_stats;
  int ln_slots;
  const float* ln_colsum;
  int ln_c;
  float ln_eps;
} dl_igemm_desc;

int dl_igemm(const dl_igemm_desc* desc, void* stream);
/* the N tile dl_igemm will use for this descriptor (host only, no launch)                         */
int dl_igemm_plan_bn(const dl_igemm_desc* desc);
/* M tiles per image of an h x w conv (slots a gn_partial buffer needs); 0 if tiles span images   */
int dl_igemm_tiles_per_image(int h, int w);
/* fills a caller-owned 256x256 bf16 device buffer (128 KB) with the identity matrix            */
int dl_fill_identity(void* dst_bf16_256x256, void* stream);

/* ---- GroupNorm (+SiLU), NHWC bf16, optional two-source concat ---------------------------- *
 * Replaces torch.nn.GroupNorm + F.silu in ResnetBlock2D.norm1/norm2, conv_norm_out,
 * Transformer2DModel.norm and the VAE attention group_norm (SURVEY.md K7).  With x1 != NULL
 * the normalised output is the channel concat [x0 | x1] (UNet up-block `torch.cat`, K10).
 * `workspace` holds per-chunk partial statistics: >= dl_groupnorm_workspace_bytes().          */
size_t dl_groupnorm_workspace_bytes(int nimg, int groups);
int dl_groupnorm(const void* x0, int c0, const void* x1, int c1, int nimg, int hw, int groups,
                 float eps, const float* gamma, const float* beta, int apply_silu, void* out,
                 void* workspace, void* stream);

/* Split form for row-strip (patch-parallel) execution, SURVEY.md §8e exchange X3: `stats` gets
 * the strip's per-(image, group) (mean, M2) as fp32 [nimg, groups, 2]; the caller all-gathers the
 * records of all ranks into stats_all [nranks, nimg, groups, 2] (equal strips: hw pixels each);
 * dl_groupnorm_apply merges them in rank order and normalises the strip.  out_img_stride
 * (elements, 0 = dense) lets the result land inside a halo-padded buffer.  The workspace must
 * be zero-initialised once (>= dl_groupnorm_split_workspace_bytes()).                          */
/* (sum, sumsq) records [nimg, slots, groups, 2] from the producing dl_igemm -> (mean, M2) records
 * [nimg, groups, 2] for dl_groupnorm_apply (nranks = 1); fp64 accumulation in fixed order.      */
int dl_groupnorm_finalize(const float* partial, int nimg, int slots, int groups, long long count,
                          float* stats, void* stream);
/* Per-CHANNEL records (dl_igemm_desc.gn_cpg == 1: [nimg, slots, n, 2], any channels-per-group, e.g. the
 * UNet's 10 / 20 / 40) of one producer, or of the two producers of a channel concat [x0 | x1] (a group may
 * straddle them) -> stats fp32 [nimg, groups, 2] (mean, M2) for dl_groupnorm_apply(nranks = 1).
 * count = pixels per image x channels per group.                                                    */
int dl_groupnorm_finalize_channels(const float* part0, int slots0, int c0, const float* part1, int slots1,
                                   int c1, int nimg, int groups, long long count, float* stats, void* stream);
size_t dl_groupnorm_split_workspace_bytes(int nimg, int groups);
int dl_groupnorm_stats(const void* x0, int c0, const void* x1, int c1, int nimg, int hw, int groups,
                       float* stats, void* workspace, void* stream);
int dl_groupnorm_apply(const void* x0, int c0, const void* x1, int c1, int nimg, int hw, int groups,
                       float eps, const float* gamma, const float* beta, int apply_silu,
                       const float* stats_all, int nranks, void* out, long long out_img_stride,
                       void* stream);

/* ---- LayerNorm over the channel dim, bf16 rows (BasicTransformerBlock.norm1/2/3, K8) ------ */
int dl_layernorm(const void* x, long long rows, int c, float eps, const float* gamma,
                 const float* beta, void* out, void* stream);

/* ---- attention (diffusers Attention / AttnProcessor2_0, K5/K6) ---------------------------- *
 * q: bf16 [batch*sq, ldq]  head h at columns [h*dh_stride, h*dh_stride+d); k, v likewise over
 * [batch*skv, ld].  out: bf16 [batch*sq, ldo], head h at columns [h*d, (h+1)*d).
 * impl: DL_ATTN_TC = tcgen05 flash kernel (product path), DL_ATTN_SIMT = CUDA-core checker.
 * v_ones = 1: column d of every V head holds 1.0 (per-head stride >= ceil16(d+1)); the PV MMA
 * then accumulates the softmax denominator on the tensor core instead of the CUDA cores.       */
enum { DL_ATTN_TC = 0, DL_ATTN_SIMT = 1, DL_ATTN_SIMT_CAUSAL = 2 /* keys <= query: CLIP text tower */ };
int dl_attention(const void* q, long long ldq, const void* k, long long ldk, const void* v,
                 long long ldv, int dh_stride, void* out, long long ldo, int batch, int sq,
                 int skv, int heads, int d, float scale, int impl, int v_ones, void* stream);

/* Wide-head flash attention (one head, head dim d a multiple of 128 up to 512): the AutoencoderKL mid-block
 * attention (diffusers UNetMidBlock2D -> Attention, reached from reference `backends/rknnlcm.py:618` vae.decode and
 * `backends/cuda_worker.py` pipe.vae).  The head dim is split over two CTAs per query tile (a 128 x 512 fp32 output is
 * all of TMEM); nothing of size sq x skv touches HBM.  q/k/v/out bf16 rows; sq % 128 == 0, skv % 64 == 0.      */
int dl_attention_wide(const void* q, long long ldq, const void* k, long long ldk, const void* v,
                      long long ldv, void* out, long long ldo, int batch, int sq, int skv, int d,
                      float scale, void* stream);

/* debug aid: CTA (0,0,0) of the tcgen05 attention kernel writes per-tile clock stamps of its MMA
 * and softmax warps into this device buffer of 256 int64 (NULL switches tracing off).          */
int dl_debug_attention_trace(void* device_buf_i64_256);

/* ---- time / guidance embedding pieces (diffusers Timesteps + TimestepEmbedding, K9) ------- */
/* out[b, :] = [cos(t_b f_i), sin(t_b f_i)], f_i = exp(-ln(1e4) i/half)  (flip_sin_to_cos)     */
int dl_timestep_sinusoid(const float* t, int batch, int dim, float* out, void* stream);
/* out[m, n] = act_out( sum_k act_in(x[m,k]) * w[n,k] + bias[n] + add[m,n] ), x/out fp32,
 * w bf16 [n,k]; silu flags select the activations.  For the tiny (M <= 64) time-MLP GEMMs.    */
int dl_small_linear(const float* x, int m, int k, const void* w, const float* bias,
                    const float* add, int n, int silu_in, int silu_out, float* out, void* stream);

/* ---- data movement (K10): nearest-2x upsample, stride-2 im2col, latent packing ------------ */
int dl_upsample2x(const void* x, int nimg, int h, int w, int c, void* out, void* stream);
/* cols[n*ho*wo, 9*c] for conv3x3 stride 2 pad 1 (Downsample2D); K index = tap*c + channel     */
int dl_im2col_s2(const void* x, int nimg, int h, int w, int c, void* cols, void* stream);
/* same over a halo-padded strip: x holds in_rows rows per image, logical row y is input row
 * y + in_row0 (rows outside [0, in_rows) read as zero); h = logical rows of the strip           */
int dl_im2col_s2_halo(const void* x, int nimg, int in_rows, int in_row0, int h, int w, int c,
                      void* cols, void* stream);
/* same layout for the VAE encoder's Downsample2D(padding=0): F.pad(x, (0,1,0,1)) then conv3x3 stride 2
 * without padding, i.e. tap (ky,kx) of output (yo,xo) reads input (2yo+ky, 2xo+kx), zero past the last
 * row / column.  h, w even; output (h/2) x (w/2).                                               */
int dl_im2col_s2_pad01(const void* x, int nimg, int h, int w, int c, void* cols, void* stream);
/* bf16 [npix, cpad] <- mat . (fp32 NHWC [npix, cin] * scale) + vec, zero-padded to cpad channels
 * (feeds conv_in).  mat/vec: optional fp32 [cin,cin] / [cin] = the VAE post_quant_conv 1x1 and the
 * `latents / scaling_factor` of reference `backends/rknnlcm.py:614` (K13); NULL = identity.     */
int dl_pack_latent(const float* x, long long npix, int cin, int cpad, float scale,
                   const float* mat, const float* vec, void* out, void* stream);
/* fp32 scores [rows, cols] -> bf16 softmax rows (VAE mid-block attention, heads=1, d=512: the
 * QK^T / PV contractions run through dl_igemm)                                                  */
int dl_softmax_rows(const float* scores, long long rows, int cols, void* out, void* stream);
int dl_nchw_to_nhwc_f32(const float* x, int nimg, int c, int hw, float* out, void* stream);
int dl_nhwc_to_nchw_f32(const float* x, int nimg, int c, int hw, float* out, void* stream);

/* ---- LCM scheduler step (diffusers LCMScheduler.step, K11; call site mirrored at reference
 * `backends/rknnlcm.py:596-598`) -------------------------------------------------------------
 * x0 = (x - sqrt(1-a_t) eps)/sqrt(a_t); den = c_out x0 + c_skip x;
 * x' = sqrt(a_prev) den + sqrt(1-a_prev) noise   (noise == NULL on the final step: x' = den)  */
typedef struct dl_lcm_coeffs {
  float sqrt_alpha_t, sqrt_beta_t, c_skip, c_out, sqrt_alpha_prev, sqrt_beta_prev;
} dl_lcm_coeffs;
int dl_lcm_step(const float* eps, const float* x, const float* noise, float* x_next,
                float* denoised, long long n, const dl_lcm_coeffs* coeffs /* host */, void* stream);
/* dl_lcm_step_ex: the step of a model whose scheduler config sets prediction_type / clip_sample
 * (`LCMScheduler.from_config(model config)`).  x0 from the model output mo, in diffusers' op order:
 *   DL_PRED_EPSILON  x0 = (x - sqrt(1-a_t) mo)/sqrt(a_t)     (= dl_lcm_step, bit for bit)
 *   DL_PRED_V        x0 = sqrt(a_t) x - sqrt(1-a_t) mo        (v_prediction)
 *   DL_PRED_SAMPLE   x0 = mo
 * then, with clip_sample != 0, x0 = clamp(x0, -clip_sample_range, clip_sample_range); the rest as
 * dl_lcm_step.  Every mul / sub / div rounded on its own.                                        */
#define DL_PRED_EPSILON 0
#define DL_PRED_V 1
#define DL_PRED_SAMPLE 2
typedef struct dl_lcm_coeffs_ex {
  dl_lcm_coeffs k;
  int prediction_type;      /* DL_PRED_* */
  int clip_sample;
  float clip_sample_range;
} dl_lcm_coeffs_ex;
int dl_lcm_step_ex(const float* model_output, const float* x, const float* noise, float* x_next,
                   float* denoised, long long n, const dl_lcm_coeffs_ex* coeffs /* host */, void* stream);

/* ---- CLIP text tower pieces (the step before the hot path: diffusers `encode_prompt` ->
 * transformers CLIPTextModel; SURVEY.md §8f rank 2) ------------------------------------------------
 * out[i, :] = bf16(tok_emb[ids[i], :] + pos_emb[i % seq, :]);  dl_act_bf16 mode 0 = quick_gelu
 * x*sigmoid(1.702x) (CLIP-L), 1 = exact GELU (OpenCLIP bigG), elementwise over n bf16 values.    */
int dl_embed_tokens(const long long* ids, const void* tok_emb, const void* pos_emb, int n, int seq,
                    int vocab, int dim, void* out, void* stream);
int dl_act_bf16(const void* x, void* out, long long n, int mode, void* stream);

/* ---- tiled VAE decode (`pipe.vae.enable_tiling()`, reference `backends/cuda_worker.py:91`;
 * diffusers AutoencoderKL.tiled_decode / blend_v / blend_h, SURVEY.md App. A.4) -----------------
 * Tiles are fp32 NHWC images.  dl_tile_blend blends the first `extent` rows (vertical = 1) or
 * columns (vertical = 0) of tile b, in place, with the last `extent` rows / columns of tile a:
 *   b[k] = a[len_a - extent + k] * (1 - k/extent) + b[k] * (k/extent).
 * dl_image_crop_u8 writes the top-left crop_h x crop_w window of a tile into a u8 NHWC canvas
 * (dst already points at the window's first pixel) with the VaeImageProcessor denormalise.     */
int dl_tile_blend(const float* a, float* b, int nimg, int ha, int wa, int hb, int wb, int c,
                  int extent, int vertical, void* stream);
int dl_image_crop_u8(const float* src, int nimg, int hs, int ws, int c, int crop_h, int crop_w,
                     void* dst_u8, long long dst_row_stride, long long dst_img_stride, void* stream);

/* ---- classifier-free guidance combine of the doubled-batch UNet output (SDXL path:
 * `StableDiffusionXLPipeline.__call__` behind reference `backends/cuda_worker.py:532`) --------
 * out = eps_uncond + guidance_scale * (eps_text - eps_uncond), fp32, un-contracted            */
int dl_cfg_combine(const float* eps_uncond, const float* eps_text, float guidance_scale,
                   float* out, long long n, void* stream);

/* ---- sampler step of the guided-model samplers (diffusers EulerDiscreteScheduler (s_churn 0),
 * EulerAncestralDiscreteScheduler, DDIMScheduler (eta 0), DPMSolverMultistepScheduler (dpmsolver++, order 2,
 * midpoint)), classifier-free guidance fused in.  One linear form restates each class's `step`:
 *   e      = out_uncond + guidance_scale * (out_text - out_uncond)   (cfg_combine's roundings; out_text NULL: e = out_uncond)
 *   x0     = a_x x + a_e e, clamped to [-clip_sample_range, clip_sample_range] when clip_sample != 0
 *   x_next = c_x x + c_e e + c_0 x0 + c_1 x0_prev + c_n noise        (x0_prev / noise NULL: that term is left out)
 * The host computes the coefficients (scheduler.py) from the diffusers lines:
 *   Euler    pred_original_sample = sample - sigma * model_output (epsilon) |
 *            model_output * (-sigma / (sigma**2 + 1) ** 0.5) + sample / (sigma**2 + 1) (v_prediction);
 *            prev_sample = sample + (sample - pred_original_sample) / sigma * (sigma_next - sigma)
 *   Euler-a  as Euler with sigma_down for sigma_next, + noise * sigma_up
 *   DDIM     prev_sample = alpha_prod_t_prev ** 0.5 * pred_original_sample + (1 - alpha_prod_t_prev) ** 0.5 * pred_epsilon
 *            (pred_epsilon from the unclamped model output: c_x, c_e)
 *   DPM++    x_t = (sigma_t / sigma_s0) * sample - (alpha_t * (exp(-h) - 1)) * D0 - 0.5 * (alpha_t * (exp(-h) - 1)) * D1,
 *            D0 = m0, D1 = (1 / r0) * (m0 - m1): c_0 / c_1 on x0 and x0_prev
 * Every mul / add / sub is rounded on its own.  fp32 in and out; n % 4 == 0, operands 16-byte aligned.  x0 receives
 * the step's x0 (the next step's x0_prev, and `denoised`).                                                     */
typedef struct dl_sampler_coeffs {
  float a_x, a_e;
  float c_x, c_e, c_0, c_1, c_n;
  int clip_sample;
  float clip_sample_range;
} dl_sampler_coeffs;
int dl_sampler_step(const float* out_uncond, const float* out_text, float guidance_scale, const float* x,
                    const float* x0_prev, const float* noise, float* x_next, float* x0, long long n,
                    const dl_sampler_coeffs* coeffs /* host */, void* stream);

/* ---- run_job_with_latents tail: fp32 adaptive_avg_pool2d -> (8,8) -> fp16 NCHW ------------- *
 * (reference `backends/cuda_worker.py:297-304`).  lat: fp32 NHWC [nimg,h,w,c]; out: fp16
 * [nimg,c,8,8].  Any h, w >= 1: adaptive_avg_pool2d bins [floor(i*h/8), ceil((i+1)*h/8)).      */
int dl_latent_pool8(const float* lat, int nimg, int h, int w, int c, void* out_f16, void* stream);

/* ---- all-gather over NVLink peer memory (SDXL patch parallel, SURVEY.md §8e X1-X3) ---------------
 * One kernel: store the local message into slot `rank` of every peer's symmetric staging buffer
 * (peer-mapped pointers stage_ptrs[r], two halves of nranks * slot_bytes each), publish an epoch in
 * every peer's signal pad (flag_ptrs[r], >= nranks u32, zero-initialised), wait for all ranks and
 * copy the gathered half to dst [nranks, nbytes].  `state`: 3 zero-initialised u32 in local device
 * memory (epoch and two CTA counters); epochs advance on the device, so the call is CUDA-graph
 * safe.  Every rank of the group must issue the same sequence of calls.  nbytes = 0 (src / dst
 * may be NULL) is a pure barrier: "every rank's earlier kernels — e.g. a dl_igemm with peer_out —
 * have completed and their peer writes are visible".                                            */
int dl_peer_allgather(const void* src, void* dst, long long nbytes, void* const* stage_ptrs,
                      void* const* flag_ptrs, int nranks, int rank, long long slot_bytes, void* state,
                      void* stream);

/* ---- fp32 precision mode (reference `CUDA_DTYPE=fp32`, `backends/cuda_worker.py:55-61`) --------
 * The same operators with fp32 activations and weights on the CUDA cores (plain tiled kernels,
 * accurate expf / erff): they exist for the parity bar of the fp32 pipeline (noise_pred within
 * 1e-4), not for speed.  Same argument meaning as their bf16 namesakes; dl_igemm_f32 reads the
 * same descriptor (a0/a1/wgt/residual/out are float; bn ignored; channels multiples of 16).  It has
 * no fused statistics and no peer stores: a descriptor with gn_partial, row_stats_out, ln_stats or
 * n_peer_out > 0 is refused.                                                                   */
int dl_igemm_f32(const dl_igemm_desc* desc, void* stream);
int dl_groupnorm_f32(const float* x0, int c0, const float* x1, int c1, int nimg, int hw, int groups,
                     float eps, const float* gamma, const float* beta, int apply_silu, float* out,
                     void* stream);
int dl_layernorm_f32(const float* x, long long rows, int c, float eps, const float* gamma,
                     const float* beta, float* out, void* stream);
int dl_attention_f32(const float* q, long long ldq, const float* k, long long ldk, const float* v,
                     long long ldv, int dh_stride, float* out, long long ldo, int batch, int sq,
                     int skv, int heads, int d, float scale, int causal, void* stream);
int dl_pack_latent_f32(const float* x, long long npix, int cin, int cpad, float scale,
                       const float* mat, const float* vec, float* out, void* stream);
int dl_im2col_s2_f32(const float* x, int nimg, int h, int w, int c, float* cols, void* stream);
int dl_im2col_s2_pad01_f32(const float* x, int nimg, int h, int w, int c, float* cols, void* stream);
int dl_softmax_rows_f32(const float* scores, long long rows, int cols, float* out, void* stream);
int dl_small_linear_f32(const float* x, int m, int k, const float* w, const float* bias,
                        const float* add, int n, int silu_in, int silu_out, float* out, void* stream);

/* ---- narrow-output conv3x3 = 1x1 GEMM + tap sum (AutoencoderKL decoder conv_out, 128 -> 3) -----------------
 * y: fp32 [nimg,h,w,ldy] with y[q, t*nout + oc] = w[oc, tap t, :] . in[q, :] (one dl_igemm with taps = 1 and the
 * weight rows regrouped tap-major); out[p, oc] = bias[oc] + sum_t y[p + offset(t), t*nout + oc], zero padding.
 * out_u8 != 0: u8 NHWC with the VaeImageProcessor tail (as DL_EPI_U8_IMAGE); else fp32 NHWC.  nout <= 4.   */
int dl_conv_tapsum(const float* y, int nimg, int h, int w, int ldy, int nout, const float* bias, void* out,
                   int out_u8, void* stream);

/* ---- PNG files assembled on the device (B200_PNG=gpu) -------------------------------------------
 * Replaces the host-side `img.save(buf, format="PNG")` that ends every job (reference
 * `backends/cuda_worker.py:234-239`; 70-100 ms of zlib per 512x512 image and core).  img: u8 NHWC
 * [nimg,h,w,3]; out: u8 [nimg, out_stride], each row one complete PNG file of dl_png_stored_size(h,w)
 * bytes: 8-bit RGB, filter 0, zlib stream of stored deflate blocks, Adler-32 / CRC-32 computed by the
 * kernels.  out 4-byte aligned, out_stride a multiple of 4 and >= the size rounded up to 4;
 * workspace: dl_png_stored_workspace_bytes(nimg, h) bytes.  Deterministic (same pixels -> same bytes). */
long long dl_png_stored_size(int h, int w);
long long dl_png_stored_workspace_bytes(int nimg, int h);
int dl_png_stored(const void* img_u8, int nimg, int h, int w, void* out, long long out_stride,
                  void* workspace, void* stream);

/* ---- image-to-image (diffusers LatentConsistencyModelImg2ImgPipeline + AutoencoderKL.encode) -----------------
 * dl_pack_image_im2col: u8 RGB NHWC init image -> the im2col operand of the encoder's conv_in (3 -> 128, 3x3,
 * padding 1) as a 1x1 GEMM with K = 64: out[p, tap*3 + c] (tap = ky*3 + kx) = 2 * (u8 / 255) - 1 (IEEE division,
 * no contraction), 0 for taps outside the h x w window and for K >= 27.  row_stride / img_stride are in bytes, so a
 * tile window of a larger canvas is read in place (its border taps are zero, not the canvas' neighbour pixels).
 * out: bf16 (or fp32 for the _f32 variant) [nimg*h*w, 64], 16-byte aligned.
 * dl_vae_sample_latents: moments fp32 NHWC [n,h,w,8] (mean | logvar) -> latents fp32 NHWC [n,h,w,4]:
 *   logvar = clamp(logvar, -30, 20); std = expf(0.5 logvar); x0 = scaling_factor * (mean + std * eps_s);
 *   out = sqrt_alpha * x0 + sqrt_one_minus_alpha * eps_n       (every mul / add rounded on its own)
 * eps_s / eps_n fp32 NCHW [n,4,h,w] as drawn; mean_out (optional) receives the mean, NHWC [n,h,w,4].         */
int dl_pack_image_im2col(const void* img_u8, int nimg, int h, int w, long long row_stride, long long img_stride,
                         void* out, void* stream);
int dl_pack_image_im2col_f32(const void* img_u8, int nimg, int h, int w, long long row_stride,
                             long long img_stride, float* out, void* stream);
int dl_vae_sample_latents(const float* moments, const float* eps_s, const float* eps_n, int nimg, int h, int w,
                          float scaling_factor, float sqrt_alpha, float sqrt_one_minus_alpha, float* out,
                          float* mean_out, void* stream);

/* ---- inpainting (diffusers StableDiffusionInpaintPipeline with LCMScheduler) -------------------------------------
 * dl_pack_image_im2col_masked: dl_pack_image_im2col of the masked image: mask u8 [nimg, h, w] (row / image strides in
 *   bytes, so a tile window is read in place like the image); a pixel with m >= 128 reads as 0.0 (the normalised
 *   middle grey of image * (binarised mask < 0.5)) before the zero padding.
 * dl_inpaint_latent_mask: u8 full-resolution masks [nimg, 8h, 8w] -> fp32 latent mask [nimg, h, w]:
 *   out[n, i, j] = mask[n, 8i, 8j] >= 128 ? 1 : 0 (binarise at 0.5, then F.interpolate's default nearest).
 * dl_pack_latent_inpaint: the operand of a 9-channel UNet's conv_in, bf16 (or fp32 for _f32) [repeat*npix, 64]:
 *   channels 0-3 latents, 4 mask, 5-8 masked_image_latents, 9-63 zero; latents / masked fp32 NHWC [npix, 4],
 *   mask fp32 [npix]; the npix pixels are written `repeat` times (classifier-free guidance halves).
 * dl_lcm_step_inpaint: dl_lcm_step (same roundings) followed by the 4-channel UNet's blend, fp32 NHWC [npix, 4]:
 *   proper = last ? image_latents : sqrt_alpha * image_latents + sqrt_one_minus_alpha * noise0
 *   x_next = (1 - mask) * proper + mask * prev_sample      (every mul / add / sub rounded on its own)
 *   with (sqrt_alpha, sqrt_one_minus_alpha) the add_noise coefficients of the next timestep; noise (the step's draw)
 *   may be NULL on the last step, noise0 (the draw that made the starting latents) may be NULL when last != 0.   */
int dl_pack_image_im2col_masked(const void* img_u8, const void* mask_u8, int nimg, int h, int w, long long row_stride,
                                long long img_stride, long long mask_row_stride, long long mask_img_stride, void* out,
                                void* stream);
int dl_pack_image_im2col_masked_f32(const void* img_u8, const void* mask_u8, int nimg, int h, int w,
                                    long long row_stride, long long img_stride, long long mask_row_stride,
                                    long long mask_img_stride, float* out, void* stream);
int dl_inpaint_latent_mask(const void* mask_u8, int nimg, int h, int w, float* out, void* stream);
int dl_pack_latent_inpaint(const float* latents, const float* mask, const float* masked, long long npix, int repeat,
                           void* out, void* stream);
int dl_pack_latent_inpaint_f32(const float* latents, const float* mask, const float* masked, long long npix,
                               int repeat, float* out, void* stream);
int dl_lcm_step_inpaint(const float* eps, const float* x, const float* noise, const float* image_latents,
                        const float* noise0, const float* mask, float* x_next, float* denoised, long long npix,
                        const dl_lcm_coeffs* k, float sqrt_alpha, float sqrt_one_minus_alpha, int last,
                        void* stream);
/* dl_lcm_step_inpaint_ex: dl_lcm_step_inpaint with the x0 of dl_lcm_step_ex (prediction type, clamp).        */
int dl_lcm_step_inpaint_ex(const float* model_output, const float* x, const float* noise,
                           const float* image_latents, const float* noise0, const float* mask, float* x_next,
                           float* denoised, long long npix, const dl_lcm_coeffs_ex* k, float sqrt_alpha,
                           float sqrt_one_minus_alpha, int last, void* stream);

/* ---- tiny autoencoder (diffusers AutoencoderTiny / TAESD) decoder input -------------------------------------------
 * latents fp32 NHWC [npix, 4] -> the 64-channel operand of the decoder's first conv, bf16 (or fp32 for _f32)
 * [npix, 64]: channels 0-3 = tanh(x / 3) * 3 (IEEE division, tanhf, rounded multiply: DecoderTiny.forward's
 * `torch.tanh(x / 3) * 3`), channels 4-63 zero.  out 16-byte aligned.                                              */
int dl_taesd_latent_in(const float* latents, long long npix, void* out, void* stream);
int dl_taesd_latent_in_f32(const float* latents, long long npix, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DREAMLAB_B200_H */
