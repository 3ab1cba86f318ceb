/*
 * libia2p_sm100a.so -- C ABI of the B200-native InstructAny2Pix denoising hot path.
 *
 * The reference (jacklishufan/InstructAny2Pix) has no FFI: its hot path is Python calling
 * torch / diffusers library ops.  Each entry point below therefore cites the reference
 * *operation sequence* it replaces (file:line under the reference root).  The Python host
 * (instructany2pix_b200/) binds these with ctypes; INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  All pointers are DEVICE pointers unless noted.
 *   - Return value: 0 = OK; < 0 = argument error (IA2P_E_*); > 0 = cudaError_t of the failing call.
 *     ia2p_last_error() returns a thread-local message for the last non-zero return.
 *   - Caller (PyTorch) owns every buffer; the library allocates nothing user-visible and keeps
 *     no pointer after return.  All work is enqueued on `stream` (a cudaStream_t); no host sync.
 *   - No CPU fallback: every launcher fails with IA2P_E_DEVICE unless the device is sm_100.
 *   - Activations are bf16 NHWC ("tokens x channels" row-major); dtype codes: IA2P_F32/BF16/F16.
 */
#ifndef IA2P_H_
#define IA2P_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { IA2P_F32 = 0, IA2P_BF16 = 1, IA2P_F16 = 2 };
enum { IA2P_E_ARG = -1, IA2P_E_DEVICE = -2, IA2P_E_SHAPE = -3, IA2P_E_ALIGN = -4, IA2P_E_DRIVER = -5 };
/* GEMM epilogues.  GELU (exact erf, the GEGLU gate's evaluation) and QUICK_GELU (x * sigmoid(1.702 x), CLIP's quick_gelu) act on
 * the LN-corrected accumulator plus bias; they need bf16 output and no residual / rowbias / LN-producer or column statistics. */
enum { IA2P_EPI_NONE = 0, IA2P_EPI_GEGLU = 1, IA2P_EPI_GELU = 2, IA2P_EPI_QUICK_GELU = 3 };
enum { IA2P_ACT_NONE = 0, IA2P_ACT_GELU_NEW = 1, IA2P_ACT_SILU = 2 };

int ia2p_version(void);
const char* ia2p_last_error(void);
/* 0 if `device` (ordinal, -1 = current) is compute capability 10.x, else IA2P_E_DEVICE. */
int ia2p_device_check(int device);

/* ---------------------------------------------------------------- sampler epilogues (HBM-bound) */

/* CFG combine + DDIM update in one pass.
 * Replaces: eps.chunk(2); eps_u + g*(eps_c - eps_u); scheduler.step(); cat([x]*2)
 *   diffusion/ip_adapter/custom_pipelines.py:332-357 (= ddim/sdxl_pipeline.py:826-850), [3P] DDIMScheduler.step.
 * eps2: [2*batch, n] (uncond half FIRST), x: [batch, n]; x_out = c_x*x + c_e*(eps_u + g*(eps_c-eps_u)).
 * x_in_next2 (nullable): [2*batch, n] receives x_out duplicated (next UNet input).  n % 4 == 0. */
int ia2p_cfg_ddim_step(const void* eps2, int eps_dtype, const void* x, void* x_out, int x_dtype,
                       void* x_in_next2, int xin_dtype, int64_t batch, int64_t n,
                       float g, float c_x, float c_e, void* stream);

/* ia2p_cfg_ddim_step with one guidance scale per request: sample b (rows b and batch + b of eps2) uses g[b].
 * Replaces the same sequence as ia2p_cfg_ddim_step for a batch of requests that each carry their own `cfg`
 * (pipeline.py:303-304 takes it per request; [3P] StableDiffusionXLPipeline applies one float to the batch).
 * g: fp32 [batch], DEVICE memory, read when the kernel runs (a CUDA graph replays whatever it holds then).
 * Results for sample b are bitwise those of ia2p_cfg_ddim_step with g = g[b]. */
int ia2p_cfg_ddim_step_rows(const void* eps2, int eps_dtype, const void* x, void* x_out, int x_dtype,
                            void* x_in_next2, int xin_dtype, int64_t batch, int64_t n,
                            const float* g, float c_x, float c_e, void* stream);

/* CFG combine + linear scheduler update with every coefficient per row (continuous batching: each batch row is a slot at its own
 * position in its own schedule).  g, c_x, c_e: fp32 [batch], DEVICE memory, read when the kernel runs.  Row b of x_out is bitwise
 * ia2p_cfg_ddim_step with the scalars (g[b], c_x[b], c_e[b]); g = 0, c_x = 1, c_e = 0 leaves a finite row unchanged.
 * x_in_next (nullable, with s_in fp32 [batch] on the device): [batch, n] receives s_in[b] * x_out, the row's next UNet input
 * (Euler's x / sqrt(sigma_next^2 + 1)), bitwise ia2p_axpby(x_out, x_out, s_in[b], 0) for finite values.  NOT duplicated. */
int ia2p_cfg_step_coef_rows(const void* eps2, int eps_dtype, const void* x, void* x_out, int x_dtype,
                            void* x_in_next, int xin_dtype, int64_t batch, int64_t n,
                            const float* g, const float* c_x, const float* c_e, const float* s_in, void* stream);

/* The step's blocked time-embedding rowbias of an S-slot CFG batch, gathered from per-slot tables, then every slot's step counter
 * advanced (a second, one-block launch).  tables: fp32 [slots, rows, 2 * sumC], row k of slot s = what
 * time_rowbias_table(timesteps, pair, 2) gives for the slot's request at step k; coef_tables: fp32 [slots, rows, ncoef];
 * step: int32 [slots], the row each slot reads, +1 after the gather up to rows - 1 (the sentinel row an idle slot stays on).
 * rowbias: fp32 [2 * slots * sumC], blocked per ResnetBlock r as [2 * slots, C_r] (slot s owns rows s and slots + s);
 * coef: fp32 [ncoef, slots].  block_lo: HOST array [nblocks + 1] of the blocks' column offsets (0 = first, last = sumC);
 * nblocks <= 64.  All device arrays are read when the kernels run. */
int ia2p_rowbias_gather(const float* tables, const float* coef_tables, int* step, float* rowbias, float* coef,
                        int64_t slots, int64_t rows, const int64_t* block_lo, int64_t nblocks, int64_t ncoef, void* stream);

/* out = c_x*x + c_e*eps.  Replaces _backward_ddim, ddim/pnp_pipeline.py:73-85 (and DDIM step without CFG). */
int ia2p_axpby(const void* eps, int eps_dtype, const void* x, void* x_out, int x_dtype, int64_t n,
               float c_x, float c_e, void* stream);

/* Inpainting loop tail: out = (1 - mask) * (c_x * orig + c_e * noise) + mask * latents, fp32, mask [B,1,HW] broadcast over C.
 * Replaces `latents = (1 - init_mask) * scheduler.add_noise(image_latents, noise, t_next) + init_mask * latents` of the [3P]
 * StableDiffusionXLInpaintPipeline loop the reference reaches through gdino/lib.py:85-102 (subject_consistency, pipeline.py:366);
 * (c_x, c_e) = add_noise coefficients of the next timestep (DDIM: sqrt(a), sqrt(1-a); Euler: 1, sigma); noise NULL on the last step. */
int ia2p_inpaint_blend(const float* latents, const float* orig_latents, const float* noise, const float* mask, float* out,
                       int64_t B, int64_t C, int64_t HW, float c_x, float c_e, void* stream);

/* Start-latent blend: out = ll/|ll| * (alpha|x| + (1-alpha)|y|), ll = alpha x + (1-alpha) y, norms over all n elements, fp32.
 * Replaces InstructAny2PixPipeline.polar_intrtpolate, pipeline.py:295-300 (call site :332-336: inverted latent vs fresh noise).
 * workspace: ia2p_polar_workspace_bytes() bytes of device memory (per-block partial sums; bit-reproducible, no atomics). */
int64_t ia2p_polar_workspace_bytes(void);
int ia2p_polar_interpolate(const float* x, const float* y, float* out, int64_t n, float alpha, void* workspace, void* stream);

/* out[b,c,p] = scale * (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise), moments = [B, 2C, HW] (mean | logvar), fp32.
 * Replaces [3P] DiagonalGaussianDistribution.sample() * scaling_factor at ddim/pnp_pipeline.py:201-204.  noise NULL -> the mode. */
int ia2p_gaussian_sample(const float* moments, const float* noise, float* out, int64_t B, int64_t C, int64_t HW, float scale,
                         void* stream);

/* Prior: x0->eps transform + CFG (cond half FIRST) + DDPM ancestral step, fp32.
 * Replaces prior/model.py:641-648 (get_eps :208-239, CFG :643-644, [3P] DDPMScheduler.step).
 * x0_pair: [2, n] = model output for (cond, uncond); x: [n]; noise: [n] or NULL (sigma ignored). */
int ia2p_prior_cfg_ddpm_step(const float* x0_pair, const float* x, const float* noise, float* x_out, int64_t n,
                             float sqrt_a, float sqrt_1ma, float g, float c_x0, float c_x, float sigma, void* stream);

/* Sinusoidal embedding [3P get_timestep_embedding]: prior/model.py:565-568,613-614; UNet time_proj / add_time_proj.
 * t: fp32 [n]; out: [n, dim] rows = flip ? [cos,sin] : [sin,cos]; freq_i = exp(-ln(1e4) * i / (dim/2 - shift)). */
int ia2p_timestep_embedding(const float* t, int64_t n, int dim, int flip_sin_to_cos, float shift,
                            void* out, int out_dtype, void* stream);

/* nearest 2x upsample, NHWC (fp32|bf16 in) -> bf16 out (conv operand).  Replaces F.interpolate in [3P] Upsample2D. */
int ia2p_upsample2x_nhwc(const void* x, int x_dtype, void* y, int64_t batch, int64_t h, int64_t w, int64_t c, void* stream);

/* y(bf16) = x (fp32|bf16|fp16): makes a tensor-core operand from a stream tensor (Downsample2D input).  n % 8 == 0. */
int ia2p_cast_to_bf16(const void* x, int x_dtype, void* y, int64_t n, void* stream);

/* ---------------------------------------------------------------- normalisation (HBM-bound) */

/* GroupNorm over NHWC bf16, optionally over the channel-concat of two tensors, optional fused SiLU.
 * Replaces [3P] ResnetBlock2D norm1/norm2 + SiLU, torch.cat([h, skip], 1), Transformer2DModel.norm, conv_norm_out.
 * xa: [batch, hw, ca], xb: [batch, hw, cb] or NULL, both x_dtype (fp32|bf16); y: [batch, hw, ca+cb] bf16;
 * raw (nullable): [batch, hw, ca+cb] bf16 receives the un-normalised concat (operand of the fused 1x1 shortcut conv).
 * workspace: ia2p_groupnorm_workspace_bytes() of scratch (per-slab partial sums; results are bit-reproducible:
 * no atomics).  (ca+cb) % groups == 0, ca % 8 == cb % 8 == 0, ca+cb <= 4096.
 * cs_a / cs_b (nullable; both or neither when xb is given): the producers' column statistics (see `colstats` below) with
 * cs_*_segments segments of batch * hw / 128 / segments tiles each; when given, the statistics pass over x is replaced by a
 * reduction of those (hw % (128 * segments) == 0 required). */
int ia2p_groupnorm_nhwc(const void* xa, int64_t ca, const void* xb, int64_t cb, int x_dtype,
                        const float* gamma, const float* beta, void* y, void* raw,
                        int64_t batch, int64_t hw, int groups, float eps, int silu,
                        const float* cs_a, int64_t cs_a_segments, const float* cs_b, int64_t cs_b_segments,
                        void* workspace, void* stream);
int64_t ia2p_groupnorm_workspace_bytes(int64_t batch, int groups);

/* LayerNorm over the last dim; (in,out) dtypes: (bf16,bf16), (fp32,bf16) [UNet: fp32 stream -> bf16 operand], (fp32,fp32)
 * [prior].  Replaces [3P] BasicTransformerBlock.norm1/2/3 and GPT-2 ln_1/ln_2/ln_f.  cols % 8 == 0, cols <= 2048. */
int ia2p_layernorm(const void* x, int x_dtype, const float* gamma, const float* beta, void* y, int y_dtype,
                   int64_t rows, int64_t cols, float eps, void* stream);

/* CLIP text embeddings: out[r] = tok[ids[r]] + pos[r % T], fp32 [n*T, C] (the residual stream).  Replaces [3P] CLIPTextEmbeddings
 * (token_embedding + position_embedding, default position_ids).  ids int64 [n, T]; tok bf16 [V, C]; pos fp32 [P >= T, C].
 * An id outside [0, V) reads nothing and yields a NaN row.  out_bf16 / stats (nullable, together): the bf16 copy and per-row
 * (sum, sum of squares), stats [n*T][1][2]: the producer format of ia2p_gemm_ln_bf16, so layer 0's layer_norm1 folds into the QKV
 * GEMM like every other LayerNorm.  C % 8 == 0. */
int ia2p_clip_embed(const int64_t* ids, int64_t n, int64_t T, const void* tok, int64_t V, const float* pos, int64_t P,
                    int64_t C, float* out, void* out_bf16, float* stats, void* stream);

/* ---------------------------------------------------------------- tcgen05 GEMM / implicit-GEMM conv (tensor-bound) */

/* out[M, N(/2 if GEGLU)] = epilogue( [A | A2][M, K1+K2] @ W[N, K1+K2]^T ),  bf16 x bf16 -> fp32 (TMEM) -> bf16.
 * Replaces nn.Linear call sites: attention_processor.py:239-247,267-270,344-383,400 (to_q/k/v/out, to_k_ip/to_v_ip),
 * [3P] proj_in/proj_out, GEGLU proj (+chunk+gelu+mul when epilogue == IA2P_EPI_GEGLU: W rows pre-interleaved in
 * 32-row value/gate groups), ff.net.2, 1x1 conv_shortcut (A2 = second half of a skip concat).
 * bias fp32 [N] | NULL; rowbias fp32 [ceil(M/rows_per_batch), N] | NULL (per-image channel bias);
 * residual [M, ldr] bf16|fp32 (res_dtype) | NULL; out bf16|fp32 (out_dtype): the residual stream is kept in fp32 so that
 * only tensor-core operands are rounded to bf16.  K1 % 64 == K2 % 64 == 0, N % 32 == 0, lda/lda2/ldo/ldr % 8 == 0. */
int ia2p_gemm_bf16(const void* A, int64_t lda, int64_t K1, const void* A2, int64_t lda2, int64_t K2,
                   const void* W, void* out, int64_t ldo, int64_t M, int64_t N,
                   const float* bias, const float* rowbias, int64_t rows_per_batch,
                   const void* residual, int64_t ldr, int res_dtype, int out_dtype, int epilogue, void* stream);

/* GroupNorm statistics from the producer (`colstats`, nullable, fp32-output calls of ia2p_gemm_ln_bf16 / ia2p_conv3x3_nhwc_bf16 /
 * ia2p_conv_up2x_nhwc_bf16): [row tiles of 128 output pixels][N][2] receives each tile's per-column (sum, sum of squares), read
 * back from the epilogue's staged slices, so the GroupNorm that consumes the tensor (ia2p_groupnorm_nhwc, cs_a / cs_b) needs no
 * statistics pass over it.  Tiles follow the output pixel order (128 consecutive pixels; needs H*W % 128 == 0 to be usable by
 * GroupNorm); conv_up2x writes 4 segments, one per output parity. */

/* Split-K workspace for the tensor-core kernels (EXPERIMENT builds only: ia2p_tc_features() & 1; the shipped library accepts and
 * ignores it).  Problems with few output rows (fewer 128 x BLOCK_N tiles than half
 * the SMs: batch-1 512^2, single interactive requests) are otherwise bound by the latency of one tile's K loop; with a workspace
 * every tile is computed by up to 8 CTAs over disjoint k-ranges, the partial accumulators meet in `workspace` and split 0 adds them
 * in a fixed order (bit-reproducible) before the normal epilogue.  workspace: device memory, 256-byte aligned,
 * ia2p_tc_workspace_bytes() bytes, its first 16 KB ZEROED once by the caller (tile arrival counters, self-resetting); it stays
 * registered for this host thread until replaced (NULL clears) and must only be used by ONE stream at a time. */
int64_t ia2p_tc_workspace_bytes(void);
int ia2p_tc_features(void);   /* experiment paths compiled into this build: bit 0 split-K, bit 1 A-operand multicast (0 in the shipped library) */
int ia2p_set_tc_workspace(void* workspace, int64_t bytes);

/* Programmatic dependent launch for the launches this host thread makes from now on: 1 = every kernel is launched with
 * programmatic stream serialisation (its prologue -- and, in ia2p_gemm_smallm, its first weight loads -- overlap the tail of the
 * previous kernel of the stream), 0 = off, -1 = the IA2P_PDL environment default (off).  Returns the previous mode.  The embedding
 * prior (a chain of ~175 tiny dependent kernels per step, prior/model.py:624-626) turns it on around its trunk; the UNet step
 * measured no gain from it (profiles/README.md). */
int ia2p_set_pdl(int mode);

/* One-shot hint for the NEXT ia2p_gemm_* / ia2p_conv* call made by this host thread: that launch also pulls `bytes` of
 * `next_weights` (the weight matrix of the tensor-core launch that will follow it) into L2, so the following kernel's first
 * wave does not start on cold DRAM misses (each layer's weights are touched once per step and never survive in L2).  The
 * pointer is only read by the kernel that consumes the hint; pass NULL / 0 to clear.  Purely a performance hint. */
int ia2p_tc_prefetch_hint(const void* next_weights, int64_t bytes);

/* first dimension of a conv's `colstats` buffer for a [B, Ho, Wo] output grid (conv_up2x: per parity segment, on its input
 * grid), or 0 when a 128-pixel tile would span several images and the statistics must not be requested; GEMMs: ceil(M / 128). */
int64_t ia2p_conv_colstats_tiles(int64_t B, int64_t Ho, int64_t Wo);

/* ia2p_gemm_bf16 + LayerNorm folding (replaces [3P] BasicTransformerBlock.norm1/2/3 followed by to_q/k/v, attn2.to_q and
 * the GEGLU projection -- SURVEY A.3 -- without a separate normalisation pass):
 *   PRODUCER (a GEMM writing the fp32 residual stream): out_bf16 (row pitch ldo2) receives a bf16 copy of the output rows and
 *     stats_out[M][ia2p_gemm_ln_parts(M, N, K)][2] the per-row partial (sum, sum of squares) of every column half-tile.
 *   CONSUMER: A = those raw bf16 rows, W = bf16(W_linear * gamma) (host pre-scaled), ln_c1[n] = sum_k W[n,k], bias[n] must
 *     already contain W_linear @ beta; the epilogue applies  rstd[m] * (acc - mean[m] * ln_c1[n]) + bias[n]  (before GEGLU)
 *     with mean / rstd of row m reduced, in fixed order, from ln_stats[M][ln_parts][2]; normalised width = K1 + K2.
 * All LN arguments are optional (NULL / 0): then this is exactly ia2p_gemm_bf16. */
int ia2p_gemm_ln_bf16(const void* A, int64_t lda, int64_t K1, const void* A2, int64_t lda2, int64_t K2,
                      const void* W, void* out, int64_t ldo, int64_t M, int64_t N,
                      const float* bias, const float* rowbias, int64_t rows_per_batch,
                      const void* residual, int64_t ldr, int res_dtype, int out_dtype, int epilogue,
                      void* out_bf16, int64_t ldo2, float* stats_out, float* colstats,
                      const float* ln_stats, int64_t ln_parts, const float* ln_c1, float ln_eps, void* stream);
/* number of (sum, sumsq) partials per row a producer with N output columns writes */
int64_t ia2p_gemm_ln_parts(int64_t M, int64_t N, int64_t K);   /* depends on the tile width the producer picks for (M, N, K) */

/* 3x3 conv (pad 1, stride 1|2) on NHWC bf16 as implicit GEMM, with an optional fused 1x1 shortcut conv
 * (extra K range) over up to two raw sources, bias, per-image channel bias (time embedding) and residual.
 * Replaces [3P] ResnetBlock2D.conv1 (+ time_emb_proj add), conv2 (+ conv_shortcut + residual add),
 * Downsample2D.conv, Upsample2D.conv (SURVEY A.3).
 * x: [B,H,W,Cin]; w: [Cout, 9*Cin + sc_ca + sc_cb], K order = (ky,kx,cin) then shortcut channels;
 * sc_a/sc_b: [B,Ho,Wo,sc_c*] | NULL; out/residual: [B,Ho,Wo,Cout].  Cin, sc_c*, % 64 == 0; Cout % 32 == 0. */
int ia2p_conv3x3_nhwc_bf16(const void* x, int64_t B, int64_t H, int64_t W, int64_t Cin, int stride,
                           const void* w, const void* sc_a, int64_t sc_ca, const void* sc_b, int64_t sc_cb,
                           void* out, int out_dtype, int64_t Cout, const float* bias, const float* rowbias,
                           const void* residual, int res_dtype, float* colstats, void* stream);

/* Nearest-2x upsample + 3x3 pad-1 conv in one op ([3P] Upsample2D = F.interpolate(scale_factor=2, "nearest") -> conv; UNet up
 * blocks, VAE decoder): four 2x2 convs over the LOW-resolution map, one per output parity, with pre-summed weights
 * w4 [4][Cout][4*Cin] bf16 (instructany2pix_b200.packing.pack_conv3x3_up2x).  x [B,H,W,Cin] bf16 -> out [B,2H,2W,Cout] fp32. */
int ia2p_conv_up2x_nhwc_bf16(const void* x, int64_t B, int64_t H, int64_t W, int64_t Cin, const void* w4, void* out,
                             int64_t Cout, const float* bias, float* colstats, void* stream);

/* Stride-2 3x3 conv with padding only at the bottom / right (input index 2*o + k): the VAE encoder's Downsample2D
 * ([3P] diffusers: padding=0 after F.pad(x, (0,1,0,1)); reached from vae.encode at ddim/pnp_pipeline.py:195-204). */
int ia2p_conv3x3_s2_padend_nhwc_bf16(const void* x, int64_t B, int64_t H, int64_t W, int64_t Cin, const void* w,
                                     void* out, int out_dtype, int64_t Cout, const float* bias, void* stream);

/* conv_in: 3x3 pad 1 conv from NCHW (fp32|bf16|fp16, few channels) to NHWC (bf16|fp32).  w fp32 [Cout,Cin,3,3].
 * The input batch is read modulo `in_batch` (CFG duplication without cat([x]*2): custom_pipelines.py:332). */
int ia2p_conv_in_nchw(const void* x, int x_dtype, int64_t in_batch, int64_t B, int64_t H, int64_t W, int64_t Cin,
                      const float* w, const float* bias, void* out, int out_dtype, int64_t Cout, void* stream);
/* conv_in of the VAE encoder straight from an 8-bit image: x uint8 [B,H,W,Cin] is read as 2 * (q / 255) - 1 in fp32 (diffusers 0.26
 * VaeImageProcessor.preprocess of a PIL image, each step rounded separately), the same 3x3 pad 1 conv as ia2p_conv_in_nchw follows;
 * no fp32 image is stored.  -> NHWC (bf16|fp32). */
int ia2p_conv_in_u8_nhwc(const void* x, int64_t B, int64_t H, int64_t W, int64_t Cin, const float* w, const float* bias,
                         void* out, int out_dtype, int64_t Cout, void* stream);
/* conv_out: 3x3 pad 1 conv from NHWC bf16 to NCHW (fp32|bf16|fp16), Cout in {3, 4, 8} (UNet eps, VAE image, VAE moments).
 * w fp32 [Cout,3,3,Cin] (K order ky,kx,cin). */
int ia2p_conv_out_nhwc(const void* x, int64_t B, int64_t H, int64_t W, int64_t Cin,
                       const float* w, const float* bias, void* out, int out_dtype, int64_t Cout, void* stream);

/* out[b,c,p] = x[(b*HW + p)*ld + c] for c < C <= 8: the leading channels of an NHWC fp32 tensor as NCHW.  Second half of conv_out
 * when it runs on the tensor cores (ia2p_conv3x3_nhwc_bf16 with the output channels zero-padded to 32): [3P] UNet conv_out
 * (4 eps channels), VAE decoder conv_out (3) / encoder conv_out (8). */
int ia2p_nhwc_prefix_to_nchw(const float* x, int64_t ld, float* out, int64_t B, int64_t HW, int64_t C, void* stream);
/* The same three leading channels as an 8-bit image out uint8 [B,H,W,3]: q = round_half_even(clamp(v / 2 + 0.5, 0, 1) * 255) in
 * fp32, bit for bit diffusers 0.26's VaeImageProcessor.postprocess(output_type="pil") (denormalize, then numpy_to_pil); NaN -> 0.
 * B*HW % 16 == 0, ld % 4 == 0, 16-byte aligned x and out.  Replaces the NCHW copy when the caller wants 8-bit images. */
int ia2p_nhwc_prefix_to_u8_image(const float* x, int64_t ld, void* out, int64_t B, int64_t HW, void* stream);

/* 1x1 conv over <= 8 channels, NCHW fp32 -> NCHW fp32: out = scale * (w x) + bias.  Replaces [3P] AutoencoderKL.post_quant_conv
 * / quant_conv with the latent (un)scaling of ddim/sdxl_pipeline.py:866 and pnp_pipeline.py:204 folded into `scale`. */
int ia2p_conv1x1_nchw_small(const float* x, const float* w, const float* bias, float* out, int64_t B, int64_t Cin,
                            int64_t Cout, int64_t HW, float scale, void* stream);

/* ---------------------------------------------------------------- attention */

/* p = softmax(scale * scores) per row, fp32 [rows, cols] (pitch ld) -> bf16 (pitch ldo).  Middle step of the VAE's single-head,
 * 512-wide attention ([3P] AutoencoderKL mid_block.attentions.0: one SDPA over L*L tokens), run as GEMM -> softmax -> GEMM. */
int ia2p_softmax_rows_f32_bf16(const float* scores, int64_t ld, void* out, int64_t ldo, int64_t rows, int64_t cols,
                               float scale, void* stream);

/* Flash self-attention, head_dim 64, non-causal.  Replaces F.scaled_dot_product_attention at
 * attention_processor.py:259-261.  q/k/v: bf16, token (b*N + i) row at ptr + row*ld, head h at cols [64h, 64h+64). */
int ia2p_flash_self_attn_bf16(const void* q, const void* k, const void* v, int64_t ld,
                              void* out, int64_t ldo, int64_t batch, int64_t n_tokens, int heads,
                              float softmax_scale, void* stream);

/* Causal self-attention for short sequences, head_dim 64: key j is masked for query i when j > i (no padding mask: CLIP attends
 * over pad tokens causally).  Replaces CLIPAttention with its causal mask ([3P] transformers CLIPTextTransformer, reached through
 * StableDiffusionXLPipeline.encode_prompt at ip_adapter.py:320-342 and the refiner at pipeline.py:358-361).  Same operand layout
 * as ia2p_flash_self_attn_bf16 (q/k/v: strided views of one fused [n*T, 3C] QKV output); fp32 softmax, masked keys contribute
 * exactly 0.  1 <= T <= 128; q/k/v/out 16-byte aligned. */
int ia2p_causal_self_attn_bf16(const void* q, const void* k, const void* v, int64_t ld,
                               void* out, int64_t ldo, int64_t n, int64_t T, int heads,
                               float softmax_scale, void* stream);

/* Decoupled cross-attention: out = softmax(Q Kt^T) Vt + ip_scale * softmax(Q Ki^T) Vi in ONE kernel.
 * Replaces the two SDPA calls + add at attention_processor.py:371-373,387-389,397.
 * q: [batch*n_q, ldq]; k_text/v_text: [batch*n_text, ldkv]; k_ip/v_ip: [batch*n_ip, ldkv_ip] (n_ip may be 0:
 * plain AttnProcessor2_0 on attn2 after IPAdapter.disable(), ip_adapter.py:153-154).  n_text <= 128, n_ip <= 16. */
int ia2p_decoupled_cross_attn_bf16(const void* q, int64_t ldq,
                                   const void* k_text, const void* v_text, int64_t ldkv, int n_text,
                                   const void* k_ip, const void* v_ip, int64_t ldkv_ip, int n_ip, float ip_scale,
                                   void* out, int64_t ldo, int64_t batch, int64_t n_q, int heads,
                                   float softmax_scale, void* stream);

/* ia2p_decoupled_cross_attn_bf16 with one IP scale per batch row: row b is softmax(Q Kt^T) Vt + ip_scale[b] softmax(Q Ki^T) Vi.
 * Replaces the same attention_processor.py:371-397 sequence for a batch of requests that each set their own `scale`
 * (ip_adapter.py:306 calls set_scale(scale) per request).  ip_scale: fp32 [batch], DEVICE memory; a CFG call has
 * batch = 2B rows [uncond; cond] and takes cat([s, s]).  ip_scale[b] == 0 gives exactly the text-only row, and row b is
 * bitwise the row of ia2p_decoupled_cross_attn_bf16 with the scalar ip_scale[b]. */
int ia2p_decoupled_cross_attn_rows_bf16(const void* q, int64_t ldq,
                                        const void* k_text, const void* v_text, int64_t ldkv, int n_text,
                                        const void* k_ip, const void* v_ip, int64_t ldkv_ip, int n_ip, const float* ip_scale,
                                        void* out, int64_t ldo, int64_t batch, int64_t n_q, int heads,
                                        float softmax_scale, void* stream);

/* ---------------------------------------------------------------- prior (GPT-2 trunk, weight-streaming) */

/* out[M,N] fp32 = act(act_in(A)[M,K] @ W[N,K]^T + bias) + residual;  A fp32 (split hi/lo bf16 on the fly),
 * W bf16.  M small (any M; processed 32 rows at a time).  Replaces GPT-2 c_attn/c_proj/c_fc/mlp.c_proj
 * ([3P], called at prior/model.py:624-626), input_sequence_embed_linear (:331,:353), UNet time/add embedding
 * MLPs and time_emb_proj (SURVEY A.2 steps 1-2).  act_in: IA2P_ACT_NONE|IA2P_ACT_SILU applied to A on load.
 * K % 32 == 0, N % 8 == 0. */
int ia2p_gemm_smallm(const float* A, int64_t lda, const void* W, const float* bias, const float* residual, int64_t ldr,
                     float* out, int64_t ldo, int64_t M, int64_t N, int64_t K, int act_in, int act, void* stream);

/* causal multi-head attention for short sequences (T <= 32), head_dim 64, fp32.
 * qkv: [batch, T, 3*E] (q | k | v), out: [batch, T, E].  Replaces GPT2Attention ([3P], SURVEY A.8). */
int ia2p_causal_attn_small_f32(const float* qkv, float* out, int64_t batch, int64_t T, int heads, void* stream);

/* The whole GPT-2-medium trunk of ONE prior step (GPT2Model(inputs_embeds=seq)["last_hidden_state"][:, -1], [3P], called at
 * prior/model.py:624-626) as a single persistent cooperative kernel: wpe add, 24 x (LN1 -> c_attn -> causal attention -> c_proj +
 * residual -> LN2 -> c_fc + gelu_new -> c_proj + residual), ln_f of the last token.  seq: [B2, T, E] fp32; wpe: [>= T, E] fp32;
 * layer_ptrs: HOST array of 12 device pointers per layer (wqkv, wo, wfc, wpr as bf16 [out, in]; bqkv, bo, bfc, bpr, ln1 gamma,
 * ln1 beta, ln2 gamma, ln2 beta as fp32); out: [B2, E] fp32.  E = 1024, heads = 16, T <= 32, n_layer <= 30.  workspace: 256-byte
 * aligned, ia2p_prior_trunk_workspace_bytes(B2 * T) bytes, ZERO-INITIALISED ONCE by the caller (it holds the grid barrier state)
 * and then reused from call to call.  Results are bit-reproducible (fixed summation order, no atomics on data). */
int64_t ia2p_prior_trunk_workspace_bytes(int64_t rows);
int ia2p_prior_trunk(const float* seq, const float* wpe, const void* const* layer_ptrs, int n_layer, const float* lnf_g,
                     const float* lnf_b, int64_t B2, int64_t T, int64_t E, int heads, void* workspace, int64_t ws_bytes,
                     float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IA2P_H_ */
