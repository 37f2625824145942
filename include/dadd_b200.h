/*
 * dadd_b200.h - C ABI of the B200 (sm_100a) kernels behind DADD's UNet-denoising hot path.
 *
 * The reference (umutdundar99/progressive-stable-diffusion) is pure Python and has no FFI; each entry
 * point below names the reference code it replaces (file:line relative to the reference tree).
 * Conventions (SURVEY.md section 8b):
 *   - plain pointers and sizes only; every pointer is DEVICE memory unless marked "host";
 *   - buffers are borrowed: they must stay alive until the work queued on `stream` has run;
 *   - work is queued on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream), nothing
 *     synchronises, so every call is CUDA-graph capturable;
 *   - return 0 on success, non-zero on error (never throws); dadd_last_error() returns the message of the
 *     calling thread's last failure;
 *   - dtype codes: DADD_F32 = 0, DADD_BF16 = 1, DADD_F16 = 2.
 */
#ifndef DADD_B200_H
#define DADD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DADD_F32 0
#define DADD_BF16 1
#define DADD_F16 2 /* IEEE half: same tensor-core rate as bf16, 3 more mantissa bits (profiles/r01_precision_experiment.txt) */

#define DADD_LAYOUT_NCHW 0 /* x[b][c][hw]  (the reference's tensors)                     */
#define DADD_LAYOUT_NHWC 1 /* x[b][hw][c]  (channels-last; what the B200 UNet runs in)    */

/* ABI version of this header (bumped on any signature change).  The host binding refuses a library whose
 * dadd_abi_version() differs from the DADD_ABI_VERSION it was written against. */
#define DADD_ABI_VERSION 15
int dadd_abi_version(void);
/* Message of the last failing call on this thread ("" if none). */
const char* dadd_last_error(void);
/* Number of kernels launched by this library since load / since the last reset (all threads). */
int64_t dadd_launch_count(void);
void dadd_reset_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * DDIM update fused with the optional classifier-free-guidance combine.
 * Replaces src/pipelines/inference/inference_pipeline_ip.py:427-430 (CFG) and :434-468 (x0, clamp, update)
 * and the copies at src/pipelines/evaluation/evaluation_pipeline.py:537-562.
 *   eps  = eps_uncond ? eps_uncond + guidance * (eps_cond - eps_uncond) : eps_cond
 *   x0   = clamp((x - sqrt_1mab_t * eps) / sqrt_ab_t, -clamp, +clamp)
 *   x    = is_last ? x0 : sqrt_ab_prev * x0 + eps_coef * eps (+ sigma * noise when noise != NULL)
 * Every operation is a separately rounded fp32 op (no FMA contraction): bit-exact with the reference's
 * eager fp32 tensor arithmetic.  x is updated in place.  eps_dtype applies to eps_cond and eps_uncond.
 */
int dadd_ddim_step(float* x, const void* eps_cond, const void* eps_uncond /* nullable */, int eps_dtype,
                   float guidance, float sqrt_ab_t, float sqrt_1mab_t, float sqrt_ab_prev, float eps_coef,
                   float sigma, const float* noise /* nullable */, float clamp, int is_last, int64_t n,
                   void* stream);

/* Same update with the per-step scalars read on the device, so that one captured CUDA graph can be replayed
 * for every step of the schedule.  coef_table is [n_steps][8] fp32 rows
 *   {sqrt_ab_t, sqrt_1mab_t, sqrt_ab_prev, eps_coef, sigma, is_last (0/1), 0, 0}
 * and step_state is int32[2] = {current step, next step} maintained by dadd_step_begin().  The step index is clamped to
 * [0, n_steps) on the device: a replay past the end of the schedule cannot read outside the tables. */
int dadd_ddim_step_table(float* x, const void* eps_cond, const void* eps_uncond /* nullable */, int eps_dtype,
                         float guidance, const float* coef_table, const int32_t* step_state, int n_steps,
                         const float* noise /* nullable; [n_steps][n] when given */, float clamp, int64_t n,
                         void* stream);

/* First node of a per-step graph: step_state[0] = step_state[1]; step_state[1] += 1; and copy row
 * step_state[0] of a [n_steps][row_len] table (the hoisted per-step time-embedding projections of all
 * resnets, SURVEY.md K3/section 7.1 step 8) into `row_out` (row index clamped to [0, n_steps)).  `table` may be NULL
 * (row_len = 0). */
int dadd_step_begin(int32_t* step_state, const void* table, void* row_out, int64_t row_bytes, int n_steps, void* stream);

/* ------------------------------------------------------------------------------------------------
 * GroupNorm (+ optional per-(sample,channel) additive term, + optional SiLU).
 * Replaces diffusers ResnetBlock2D.norm1/norm2 + nonlinearity, conv_norm_out + conv_act and
 * Transformer2DModel.norm reached through src/models/unet/unet.py:140-146 (SURVEY.md K4/K4b):
 *   y = act(GroupNorm_G(x + chan_add[b * chan_add_stride + c]; eps) * gamma[c] + beta[c]),  act = SiLU or identity.
 * Statistics in fp32 (shifted sums + Chan combine).  x/y: `dtype`; gamma/beta/chan_add: fp32.
 * C % G == 0 and C % 8 == 0 required; for NHWC additionally (C/8) <= 512.
 * NHWC: samples up to ~2.3 MB with >= 8 channels per group (every 256x256 UNet site) run as ONE launch - a thread-block
 * cluster per sample stages its slab in shared memory and combines statistics through distributed shared memory; larger
 * samples (512x512 latents, the VAE decoder) run as flat passes (partial statistics per pixel chunk, then normalise with
 * the group statistics finalised per CTA or, for many chunks, by a per-sample pass; the second read of x comes from L2).  Callers always pass `workspace`: at least dadd_groupnorm_workspace_bytes(B, C, HW, G, layout) bytes of device memory,
 * 16-byte aligned, borrowed until the queued work has run.  NCHW needs none (0 bytes, NULL allowed).
 */
int64_t dadd_groupnorm_workspace_bytes(int B, int C, int HW, int G, int layout);
int dadd_groupnorm_fwd(const void* x, const float* gamma, const float* beta, const float* chan_add /* nullable */,
                       int64_t chan_add_stride /* elements between samples */, void* y, int B, int C, int HW, int G, float eps, int apply_silu, int layout, int dtype,
                       void* workspace /* nullable for NCHW */, int64_t workspace_bytes, void* stream);

/* GroupNorm of a channel concatenation that is never materialised: the input is [x1 | x2] along channels (the
 * `torch.cat([hidden, skip], dim=1)` feeding every resnet of the up path, diffusers UpBlock2D / CrossAttnUpBlock2D reached
 * through src/models/unet/unet.py:140-146); y is the normalised concatenation [B][HW][C1 + C2], NHWC, 16-bit `dtype`.
 * x1: [B][HW][C1], x2: [B][HW][C2]; C1 % 8 == 0, C2 % 8 == 0, (C1 + C2) % G == 0, (C1 + C2) / 8 <= 512
 * (dadd_groupnorm_cat_supported()).  Same kernels, path selection and workspace rule as dadd_groupnorm_fwd(NHWC) with
 * C = C1 + C2: workspace >= dadd_groupnorm_workspace_bytes(B, C1 + C2, HW, G, DADD_LAYOUT_NHWC). */
int dadd_groupnorm_cat_supported(int B, int C1, int C2, int HW, int G, int dtype);
/* Which NHWC 16-bit kernel dadd_groupnorm_fwd / dadd_groupnorm_cat_fwd take: 0 = the cluster / flat kernels above (default: the
 * faster ones on B200 today, profiles/r02_groupnorm_stream.txt), 1 = the one-launch STREAMING kernel wherever it serves the shape
 * (C1, C2 % 64 == 0, HW % 16 == 0, G even; persistent CTAs, TMA slab ring, tensor-core statistics, per-group partial sums exchanged
 * through `workspace` behind release flags that carry a device-side launch generation; csrc/groupnorm_stream.cu).  Process-wide;
 * returns the previous value.  The environment variable DADD_GN_IMPL=stream selects 1 at load time. */
int dadd_groupnorm_select(int impl);
int dadd_groupnorm_cat_fwd(const void* x1, int C1, const void* x2, int C2, const float* gamma, const float* beta,
                           const float* chan_add /* nullable */, int64_t chan_add_stride, void* y, int B, int HW, int G,
                           float eps, int apply_silu, int dtype /* DADD_BF16 | DADD_F16 */, void* workspace,
                           int64_t workspace_bytes, void* stream);

/* LayerNorm over the last dimension (the 48 LayerNorms of the BasicTransformerBlocks and the three of
 * src/models/feature_purifier.py:46-47,62).  x,y: [rows][C] `dtype`; gamma/beta fp32; C % 8 == 0, C <= 2048. */
int dadd_layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, int64_t rows, int C, float eps,
                       int dtype, void* stream);

/* Residual add fused with the LayerNorm that consumes it (BasicTransformerBlock: hidden = attn(...) + hidden;
 * norm_hidden = norm(hidden), SURVEY.md A.5):  s = x + r rounded to `dtype`, y = LayerNorm(s) * gamma + beta; when sum_out is
 * non-NULL it receives s, or s + sum_bias[c] when sum_bias (fp32 [C]) is given - the bias of the NEXT residual branch's output
 * projection (ff.net[2].bias) rides on the stored residual, so that `ff(norm) + hidden` becomes one GEMM that accumulates onto
 * it.  LayerNorm always sees the unbiased s.  Same shapes / limits as dadd_layernorm_fwd; x, r, sum_out, y: [rows][C]. */
int dadd_add_layernorm_fwd(const void* x, const void* r, void* sum_out /* nullable */, const float* sum_bias /* nullable */,
                           const float* gamma, const float* beta, void* y, int64_t rows, int C, float eps, int dtype,
                           void* stream);

/* Channel bias and/or residual add in one vectorised pass: y[r][c] = a[r][c] (+ res[r][c]) (+ bias[c]).
 * Replaces the bias add after a library convolution and the residual adds of ResnetBlock2D / Transformer2DModel /
 * the feed-forward (diffusers graph reached through src/models/unet/unet.py:140-146).  a, res, y: [rows][C] `dtype`
 * (NHWC activations viewed as rows of C channels, or token matrices); bias: fp32 [C]; at least one of res, bias.
 * y may alias a or res.  C % 8 == 0. */
int dadd_bias_residual_fwd(const void* a, const void* res /* nullable */, const float* bias /* nullable */, void* y,
                           int64_t rows, int C, int dtype, void* stream);

/* Nearest-neighbour 2x upsampling of an NHWC activation: y[b][2h+i][2w+j][c] = x[b][h][w][c], i, j in {0, 1}.  Replaces
 * F.interpolate(x, scale_factor=2.0, mode="nearest") of diffusers' Upsample2D (up path of the UNet reached through
 * src/models/unet/unet.py:140-146, and of the VAE decoder, src/models/vae/vae.py:112).  x: [B][H][W][C], y: [B][2H][2W][C],
 * C % 8 == 0. */
int dadd_upsample_nearest2x_fwd(const void* x, void* y, int B, int H, int W, int C, int dtype, void* stream);

/* y = x * sigmoid(1.702 x): the `quick_gelu` activation of the CLIP ViT-L/14 vision tower (transformers
 * CLIPVisionModelWithProjection, loaded by the reference at src/models/image_encoder.py:34-38).  n % 8 == 0; y may alias x. */
int dadd_quick_gelu_fwd(const void* x, void* y, int64_t n, int dtype, void* stream);

/* GEGLU gate of the transformer feed-forward: y[r][j] = x[r][j] * gelu_erf(x[r][inner + j]), x: [rows][2*inner]. */
int dadd_geglu_fwd(const void* x, void* y, int64_t rows, int inner, int dtype, void* stream);

/* Linear layer as a persistent tcgen05 GEMM with bias and residual add fused into its epilogue:
 *   y[m][n] = sum_k x[m][k] w[n][k] (+ bias[n]) (+ residual[m][n])
 * Replaces nn.Linear / 1x1-conv calls of diffusers' Transformer2DModel and BasicTransformerBlock (proj_in, to_q/to_k/to_v,
 * to_out[0], ff.net[2], proj_out) and ResnetBlock2D.conv_shortcut reached through src/models/unet/unet.py:140-146, together
 * with the residual adds that follow them (`ff(x) + x`, `proj_out(x) + residual`, `shortcut(x) + h`).
 * x: [M][K], w: [N][K] (nn.Linear layout), y / residual: [M][N], all 16-bit `dtype`, dense rows, 16-byte aligned; bias: fp32 [N]
 * (nullable); residual nullable and may alias y.  The product is rounded to 16 bits before the residual is added (as the
 * unfused GEMM + add).  K % 8 == 0 and N % 64 == 0: dadd_linear_supported() says whether a shape qualifies.  Persistent tcgen05
 * GEMM, tiles 128 x {256, 192, 128}; from K = 512 on the CTAs run as pairs (cta_group::2: M = 256 MMAs over both CTAs' shared memory
 * and TMEM).  Measured 4-17 % behind cuBLAS on the UNet's shapes (profiles/r02_linear_gemm.txt): the host keeps cuBLAS as its default. */
int dadd_linear_supported(int64_t M, int N, int K);
int dadd_linear_fwd(const void* x, const void* w, const float* bias /* nullable */, const void* residual /* nullable */, void* y,
                    int64_t M, int N, int K, int dtype /* DADD_BF16 | DADD_F16 */, void* stream);

/* Feed-forward input projection fused with the GEGLU gate (tcgen05 GEMM, GELU in the epilogue):
 *   y[m][j] = (x w[j]^T + bias[j]) * gelu_erf(x w[inner + j]^T + bias[inner + j]),  j < inner.
 * Replaces `hidden, gate = proj(x).chunk(2, -1); hidden * F.gelu(gate)` of diffusers' GEGLU (FeedForward.net[0] of every
 * BasicTransformerBlock reached through src/models/unet/unet.py:140-146) and the (M, 2 inner) intermediate it writes.
 * x: [M][K], w: [2 inner][K] (nn.Linear weight layout), y: [M][inner], all 16-bit `dtype`, dense rows, 16-byte aligned;
 * bias: fp32 [2 inner].  K % 8 == 0, inner % 128 == 0. */
int dadd_ff_geglu_fwd(const void* x, const void* w, const float* bias, void* y, int64_t M, int K, int inner,
                      int dtype /* DADD_BF16 | DADD_F16 */, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused multi-pathway cross-attention core.
 * Replaces the three explicit matmul/softmax/matmul pathways and the gate merge of
 * SplitInjectionAttentionProcessor.__call__ (src/models/attention_processor_routing_gates.py:148-178) and, with
 * n_seg = 1, seg_len = 32, the single softmax of OrdinalIPAttnProcessor2_0.__call__
 * (src/models/attention_processor_base.py:96-118):
 *   o[b][n][h*d + :] = sum_s gates[s] * softmax(q_bh[n] . k_s^T * scale) v_s ,  s over n_seg segments of seg_len tokens
 * q: 16-bit (`dtype`) [B][N][*] with row stride q_stride elements, head h at column h*d (i.e. the to_q output as is);
 * k_cat, v_cat: `dtype` [B][H][n_seg*seg_len][d] (step-invariant; projected once per sampling call, token order
 * dis | anat | delta = encoder_hidden_states[:, :16], [:, 16:32], [:, -16:], routing_gates.py:129-131);
 * gates: fp32[n_seg] ON DEVICE in token order (dis_gate, anat_gate, delta_scale);
 * o: `dtype` [B][N][*] with row stride o_stride, written at column h*d (heads merged, ready for to_out).
 * d in {40, 80, 160} (d % 8 == 0, d <= 160); seg_len % 16 == 0; n_seg*seg_len <= 64.
 * delta_scale == 0 must be expressed as n_seg = 2 (the pathway is skipped, routing_gates.py:160,177).
 * impl: 0 = shape dispatch (N >= 128, d <= 128 and (seg_len, n_seg) in {(16,2), (16,3), (32,1)} -> tcgen05/TMEM/TMA kernel:
 *       persistent CTAs, a query row per thread and TMEM lane, TMA ring of Q / K_cat / V_cat tiles, TMA-store epilogue;
 *       otherwise the warp-level mma.sync kernel), 1 = force mma.sync, 2 = force tcgen05 (fails if unsupported).
 */
int dadd_cross_attn_fwd(const void* q, int64_t q_stride, const void* k_cat, const void* v_cat, void* o,
                        int64_t o_stride, int B, int H, int N, int d, int seg_len, int n_seg, const float* gates,
                        float scale, int dtype /* DADD_BF16 | DADD_F16 */, int impl, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Self-attention core (attn1): o = softmax(q k^T * scale) v per (b, h), no mask.
 * Replaces F.scaled_dot_product_attention inside diffusers' AttnProcessor2_0, installed by
 * src/models/attention_processor_routing_gates.py:284-286 and attention_processor_base.py:196-197.
 * q, k, v: 16-bit (`dtype`: DADD_BF16 | DADD_F16) [B][N][*] with row strides (elements); head h at column h*d (so the
 * three can alias one fused [B][N][3C] projection output); o: same dtype and convention.  d % 8 == 0, d <= 160 - or d = 256 / 512: wide single
 * heads (the VAE mid block's attention, src/models/vae/vae.py:90-112) on a column-split mma.sync kernel, any N, `impl` ignored.
 * impl: 0 = shape dispatch (N >= 128 -> tcgen05/TMEM/TMA flash kernel, else warp-level mma.sync kernel),
 *       1 = force mma.sync, 2 = force tcgen05 (N >= 128 required).
 */
int dadd_self_attn_fwd(const void* q, const void* k, const void* v, int64_t q_stride, int64_t k_stride,
                       int64_t v_stride, void* o, int64_t o_stride, int B, int H, int N, int d, float scale,
                       int dtype, int impl, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Feature Purifier pieces (src/models/feature_purifier.py:81-95), fp32 (runs once per sampling call).
 * (1) multi-head attention core of nn.MultiheadAttention(768, 8): q [B][Lq][D], k,v [B][Lk][D] (already
 *     in-projected), o [B][Lq][D] (before out_proj); Lq <= 256, D/heads <= 128, and one (sample, head) must fit
 *     shared memory: ((Lq + 2 Lk)(D/heads + 1) + Lq Lk) floats <= 227 KB.  Also the core of the Perceiver resampler
 *     (ImageProjectionPlus, src/models/image_encoder.py:213-220: 16 queries over the 257 CLIP patch tokens).
 * (2) gating epilogue: y = LayerNorm(img - sigmoid(gate_logits) * disease; gamma, beta, eps), all [rows][D].
 */
int dadd_purifier_attn_fwd(const float* q, const float* k, const float* v, float* o, int B, int Lq, int Lk, int D,
                           int heads, void* stream);
int dadd_purifier_gate_ln_fwd(const float* img, const float* gate_logits, const float* disease, const float* gamma,
                              const float* beta, float* y, int64_t rows, int D, float eps, void* stream);

/* AOE table lookup (src/models/ordinal_embedder.py:107-127,155-171,15-40): table E[k] = base + cumsum(deltas)[k-1],
 * labels clamped to [0, K-1], lo = floor, hi = min(lo+1, K-1), out[b] = E[lo]*(1-a) + E[hi]*a, a = y - lo.
 * base [D], deltas [K-1][D], labels [B], out [B][D], all fp32.  Integer indices are exact. */
int dadd_aoe_interp_fwd(const float* base, const float* deltas, const float* labels, float* out, int B, int K, int D,
                        void* stream);

/* Latents -> displayable images tail of _latents_to_images (src/pipelines/inference/inference_pipeline_ip.py:483-485):
 * y = clamp((clamp(x, -1, 1) + 1) / 2, 0, 1); x `dtype` (decoder output), y fp32. */
int dadd_image_post_fwd(const void* x, float* y, int64_t n, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training step (SURVEY.md 8f row f1): what Lightning autograd + torch.optim run for the reference at
 * src/models/diffusion_module_ip.py:392-462 (training_step: MSE x Min-SNR weight), :500-536 (AdamW groups) and
 * src/pipelines/training/training_pipeline_ip.py:103-123 (gradient_clip_val, precision "16-mixed", DDP).
 * All reductions are two-stage and atomics-free (bit-reproducible).
 *
 * LayerNorm backward: x, dy, dx [rows][C] 16-bit; gamma [C]; dgamma / dbeta are the two rows of ONE fp32 (2, C) buffer
 * (dbeta == dgamma + C); workspace: dadd_layernorm_bwd_workspace_bytes(C).  Statistics are recomputed from x. */
int64_t dadd_layernorm_bwd_workspace_bytes(int C);
int dadd_layernorm_bwd(const void* x, const void* dy, const float* gamma, void* dx, float* dgamma, float* dbeta,
                       float* workspace, int64_t rows, int C, float eps, int dtype, void* stream);
/* GEGLU backward: proj [M][2 inner] = [value | gate], dy [M][inner] -> dproj [M][2 inner]; exact (erf) GELU. */
int dadd_geglu_bwd(const void* proj, const void* dy, void* dproj, int64_t M, int inner, int dtype, void* stream);
/* GroupNorm (+ chan_add[b][c]) (+ SiLU) backward, NHWC: x, dy, dx [B][HW][C] 16-bit; gamma, beta, dgamma, dbeta [C] fp32;
 * chan_add / dchan_add [B][C] fp32 or NULL (dchan_add needs chan_add).  Statistics are recomputed from x. */
int64_t dadd_groupnorm_bwd_workspace_bytes(int B, int C, int HW, int G);
int dadd_groupnorm_bwd(const void* x, const float* chan_add, const void* dy, const float* gamma, const float* beta,
                       void* dx, float* dgamma, float* dbeta, float* dchan_add, float* workspace, int B, int HW, int C,
                       int G, float eps, int apply_silu, int dtype, void* stream);
/* Backward of dadd_cross_attn_fwd's core (attention_processor_routing_gates.py:148-178) for the training step: q, dout, dq
 * [B][N][*] 16-bit with row strides (head h at column h*d), k_cat / v_cat [B][H][L][d] 16-bit (L = n_seg * seg_len <= 48),
 * gates [n_seg] fp32 (device); dk, dv [B][H][L][d] fp32.  workspace: dadd_cross_attn_bwd_workspace_bytes(...). */
int64_t dadd_cross_attn_bwd_workspace_bytes(int B, int H, int N, int d, int L);
int dadd_cross_attn_bwd(const void* q, int64_t q_stride, const void* k_cat, const void* v_cat, const float* gates,
                        const void* dout, int64_t do_stride, void* dq, int64_t dq_stride, float* dk, float* dv,
                        float* workspace, int B, int H, int N, int d, int L, int seg_len, float scale, int dtype, void* stream);
/* loss[0] = mean_b weight[b] * mean_e (pred - target)^2 (diffusion_module_ip.py:449-452); grad (optional) = upstream *
 * dloss/dpred.  pred, target, grad [B][E] fp32; workspace: dadd_minsnr_mse_workspace_bytes(B). */
int64_t dadd_minsnr_mse_workspace_bytes(int B);
int dadd_minsnr_mse(const float* pred, const float* target, const float* weight, float* loss, float* grad,
                    float* workspace, int B, int64_t E, float upstream, void* stream);
/* Gradient-norm clipping and AdamW over flat fp32 buckets, no host synchronisation:
 * dadd_sumsq writes n_partials partial sums of g^2 (g may be NULL when n == 0); dadd_clip_coef turns ALL partials of a step into
 * coef_and_norm[0] = grad_scale * min(1, max_norm / (norm + 1e-6)) (max_norm <= 0: no clipping) and [1] = norm =
 * grad_scale * sqrt(sum) (torch.nn.utils.clip_grad_norm_; grad_scale = 1 / world size when the buckets hold SUMS);
 * dadd_adamw_step applies torch.optim.AdamW's update with g scaled by coef[0] (coef may be NULL).  A non-finite norm (fp16
 * overflow under a loss scale; fold 1 / loss_scale into grad_scale) makes coef[0] NaN and the AdamW launches no-ops. */
int dadd_sumsq(const float* g, int64_t n, float* partials, int n_partials, void* stream);
int dadd_clip_coef(const float* partials, int n, float max_norm, float grad_scale, float* coef_and_norm, void* stream);
int dadd_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                    float weight_decay, float bias_corr1, float bias_corr2, const float* coef, void* stream);
/* The same update with the step-dependent scalars on the device: dev_state[0] scales lr (the schedule), dev_state[1] is the step
 * number t of the bias corrections 1 - beta^t, i.e. the count of APPLIED updates: the caller advances it after dadd_clip_coef
 * only when coef[0] is finite (a skipped step does not count, as under torch.amp.GradScaler).  Lets ONE captured CUDA graph of
 * the whole training step (forward, backward, gradient all-reduce, clip, AdamW) replay for every step: nothing the host passes
 * changes between replays. */
int dadd_adamw_step_dev(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                        float weight_decay, const float* dev_state /* {lr scale, step} */, const float* coef, void* stream);
/* EMA weight averaging of a flat fp32 parameter bucket: avg += (p - avg) * (1 - decay); first != 0: avg = p.  Replaces the
 * AveragedModel.update_parameters call of the reference's EMAWeightAveraging callback (src/callbacks/ema_callback.py:168-197,414-436:
 * torch.optim.swa_utils.get_ema_avg_fn(decay), decay 0.999, every 4th step from step 100 in configs/train_ip.yaml:83-85). */
int dadd_ema_update(float* avg, const float* p, int64_t n, float decay, int first, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Pairwise squared-distance statistics of two fp32 feature sets, for the CMMD, improved precision / recall, density / coverage
 * and realism metrics.
 * Replaces the distance matrices of the evaluation metrics (src/pipelines/evaluation/evaluation_pipeline.py:577-839,978-1179:
 * CMMD's `mmd` of google-research/cmmd and the k-NN radii / coverage of Kynkaanniemi et al. 2019), none of which is
 * materialised here.  x: [M][D], y: [N][D], dense row-major fp32, 16-byte aligned;
 *   d2[i][j] = max(|x_i|^2 + |y_j|^2 - 2 x_i . y_j, 0), the dot products by error-compensated TF32 (3 tcgen05 passes, fp32 accumulate).
 * mode DADD_PAIRWISE_RBF_SUM: out = double[1] = sum over all (i, j) of exp(-gamma d2[i][j]) (fixed-order, atomics-free sums:
 *      bit-reproducible);
 *      DADD_PAIRWISE_KNN:     out = float[M], the k-th smallest d2[i][j] over j (1 <= k <= 16; N > k, or N > k + 1 with same_set);
 *      DADD_PAIRWISE_COVER:   out = uint8[M], 1 where some j has d2[i][j] <= radii[j];
 *      DADD_PAIRWISE_COUNT:   out = int32[M], the number of j with d2[i][j] <= radii[j];
 *      DADD_PAIRWISE_RATIO_MAX: out = float[M], the max over j of radii[j] / (d2[i][j] + eps) (IEEE fp32 division, 0 when no
 *                             ratio is positive), eps passed in `gamma`: finite and > 0.
 * COVER, COUNT and RATIO_MAX need radii (float[N]) and reject same_set.  Counts, flags and maxima are merged in a fixed order:
 * every mode is bit-reproducible and independent of the grid.
 * same_set (RBF_SUM, KNN): y is x (pass y = NULL or x, N = M); KNN then excludes j == i by index.  D % 8 == 0.
 * workspace: at least dadd_pairwise_workspace_bytes(...) bytes (-1: the arguments are rejected), 16-byte aligned: the tf32
 * hi / lo split of the rows ((M + N) * D * 8 bytes, M * D * 8 with same_set), the row norms and the per-slice partials (RBF_SUM:
 * one double per (128-row block, column slice); KNN: M * slices * k floats; COVER, COUNT: M * slices int32 counts; RATIO_MAX:
 * M * slices floats); never an M x N buffer. */
#define DADD_PAIRWISE_RBF_SUM 0
#define DADD_PAIRWISE_KNN 1
#define DADD_PAIRWISE_COVER 2
#define DADD_PAIRWISE_COUNT 3
#define DADD_PAIRWISE_RATIO_MAX 4
int64_t dadd_pairwise_workspace_bytes(int64_t M, int64_t N, int D, int mode, int k, int same_set);
int dadd_pairwise(const float* x, const float* y /* NULL or x with same_set */, int64_t M, int64_t N, int D, int mode, int k,
                  int same_set, float gamma /* RBF_SUM: gamma; RATIO_MAX: eps */,
                  const float* radii /* COVER, COUNT, RATIO_MAX */, void* out, void* workspace,
                  int64_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DADD_B200_H */
