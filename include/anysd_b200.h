/* anysd_b200 -- C ABI of the B200-native AnySD denoising hot path.
 *
 * The reference (DCDmllm/AnyEdit) has no FFI boundary on this path: its hot path is eager
 * PyTorch modules (SURVEY.md 8b).  This header is therefore the *new* boundary a maintainer
 * binds to; every entry point names the reference code whose arithmetic it replaces
 * (paths relative to the reference root).  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - plain C: raw device pointers, sizes, a cudaStream_t passed as void*; no torch types.
 *   - no ownership transfer: every buffer (workspaces included) belongs to the caller.
 *   - asynchronous on the given stream, no hidden synchronisation, CUDA-graph capturable.
 *   - returns 0 on success, a negative ANYSD_E* code on failure; anysd_last_error() returns a
 *     thread-local message.  There is no CPU fallback: without a CUDA device calls fail.
 *   - activations are NHWC fp16 ("tokens" [N, H*W, C]); statistics/accumulators are fp32.
 */
#ifndef ANYSD_B200_H_
#define ANYSD_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ANYSD_OK 0
#define ANYSD_EINVAL (-1)   /* bad argument / unsupported shape (ValueError in the Python mirror) */
#define ANYSD_ECUDA (-2)    /* CUDA runtime / launch failure (RuntimeError) */
#define ANYSD_EUNSUPPORTED (-3)

#define ANYSD_F32 0
#define ANYSD_F16 1
#define ANYSD_I64 2

typedef void* anysd_stream_t; /* cudaStream_t */

const char* anysd_last_error(void);
int anysd_version(void);
/* sm count and compute capability of the current device */
int anysd_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- layout ------------------------------------------------------------------------------
 * x.type(self.dtype) + torch.cat([x] + c_concat, dim=1)   ldm/models/diffusion/ddpm.py:1344-1346,
 * ldm/modules/diffusionmodules/openaimodel.py:774: NCHW (f32|f16) -> channel slice
 * [dst_c_off, dst_c_off+C) of an NHWC fp16 tensor with dst_C channels. */
int anysd_nchw_to_nhwc_f16(const void* src, int src_dtype, void* dst, int N, int C, int H, int W,
                           int dst_C, int dst_c_off, anysd_stream_t stream);
/* ControlNet residual injection, `h += control.pop()` / `hs.pop() + control.pop()` of ControlledUnetModel.forward
 * (AnyEdit_Collection/other_modules/cldm/cldm.py:33-41): dst (NHWC fp16 [N,H,W,C]) += src (NCHW f32|f16). */
int anysd_add_nchw_into_nhwc_f16(const void* src, int src_dtype, void* dst, int N, int C, int H, int W,
                                 anysd_stream_t stream);
/* h.type(x.dtype) on the way out (openaimodel.py:782): NHWC (f16|f32) with src_C channels per pixel (the first C
 * are converted) -> NCHW (f32|f16). */
int anysd_nhwc_to_nchw(const void* src, int src_dtype, int src_C, void* dst, int dst_dtype, int N, int C, int H, int W,
                       anysd_stream_t stream);
/* th.cat([h, hs.pop()], dim=1) (openaimodel.py:780) on NHWC rows: dst[r] = a[r] ++ b[r]. */
int anysd_concat_channels_f16(const void* a, int Ca, const void* b, int Cb, void* dst, long long rows,
                              anysd_stream_t stream);
int anysd_cast_f32_to_f16(const float* src, void* dst, long long n, anysd_stream_t stream);

/* ---- time / task embedding ---------------------------------------------------------------
 * timestep_embedding (ldm/modules/diffusionmodules/util.py:154-174): cos half first. */
int anysd_timestep_embedding_f16(const void* t, int t_dtype, void* out_f16, int N, int dim, float max_period,
                                 anysd_stream_t stream);
/* emb = time_embed(t_emb) [+ label_emb(y) | task_embs[edit_code]] (openaimodel.py:768-772;
 * train.py:694-695) and the SiLU that opens every ResBlock.emb_layers (openaimodel.py:217-223):
 * emb_out[n] = emb_lin[n] + table[idx[n]] ; silu_out = fp16(silu(emb_out)). table/idx/emb_out may be NULL. */
int anysd_emb_finalize(const float* emb_lin, const float* table, const long long* idx, int table_rows,
                       float* emb_out, void* silu_out_f16, int N, int D, anysd_stream_t stream);

/* Task-aware router gate (AnySD.model.MoE, source absent -- train.py:420-424, 694-695; restated in
 * oracle/anysd_oracle.py): gate[b, l, :] = softmax_e(W[l, e, :] . table[idx[b], :] + bias[l, e]) for all
 * L cross-attention layers at once.  table fp32 [T, D], W fp16 [L, E, D], bias fp32 [L, E], gate fp32 [B, L, E]. */
int anysd_router_gate_f32(const float* table, const long long* idx, int table_rows, const void* W,
                          const float* bias, float* gate, int B, int L, int E, int D, anysd_stream_t stream);

/* ---- normalisation -----------------------------------------------------------------------
 * GroupNorm32 + SiLU (util.py:202-219; openaimodel.py:200-203, 224-227, 726-728) and the
 * SpatialTransformer GroupNorm (attention.py:88-89, 326; eps 1e-6, no SiLU).  Statistics in fp32.
 * The input may be the channel concat of two NHWC tensors (x2 != NULL): the skip concat
 * (openaimodel.py:780) is then never materialised for the norm. y: NHWC fp16 [N, HW, C1+C2]. */
/* The workspace must be zero-filled once before its first use (it holds per-image completion counters that every
 * launch re-arms); it may then be reused by any number of stream-ordered calls. */
size_t anysd_groupnorm_workspace_bytes(int N, int G, int C);
int anysd_groupnorm_nhwc_f16(const void* x1, int C1, const void* x2, int C2, const float* gamma,
                             const float* beta, void* y, int N, int HW, int G, float eps, int fuse_silu,
                             void* workspace, size_t workspace_bytes, anysd_stream_t stream);
/* 1 when anysd_groupnorm_nhwc_f16 serves (C1 + C2 channels, HW pixels, G groups) with its register-resident kernel (one read,
 * one write, one launch: the statistics need no help from the producer's epilogue), 0 when it takes the statistics + apply
 * path.  A function of the geometry only.  Host-side query, no launch. */
int anysd_groupnorm_resident(int C1, int C2, int HW, int G);
/* GroupNorm whose statistics were produced by the epilogue(s) of the contraction(s) that wrote x (anysd_gemm_params::stats):
 * a fixed-order fold of the slab partials per (image, group) in double, then ONE streaming pass y = [silu](x a + b).
 * x: NHWC fp16 [N, HW, C]; its channels [0, C1) come with stats1 ([>= N, S, C1, 2]) and, when the tensor is a channel concat
 * (openaimodel.py:780), channels [C1, C) with stats2 ([>= N, S, C - C1, 2]); stats2 NULL <=> C1 == C. */
int anysd_groupnorm_apply_nhwc_f16(const void* x, int C, const float* stats1, int C1, const float* stats2, int S,
                                   const float* gamma, const float* beta, void* y, int N, int HW, int G, float eps,
                                   int fuse_silu, void* workspace, size_t workspace_bytes, anysd_stream_t stream);
/* nn.LayerNorm(dim) (attention.py:262-264), one row per token. */
int anysd_layernorm_f16(const void* x, const float* gamma, const float* beta, void* y, long long M, int C,
                        float eps, anysd_stream_t stream);

/* ---- tensor-core contraction ---------------------------------------------------------------
 * One entry point for every dense contraction on the path:
 *   nn.Linear / 1x1 conv   attention.py:154-161 (to_q/k/v/out), :52-56 (GEGLU proj), :70 (FF out),
 *                          :298-318 (proj_in/out); openaimodel.py:240 (skip_connection),
 *                          :526-530 (time_embed), :217-223 (emb_layers)
 *   3x3 conv, pad 1        openaimodel.py:203, 228-230 (ResBlock), :552 (input), :729 (out),
 *                          :148-150 (Downsample, stride 2), :104-117 (Upsample: nearest x2 folded in)
 * out[m, n] = act(sum_k A[m,k] W[n,k] + bias[n] + rowadd[m / rows_per_batch, n]) + residual[m, n]
 * fp16 operands, fp32 accumulate.  act: 0 none, 1 SiLU, 2 GEGLU (W rows interleaved (a_j, gate_j);
 * out has N/2 columns: (acc_a + b_a) * gelu_erf(acc_g + b_g)), 3 GELU (erf; nn.GELU of the CLIP-H MLP and the Resampler
 * FeedForward), 4 QuickGELU (x sigmoid(1.702 x), the CLIP-L MLP). */
typedef struct {
    const void* A;          /* dense: fp16 [M, lda]; conv: NHWC fp16 image [Nimg, H, W, Cin] */
    const void* W;          /* fp16 [N, ldw], row n = output channel, K contiguous ((ky,kx,ci) for conv) */
    const float* bias;      /* [N] or NULL */
    const float* rowadd;    /* fp32 [*, ld_rowadd] or NULL */
    const void* residual;   /* fp16 [M, ldr] or NULL */
    void* out;              /* [M, ldo] fp16 or fp32 */
    int M, N, K;
    int lda, ldw, ldo, ldr, ld_rowadd;
    int rows_per_batch;
    int act;
    int out_dtype;          /* ANYSD_F16 | ANYSD_F32 */
    int conv;               /* 0 dense, 1 conv3x3 pad 1 */
    int Nimg, H, Wd, Cin;   /* conv: input image dims (before the folded upsample) */
    int stride;             /* conv: 1 | 2 */
    int upsample;           /* conv: 1 = nearest x2 before the conv */
    void* workspace;        /* optional scratch (conv with upsample: >= Nimg*2H*2W*Cin fp16), may be NULL */
    size_t workspace_bytes;
    int conv_pad;           /* conv: 0 = zero pad 1 on every side; 1 = pad right / bottom only (the first-stage Downsample,
                               ldm/modules/diffusionmodules/model.py:83-85: F.pad(x, (0,1,0,1)) + conv3x3 stride 2 pad 0) */
    float* stats;           /* optional: GroupNorm statistics of the OUTPUT, written by the epilogue (the consumer's GroupNorm32,
                               util.py:202-219, then needs no statistics pass): fp32 [stats_images, S, N, 2] = per image, per
                               32-row slab (S = rows_per_batch / 32 = anysd_gemm_stats_slabs()), per channel {sum, sum of
                               squares} of the fp32 results.  rows_per_batch must be the rows of one image.  Every cell is
                               written exactly once in a fixed order: deterministic, independent of the batch.  NULL: off. */
    int stats_images;       /* image slots in `stats` (>= number of images, rounded up to the conv's images-per-tile) */
    void* splitk_workspace; /* optional scratch for split-K (few output tiles, long K): anysd_gemm_splitk_workspace_bytes() bytes */
    size_t splitk_workspace_bytes;
    void* splitk_counters;  /* optional: >= 64 KB of device memory, ZERO before the first use (every launch re-arms it); may be
                               shared by all stream-ordered launches of a device.  Without both, the plain schedule runs. */
    size_t splitk_counters_bytes;
    /* LayerNorm folded into the contractions either side of it (nn.LayerNorm norm1/2/3 of BasicTransformerBlock,
       attention.py:262-264, 271-274): the PRODUCER of x emits per-row moments from its epilogue, the CONSUMER takes the
       un-normalised x as A with gamma folded into W and applies  out = act(rstd_m (acc - mean_m colsum_n) + bias_n) + residual
       -- algebraically LayerNorm(x) W^T + b without the normalised tensor ever being written or re-read. */
    float* row_stats;       /* optional OUTPUT: fp32 [N / 64, M, 2] = per 64-column slab, per row {sum, sum of squares} of the fp32
                               results (after bias / residual).  Dense, fp16 output, act 0, N % 64 == 0.  Every cell written once. */
    const float* ln_stats;  /* optional INPUT: the row_stats ([K / 64, M, 2]) of A's producer; K % 64 == 0.  Then W must hold
                               W[n,k] gamma[k], bias[n] = b[n] + sum_k beta[k] W[n,k] (required) and */
    const float* ln_colsum; /* fp32 [N]: sum_k of the fp16 values of the packed W row n (16-byte aligned) */
    float ln_eps;
} anysd_gemm_params;
int anysd_gemm_f16(const anysd_gemm_params* p, anysd_stream_t stream);
/* Slabs per image of the statistics layout for this contraction, or 0 when the shape cannot produce them (rows of one
 * image not a multiple of 32, conv patches not tiling the image exactly, GEGLU / fp32 output, non-tcgen05 shape). */
int anysd_gemm_stats_slabs(const anysd_gemm_params* p);
/* Bytes of `splitk_workspace` with which this contraction runs split-K (0: the schedule does not split it).  Whether a layer is
 * split depends on its per-image geometry only (<= 128 output rows per image and a long K), never on the batch; the partial
 * sums are added in split order by whichever unit finishes last.  The result therefore depends neither on the batch nor on the
 * arrival order -- but a caller that withholds the scratch gets the unsplit summation order (differs in fp32 rounding). */
size_t anysd_gemm_splitk_workspace_bytes(const anysd_gemm_params* p);
/* What anysd_gemm_f16 would launch for these exact params (same validation, same selection code, the split-K scratch as
 * attached): kernel 0 mma.sync, 1 tcgen05, 2 persistent tcgen05; for kernel 2 also ctas (1 | 2: CTA pairs), bn (tile width
 * 64 | 128 | 192 | 256), splits (K split, 1 = unsplit), ext (1 = the extended epilogue: GroupNorm statistics / split-K /
 * GELU / QuickGELU) and ln (1 = the LayerNorm-fold epilogue: row_stats or ln_stats); all 0 for kernels 0 and 1.  Returns the
 * error code anysd_gemm_f16 would return, ANYSD_OK otherwise.  Any output pointer may be NULL. */
int anysd_gemm_schedule(const anysd_gemm_params* p, int* kernel, int* ctas, int* bn, int* splits, int* ext, int* ln);

/* ---- attention ---------------------------------------------------------------------------
 * CrossAttention.forward (attention.py:163-194) / xformers memory_efficient_attention (:233):
 * out = softmax(q k^T * scale) v per (batch, head); fp16 q/k/v, fp32 scores/softmax/accumulate.
 * q: [B, n_q, ld_q] with head h at columns [h*d, (h+1)*d); same for k, v ([B, n_kv, ld_k|ld_v]) and out.
 * gate != NULL: out = out_prev * (accumulate ? 1 : 0) + gate[b] * attn  -- the task-router expert sum
 * (SURVEY.md a22; oracle/anysd_oracle.py). */
typedef struct {
    const void* q; const void* k; const void* v; void* out;
    long long q_batch_stride, k_batch_stride, v_batch_stride, o_batch_stride; /* elements */
    int ld_q, ld_k, ld_v, ld_o;                                               /* elements */
    int B, heads, n_q, n_kv, d;
    float scale;
    const float* gate;      /* [B] stride gate_stride, or NULL */
    int gate_stride;
    int accumulate;
    int head_stride;        /* elements between consecutive heads inside a q/k/v row; 0 = d.  The tcgen05 kernel
                               needs head_stride >= ceil16(d) with zero padding columns when d % 16 != 0 */
    int aux_cols;           /* 1 = "operands carry the softmax bookkeeping" (tcgen05 kernel only; needs d % 16 == 8,
                               head_stride >= d + 8, EUNSUPPORTED otherwise).  Contract, per head:
                                 q: columns [0,d) hold q * scale * log2(e) (the caller folds both into Wq; `scale` is
                                    ignored), columns d.. are zero;
                                 k: columns d and d+1 hold 1.0;    v: column d holds 1.0;   other padding zero.
                               The kernel writes its running reference into q's padding inside shared memory, so the
                               scores leave the tensor core already shifted (exp2 only) and the softmax denominator is
                               column d of P.V.  Same result as aux_cols = 0 up to fp32 rounding. */
    float* lse;             /* optional OUTPUT (tcgen05 kernels only, gate == NULL): fp32 [B, heads, n_q], the base-2 log-sum-exp of
                               every score row, lse2_i = log2 sum_j 2^(scale log2(e) q_i.k_j) -- what anysd_attention_bwd_f16 needs
                               to recompute the probabilities without its own pass over K (train.py:694-709 backward). */
} anysd_attn_params;
int anysd_attention_f16(const anysd_attn_params* p, anysd_stream_t stream);

/* ---- sampler step ------------------------------------------------------------------------
 * DDIMSampler.p_sample_ddim (ldm/models/diffusion/ddim.py:211-212, 228-250), eps-parameterisation:
 *   e = e_u + s (e_c - e_u);  pred_x0 = (x - sqrt(1-a_t) e) / sqrt(a_t);
 *   x_prev = sqrt(a_prev) pred_x0 + sqrt(1 - a_prev - sigma^2) e + sigma * noise
 * all fp32, NCHW.  eps holds [uncond ; cond] (2B rows) when cfg != 0, else B rows.
 * coef[5] = {sqrt(1-a_t), 1/sqrt(a_t) as sqrt(a_t) divisor, sqrt(a_prev), sqrt(1-a_prev-sigma^2), sigma}
 * lives on the device so that one CUDA graph serves all steps.  noise/pred_x0 may be NULL.
 * v_param != 0: the model output is v (ddim.py:214-218, 224-226); coef[5] = sqrt(acp[t]), coef[6] = sqrt(1-acp[t]):
 *   e = coef[5] v + coef[6] x;  pred_x0 = coef[5] x - coef[6] v  (ddpm.py predict_eps/start_from_z_and_v). */
int anysd_cfg_ddim_step_f32(const float* x, const float* eps, const float* noise, const float* coef,
                            float guidance_scale, int cfg, int v_param, float* x_prev, float* pred_x0, long long n_per_batch,
                            int B, anysd_stream_t stream);

/* InstructPix2Pix three-way guidance (tools/global_tool.py:166-177; SURVEY.md 8f rank 4) + the same DDIM update:
 * eps holds [text ; image ; uncond] (3B rows);  e = e_unc + text_scale (e_txt - e_img) + image_scale (e_img - e_unc). */
int anysd_cfg3_ddim_step_f32(const float* x, const float* eps, const float* noise, const float* coef, float text_scale,
                             float image_scale, float* x_prev, float* pred_x0, long long n_per_batch, int B,
                             anysd_stream_t stream);

/* PLMSSampler.p_sample_plms (ldm/models/diffusion/plms.py:178-244): CFG combine, Adams-Bashforth combination of the eps
 * history, DDIM update (sigma = 0) and the history push in one kernel.  hist = three [B, n_per_batch] fp32 planes (o1, o2, o3),
 * zero-initialised by the caller.  coef[10] = {sqrt(1-a_t), sqrt(a_t), sqrt(a_prev), sqrt(1-a_prev), c0, c1, c2, c3, den, push}:
 * e' = (((c0 e - c1 o1) + c2 o2) - c3 o3) / den, evaluated left to right like the reference's tensor expressions. */
int anysd_cfg_plms_step_f32(const float* x, const float* eps, const float* coef, float guidance_scale, int cfg, float* hist,
                            float* x_prev, float* pred_x0, long long n_per_batch, int B, anysd_stream_t stream);

/* DPM-Solver++(2M) as DPMSolverSampler configures it (ldm/models/diffusion/dpm_solver/sampler.py:61-87; dpm_solver.py:352-365
 * data prediction, :469-513 first-order update, :723-778 second-order multistep update): coef[6] = {sigma_s, alpha_s,
 * sigma_t/sigma_s, c, 0.5 c (0 for a first-order step), 1/r0};  m = (x - sigma_s e)/alpha_s;
 * x_next = ((sigma_t/sigma_s) x - c m) - (0.5 c)((1/r0)(m - m_prev));  m_prev <- m (zero-initialised by the caller). */
int anysd_cfg_dpmpp_step_f32(const float* x, const float* eps, const float* coef, float guidance_scale, int cfg, float* m_prev,
                             float* x_next, float* x0_out, long long n_per_batch, int B, anysd_stream_t stream);

/* ==== first stage (SURVEY.md 8f rank 1): AutoencoderKL encode / decode run on the kernels above; two helpers ==============
 * AttnBlock (ldm/modules/diffusionmodules/model.py:176-203) has ONE head of width C (512 in the SD autoencoder): wider than
 * the attention tile, so it runs as S = q k^T (anysd_gemm_f16, fp32 out) -> P = softmax(S * scale) (this kernel, fp16) ->
 * O = P v (anysd_gemm_f16).  S: fp32 [rows, ld_s], P: fp16 [rows, ld_p], n valid columns. */
int anysd_softmax_rows_f32(const float* S, long long ld_s, void* P, long long ld_p, int rows, int n, float scale,
                           anysd_stream_t stream);
/* DiagonalGaussianDistribution (ldm/modules/distributions/distributions.py:24-62) from the moments [B, 2Z, HW] (fp32 NCHW):
 * logvar = clamp(moments[:, Z:], -30, 20); sample = scale * (mean + exp(0.5 logvar) * noise), noise NULL: scale * mean (the
 * mode); scale = get_first_stage_encoding's scale_factor (ddpm.py), 1 for the plain distribution.
 * sample / logvar: fp32 [B, Z, HW], either may be NULL. */
int anysd_gaussian_posterior_f32(const float* moments, const float* noise, float* sample, float* logvar, float scale,
                                 int B, long long z_hw, anysd_stream_t stream);

/* ==== condition encoders (SURVEY.md 8f rank 2): the CLIP towers and the Resampler run on the kernels above; two helpers ====
 * CLIPTextEmbeddings (transformers modeling_clip.py; FrozenCLIPEmbedder, ldm/modules/encoders/modules.py:107-150):
 * out[b, i, :] = tok_table[ids[b, i], :] + pos_table[i, :]; fp16 tables [vocab, D] / [>= n, D], out fp16 [B*n, D]. */
int anysd_embed_tokens_f16(const long long* ids, const void* tok_table, const void* pos_table, void* out, int B, int n, int D,
                           int vocab, anysd_stream_t stream);
/* softmax(q k^T scale [+ causal mask]) v per (batch, head) for SHORT sequences (n_kv <= 256): the causal 77-token
 * self-attention of the CLIP text tower (the tcgen05 attention has no mask path).  Row-major fp16 q [B*n_q, ld_q] with head h
 * at columns [h d, (h+1) d), same for k, v ([B*n_kv, ld_k|ld_v]) and out; causal != 0: key j masked for query i when j > i. */
int anysd_attention_small_f16(const void* q, const void* k, const void* v, void* out, int B, int heads, int n_q, int n_kv, int d,
                              int ld_q, int ld_k, int ld_v, int ld_o, float scale, int causal, anysd_stream_t stream);

/* ==== training step (SURVEY.md a24; train.py:629-710) =====================================================
 * The reference back-propagates mse_loss(MoE(...), noise) through the frozen UNet with torch autograd
 * (train.py:694-703); trainables are the adapter experts, the router and the task-embedding table
 * (train.py:486-492).  Below: every non-contraction backward op of the path.  dX of linears / convs reuses
 * anysd_gemm_f16 with transposed / 180-degree-rotated weight packs (anyedit_b200/training.py).
 * Activation gradients are fp16 (the caller scales the loss), statistics and parameter gradients fp32. */

/* noisy = sqrt(acp[t]) x0 + sqrt(1 - acp[t]) noise  (train.py:641 add_noise == ddpm.py:356-359); fp32 NCHW,
 * t int64 [B], tables fp32 [T] on the device. */
int anysd_q_sample_f32(const float* x0, const float* noise, const long long* t, const float* sqrt_acp,
                       const float* sqrt_1m_acp, float* out, int B, long long n_per_batch, anysd_stream_t stream);

/* F.mse_loss(pred.float(), target.float(), "mean") (train.py:696) and its gradient.  pred/target fp32 NCHW
 * [N, C, HW]; *loss = mean; d_pred fp16 NHWC [N, HW, Cpad] = grad_scale * 2 (pred - target) / numel with zero
 * padding channels (the layout the output conv's backward contraction consumes).  Deterministic two-stage sum.
 * grad_scale_dev (may be NULL): one more factor read from device memory -- the dynamic loss scale (see below). */
size_t anysd_mse_workspace_bytes(void);
int anysd_mse_loss_f32(const float* pred, const float* target, int N, int C, int HW, int Cpad, float grad_scale,
                       const float* grad_scale_dev, void* d_pred, float* loss, void* workspace, size_t workspace_bytes,
                       anysd_stream_t stream);

/* GEGLU (attention.py:49-56) un-fused for training: pre [M, 2*inner] fp16 with (a_j, gate_j) interleaved (the
 * packing of anysd_gemm_f16 act = 2), out[m, j] = a_j * gelu(gate_j); backward writes d_pre in the same layout. */
int anysd_geglu_f16(const void* pre, void* out, long long M, int inner, anysd_stream_t stream);
int anysd_geglu_bwd_f16(const void* pre, const void* d_out, void* d_pre, long long M, int inner, anysd_stream_t stream);

/* dx = dy * silu'(x), fp32 (time-embedding path, openaimodel.py:217-223, 526-530) */
int anysd_silu_bwd_f32(const float* x, const float* dy, float* dx, long long n, anysd_stream_t stream);

/* Backward of anysd_groupnorm_nhwc_f16 (util.py:202-219): x = channel concat of x1 [N,HW,C1] and x2 [N,HW,C2]
 * (x2 may be NULL), dy and dx dense [N, HW, C1+C2] fp16; statistics are recomputed. */
int anysd_groupnorm_bwd_nhwc_f16(const void* x1, int C1, const void* x2, int C2, const float* gamma, const float* beta,
                                 const void* dy, void* dx, int N, int HW, int G, float eps, int fuse_silu,
                                 anysd_stream_t stream);

/* Backward of anysd_layernorm_f16 w.r.t. x (attention.py:262-264); x, dy, dx [M, C] fp16. */
int anysd_layernorm_bwd_f16(const void* x, const float* gamma, const void* dy, void* dx, long long M, int C, float eps,
                            anysd_stream_t stream);

/* Backward of anysd_attention_f16 (CrossAttention.forward, attention.py:163-194), recomputing the probabilities
 * from q, k, v (nothing saved by the forward).  Natural-log score = qk_scale * (q . k): pass the softmax scale, or
 * ln(2) when q was packed with scale*log2(e) (aux_cols).  d_out [B, n_q, ld_do] with head h at columns
 * [h*d, (h+1)*d); q/k/v and dq/dk/dv use head_stride (padding columns of dq/dk/dv are written as zeros).
 * gate: forward's per-sample factor; d_gate[b*gate_stride] += sum(dO . attn) (atomic, fp32) when not NULL.
 * dk/dv may both be NULL (frozen text K/V).  workspace >= anysd_attention_bwd_workspace_bytes(B, heads, n_q). */
typedef struct {
    const void* q; const void* k; const void* v; const void* d_out;
    void* dq; void* dk; void* dv;
    long long q_batch_stride, k_batch_stride, v_batch_stride, do_batch_stride, dq_batch_stride, dk_batch_stride,
        dv_batch_stride;                                                       /* elements */
    int ld_q, ld_k, ld_v, ld_do, ld_dq, ld_dk, ld_dv;
    int B, heads, n_q, n_kv, d, head_stride;
    float qk_scale;
    const float* gate; int gate_stride; float* d_gate;
    int accumulate_dq;      /* 1: dq += (the experts share the text attention's q) */
    void* workspace; size_t workspace_bytes;
    const void* out;        /* optional: the forward output of exactly this attention ([B, n_q, ld_o], head h at h*d, no
                               gate, nothing accumulated into it): D = dO . O then costs one pass instead of a second
                               sweep over K/V.  NULL: recomputed. */
    long long o_batch_stride; int ld_o;
    const float* lse;       /* optional: the forward's anysd_attn_params::lse ([B, heads, n_q], base 2).  With `lse`, `out` and */
    void* dout_padded;      /* `dout_padded` (scratch, fp16 [B, n_q, heads * head_stride]) the backward runs on the tcgen05 kernels
                               (attention_bwd_tc5.cu) when the shape allows: ceil16(d) <= 64 == head_stride, n_q and n_kv multiples
                               of 128, stacked batches, no gate; otherwise both are ignored. */
} anysd_attn_bwd_params;
size_t anysd_attention_bwd_workspace_bytes(int B, int heads, int n_q);
int anysd_attention_bwd_f16(const anysd_attn_bwd_params* p, anysd_stream_t stream);

/* ---- expert streams of one cross-attention layer in one launch (restated spec, oracle/anysd_oracle.py; template
 * ip_adapter/attention_processor.py:160-176):  out += sum_e gates[b, e] * softmax(c q K_e^T) V_e.
 * kv [B, n_kv, ld_kv] holds, for expert e, K at columns [e*set_stride + h*head_stride, ...) and V v_offset columns
 * further (the layout one GEMM over the stacked to_k_ip / to_v_ip weights produces); n_kv <= 64 visual tokens.
 * qk_scale as in anysd_attention_bwd_f16.  out [B, n_q, ld_o] fp16 is accumulated onto (the text attention's output). */
typedef struct {
    const void* q; const void* kv; void* out;
    int ld_q, ld_kv, ld_o;
    int B, heads, n_q, n_kv, d, head_stride, E;
    int set_stride, v_offset;
    float qk_scale;
    const float* gates; int gate_b_stride;      /* gates[b * gate_b_stride + e] */
} anysd_expert_attn_params;
int anysd_expert_attention_f16(const anysd_expert_attn_params* p, anysd_stream_t stream);
/* backward: dq [B, n_q, ld_dq] += (onto the text attention's dq), dkv written in the layout of kv, d_gates indexed like
 * gates and accumulated atomically; workspace >= anysd_expert_attention_bwd_workspace_bytes(B, heads, E, n_q). */
size_t anysd_expert_attention_bwd_workspace_bytes(int B, int heads, int E, int n_q);
int anysd_expert_attention_bwd_f16(const anysd_expert_attn_params* p, const void* d_out, int ld_do, void* dq, int ld_dq,
                                   void* dkv, float* d_gates, void* workspace, size_t workspace_bytes,
                                   anysd_stream_t stream);

/* out[n, c] (+)= sum_rows x[n, r, c]: gradient of the per-image time-embedding row add (openaimodel.py:262-263) */
int anysd_colsum_f16(const void* x, float* out, int N, int rows, int C, int ld_out, int accumulate, anysd_stream_t stream);
/* y += x (gradient accumulation where a tensor feeds two consumers: residual / skip connections) */
int anysd_add_f16(void* y, const void* x, long long n, anysd_stream_t stream);
/* backward of anysd_concat_channels_f16 (th.cat([h, hs.pop()], 1), openaimodel.py:780) */
int anysd_split_channels_f16(const void* src, void* a, int Ca, void* b, int Cb, long long rows, anysd_stream_t stream);
/* Downsample (conv stride 2, openaimodel.py:148-150) backward = rotated conv over the zero-inserted gradient */
int anysd_zero_insert2x_f16(const void* src, void* dst, int N, int H, int W, int C, anysd_stream_t stream);
/* Upsample (nearest x2, openaimodel.py:110-115) backward = 2x2 sum pooling */
int anysd_sumpool2x_f16(const void* src, void* dst, int N, int H, int W, int C, anysd_stream_t stream);

/* Weight gradient with few rows: out[ka, kb] (+)= alpha * sum_m A[m, col(ka)] B[m, kb]; A, B fp16, out fp32.
 * Column mapping of A for logical row ka of out: group_c > 0: e = ka / group_c, c = ka % group_c, base = e * group_stride
 * (all experts of a layer in one launch); head_d > 0: padded heads, column = base + (c / head_d) * head_stride + c % head_d.
 * (dW of to_k_ip / to_v_ip: A = dK_e / dV_e, B = visual tokens; ip_adapter/attention_processor.py:160-166) */
int anysd_gemm_tn_f32(const void* A, int lda, int head_d, int head_stride, int group_c, int group_stride, const void* B,
                      int ldb, float* out, int ldo, int M, int Ka, int Kb, float alpha, int accumulate,
                      anysd_stream_t stream);

/* out[ka, m] = A[m, col(ka)] (fp16, column mapping as above), columns m in [M, ldo) zero: the K-major operand that lets
 * anysd_gemm_f16 compute the same weight gradient on the tensor cores (K = ldo >= M, a multiple of 8). */
int anysd_gather_transpose_f16(const void* A, int lda, int head_d, int head_stride, int group_c, int group_stride, void* out,
                               int ldo, int M, int Ka, anysd_stream_t stream);

/* Router backward (restated spec, oracle/anysd_oracle.py): gates = softmax(W te + b) per (sample, layer);
 * dW [L,E,D] +=, db [L,E] +=, d_te [N,D] += (atomic).  gates/d_gates fp32 [N,L,E], te fp32 [N,D], W fp16 [L,E,D]. */
int anysd_router_bwd_f32(const float* gates, const float* d_gates, const float* te, const void* W, int N, int L, int E,
                         int D, float alpha, float* dW, float* db, float* d_te, anysd_stream_t stream);
/* table_grad[idx[n], :] += alpha * src[n, :] (backward of the task-embedding gather, openaimodel.py:770-772 slot) */
int anysd_scatter_add_rows_f32(const float* src, const long long* idx, int rows, int D, int table_rows, float alpha,
                               float* table_grad, anysd_stream_t stream);

/* torch.optim.AdamW single-tensor step (train.py:486-492), step counted from 1; grad is multiplied by grad_scale
 * (1 / loss scale) before use. */
int anysd_adamw_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                    float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale,
                    anysd_stream_t stream);

/* Mixed-precision step control without host synchronisation (what accelerate's GradScaler does around train.py:694-709).
 * scaler = 4 floats on the device: {loss scale, growth tracker, optimizer steps taken, found_inf}.
 *   grad_check        found_inf = 1 when any element of grad[0..n) is inf / nan (run after the gradient all-reduce)
 *   adamw_scaled      AdamW over one flat fp32 buffer; a no-op when found_inf; step number = steps taken + 1; the gradient
 *                     is multiplied by inv_world / loss scale on the fly (the 1/world of the DDP mean, train.py:536)
 *   loss_scale_update found_inf ? (scale *= backoff, tracker = 0) : (steps += 1; ++tracker == interval -> scale *= growth);
 *                     then found_inf = 0 */
int anysd_grad_check_f32(const float* grad, long long n, float* scaler, anysd_stream_t stream);
int anysd_adamw_scaled_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                           float beta1, float beta2, float eps, float weight_decay, float inv_world, const float* scaler,
                           anysd_stream_t stream);
int anysd_loss_scale_update_f32(float* scaler, float growth, float backoff, int interval, anysd_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ANYSD_B200_H_ */
