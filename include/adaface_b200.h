/*
 * adaface_b200.h - C ABI of the B200-native AdaFace denoising hot path (libadaface_b200.so).
 *
 * The reference (askerlee/adaprompt) is 100 % Python and has no FFI layer for this path
 * (SURVEY.md section 8(b)); every op below replaces a *PyTorch library call site* inside the
 * reference modules, cited per function.  The Python host mirror of those modules
 * (adaprompt_b200/{unet,attention,ddim,...}.py) binds these symbols with ctypes - see
 * INTEGRATION.md for the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / ATen types; all pointers are DEVICE pointers
 *     unless a parameter name says host;
 *   - the library never allocates or frees device memory and keeps no state besides
 *     compiled-in tables: the caller (PyTorch) owns inputs, outputs, workspaces, KV caches;
 *   - every launch goes to the caller's stream and is CUDA-graph capturable (no host sync);
 *   - return value: 0 = ok, < 0 = bad argument / unsupported shape, > 0 = cudaError_t;
 *     af_last_error() returns the message (thread local);
 *   - activations are NHWC ("tokens x channels"); the residual stream is fp32, GEMM operands
 *     are bf16, accumulation is fp32 in TMEM.
 *   - sm_100a only.  There is no CPU fallback.
 */
#ifndef ADAFACE_B200_H
#define ADAFACE_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AF_VERSION 202
#define AF_DTYPE_F32 0
#define AF_DTYPE_BF16 1
#define AF_GN_MAX_CHUNKS 64
#define AF_PAIR_AUTO 0
#define AF_PAIR_NEVER 1
#define AF_PAIR_ALWAYS 2

typedef struct CUstream_st* af_stream_t; /* == cudaStream_t */

int af_version(void);
const char* af_last_error(void);
int af_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* Fused GEMM epilogue:  out = [geglu]( acc + bias[col] + rowbias[row / rows_per_group, col] + residual[row, col] ) */
typedef struct af_epilogue {
  const float* bias;      /* [N] or NULL (nn.Linear / nn.Conv2d bias) */
  const float* rowbias;   /* [groups, N] or NULL: per-sample time-embedding add, openaimodel.py:268-277 */
  int rows_per_group;     /* rows sharing one rowbias row (H*W); <= 0: derived for conv */
  long long ld_rowbias;   /* row pitch of rowbias in floats; <= 0: N */
  const float* residual;  /* [M, ldr] fp32 or NULL: residual adds attention.py:277,281,283,341 / openaimodel.py:279 */
  long long ldr;          /* <= 0: same as ldo */
  void* out;              /* [M, ldo] */
  long long ldo;          /* row pitch in elements; <= 0: N (N/2 for geglu) */
  int out_dtype;          /* AF_DTYPE_F32 | AF_DTYPE_BF16 */
  int geglu;              /* 1: GEGLU (attention.py:32-39): weight rows packed per 256-col tile as [128 value | 128 gate];
                             out[:, j] = (x.Wv_j + bv_j) * gelu(x.Wg_j + bg_j), N/2 bf16 output columns */
  int act;                /* 0 none; 1 quick_gelu x*sigmoid(1.702x) applied to (acc + bias) before the residual add
                             (CLIP text MLP, transformers QuickGELUActivation driven from arc2face_models.py:220) */
  float* gn_stats;        /* NULL, or [slots][N][2] fp32: per-channel (sum, sum of squares) of the values written, one
                             slot per 32 consecutive output rows (GEMM: slot = row / 32, rows-per-sample must be a
                             multiple of 32; conv: af_conv3x3_gn_slots() slots per sample).  Feeds af_groupnorm_finalize
                             so the GroupNorm that consumes this tensor never re-reads it for statistics. */
  int pair_mode;          /* tile schedule: AF_PAIR_AUTO (0) = CTA pairs (tcgen05 cta_group::2: two SMs share one 256-row tile and
                             each stages half of the weight tile) where measured to win (linear GEMMs, N tile >= 160, >= 2
                             waves), AF_PAIR_NEVER, AF_PAIR_ALWAYS (wherever legal).  Results are bit-identical between the
                             schedules (same accumulation order). */
  long long* trace;       /* NULL, or a caller-owned device buffer of >= 4*32*8 int64: timeline probe (measurement aid, results
                             unaffected) - CTA 0 records clock64 stamps [actor: TMA producer, MMA issuer, epilogue warp 0,
                             extra epilogue stamps][its first 32 tiles][8 events] */
  void* splitk_ws;        /* NULL (whole-tile schedule only), or a caller-owned device workspace whose first
                             AF_SPLITK_FLAG_BYTES are ZERO when the call is issued (the kernel leaves them zero again):
                             the tiles of the last, partial wave are cut into K ranges on different SMs, the partial fp32
                             accumulators travel through this buffer and are added in K order (bit-reproducible).  The
                             block that adds them waits for the blocks holding the other ranges: launches that pass a
                             workspace must not run CONCURRENTLY with each other on one device (stream-ordered use only;
                             concurrent GEMMs pass NULL), and never share a workspace across streams. */
  long long splitk_ws_bytes; /* size of splitk_ws; bounds the number of partial tiles (128 x BN fp32 each) */
  int split_k;            /* 0 = auto (cost model), 1 = never, n > 1 = cut every remainder tile into n K ranges (tests) */
} af_epilogue;
#define AF_SPLITK_FLAG_BYTES 16384

/* D[M,N] = [A0 | A1][M, K0+K1] . Wt[N, K0+K1]^T, bf16 operands (row-major, K contiguous), fp32 accumulate.
 * Replaces nn.Linear (attention.py:35,55,157-165) and 1x1 nn.Conv2d (attention.py:302,313; openaimodel.py:245);
 * the optional second source A1 is the skip-connection concat of openaimodel.py:1019 read in place.
 * bn_hint: 0 = auto, or 64/128/160/256 (N tile). */
int af_gemm_bf16(const void* A0, long long lda0, int K0, const void* A1, long long lda1, int K1, const void* Wt,
                 int M, int N, const af_epilogue* ep, int bn_hint, af_stream_t stream);

/* Schedule introspection (no launch, no device needed - 148 SMs are assumed without one): what af_gemm_bf16 /
 * af_conv3x3_bf16 would choose for these sizes and this epilogue.  They apply the launch's own checks of sizes and
 * epilogue options (not those of pointers, operand pitches and buffer extents): sizes or options the launch refuses
 * return its negative code and message (af_last_error).  out[0] = N-tile width, out[1] = 1 if CTA pairs,
 * out[2] = K ranges per remainder tile (1 = whole tiles only), out[3] = work units, out[4] = whole-K tiles in front of the
 * split ones, out[5] = 1 if the bf16 output leaves in 64-column epilogue items.  Host-side logic tests use these. */
int af_gemm_plan(int M, int N, int K, const af_epilogue* ep, int bn_hint, int* out);
int af_conv3x3_plan(int C0, int C1, int B, int H, int W, int Cout, int stride, const af_epilogue* ep, int bn_hint,
                    int* out);

/* 3x3 convolution, pad 1, stride 1 or 2, NHWC bf16 input(s) [B,H,W,C0] (+ [B,H,W,C1] concat), weights
 * Wt[Cout][ky][kx][C0+C1] bf16, as an implicit GEMM (no im2col buffer).  Output rows are output pixels
 * (n, oh, ow) row-major.  Replaces nn.Conv2d 3x3 at openaimodel.py:155 (stride 2), :208, :234, :120-122. */
int af_conv3x3_bf16(const void* X0, int C0, const void* X1, int C1, const void* Wt, int B, int H, int W, int Cout,
                    int stride, const af_epilogue* ep, int bn_hint, af_stream_t stream);
/* statistic slots per sample that af_conv3x3_bf16 writes for an Ho x Wo output (0: unsupported geometry). */
int af_conv3x3_gn_slots(int Ho, int Wo);
/* 3x3 convolution, stride 2, on the input padded by one zero row at the bottom and one zero column at the right
 * (F.pad(x, (0,1,0,1)) then padding 0: the VAE encoder's Downsample, ldm/modules/diffusionmodules/model.py:61-79).
 * Output pixel (oh, ow) reads input rows 2*oh .. 2*oh+2 and columns 2*ow .. 2*ow+2.  X NHWC bf16 [B,H,W,C], H and W
 * even, C % 64 == 0; Wt[Cout][ky][kx][C] bf16, Cout % 8 == 0; output [B,H/2,W/2,Cout] through the epilogue as in
 * af_conv3x3_bf16 (GroupNorm statistics: af_conv3x3_gn_slots(H/2, W/2)). */
int af_conv3x3_down01_bf16(const void* X, int C, const void* Wt, int B, int H, int W, int Cout, const af_epilogue* ep,
                           int bn_hint, af_stream_t stream);

/* Flash attention, 8-head SD-1.5 geometry (d in {40,80,160}); replaces attention.py:198-242.
 * Q [B,Nq,ldq], K [B,Nk,ldk] bf16 with head h at column h*DP (DP = 48 for d = 40, zero padded, else d);
 * Q pre-scaled by d^-1/2 * log2(e).  Vt [heads*d, ldvt] bf16 = V transposed.  Sample b's keys start at row
 * b*kv_stride of K and at column b*kv_stride of Vt (kv_stride >= Nk; the cached 77-token context uses 80).
 * key_mask [B,Nk] bytes (1 = attend) or NULL (attention.py:223-232).  Masked scores are filled with -finfo.max as in
 * the reference, so every query row of a sample whose mask keeps no key gets the mean of V over the sample's Nk keys
 * (fp32 sum, bf16 result), and lse (af_attention_bf16_lse) is +inf in those rows.  O [B,Nq,heads*d] bf16. */
int af_attention_bf16(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt, long long ldvt,
                      int kv_stride, const unsigned char* key_mask, void* O, int B, int heads, int Nq, int Nk, int d,
                      af_stream_t stream);

/* Same, also writing lse [B][heads][Nq] fp32 = log2-sum-exp of every query row (in the exp2 domain of the pre-scaled
 * scores) when lse != NULL: the backward pass recomputes P = exp2(S - lse) from it (training step, SURVEY.md 8 T1). */
int af_attention_bf16_lse(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt, long long ldvt,
                          int kv_stride, const unsigned char* key_mask, void* O, float* lse, int B, int heads, int Nq,
                          int Nk, int d, af_stream_t stream);

/* Cross-attention over <= 96 prompt tokens with the score matrix materialised (operands as af_attention_bf16): the two
 * optional behaviours of CrossAttention.forward that need the scores themselves - save_attn_vars (attention.py:245-255:
 * q_out = q * sqrt(scale) [B][heads][N][d], attnscore = sim after replacement, attn = softmax; any of them may be NULL)
 * and conv attention (attention.py:208-216): override_scores [B][heads][N][n_ov] replace the score columns ov_cols
 * [B][n_ov] (int32, -1 = keep) before the softmax.  O [B*N, heads*d] bf16 or NULL.  Scores are in the reference's domain
 * (q.k * d^-1/2). */
int af_xattn_explicit(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt, long long ldvt,
                      int kv_stride, const float* override_scores, const int* ov_cols, int n_ov, void* O, float* attn,
                      float* attnscore, float* q_out, int B, int heads, int N, int nk, int d, af_stream_t stream);
/* replace_rows_by_conv_attn (ldm/util.py:700-878) from POINTWISE scores: score fp32 [B][heads][Hf*Wf][nk] (attnscore of
 * af_xattn_explicit), cols int32 [B][ks*ks] = the prompt positions of the first ks*ks subject tokens of each sample
 * (cols[b][0] < 0: sample without the subject -> zeros).  override_scores [B][heads][Hf*Wf][ks*ks]: column m is the
 * ks x ks grouped convolution of the query map with those tokens' keys, divided by ks^1.5 and shifted by token m's
 * offset (dy, dx), zero outside the map. */
int af_conv_attn_scores(const float* score, const int* cols, int B, int heads, int Hf, int Wf, int nk, int ks,
                        float* override_scores, af_stream_t stream);

/* Backward of af_attention_bf16_lse for the long self-attention layers (d = 40 / 80, N keys = N queries, N % 128 == 0, no mask):
 * dQ, dK, dV from dO, the forward operands and the saved lse, with P / dS recomputed tile by tile in tensor memory
 * (autograd of attention.py:198-242 in the Stage-1 step, ddpm.py:2483-2532).  All matrices bf16 row-major [B*N, ld] with
 * head h at columns h*DP (DP = 48 zero-padded for d = 40, else d; dV: h*d): Q (pre-scaled, log2 domain), K, Vp = V padded, dOp = dO padded;
 * QT / KT / dOT = their [heads*48, ld >= B*N] transposes (token contiguous).  lse, delta fp32 [B][heads][N]
 * (delta_i = sum_c dO_ic O_ic).  dQ / dK [B*N, >= heads*48], dV [B*N, >= heads*40]. */
int af_attention_bwd_bf16(const void* Q, long long ldq, const void* K, long long ldk, const void* Vp, long long ldv,
                          const void* dOp, long long lddo, const void* QT, long long ldqt, const void* KT, long long ldkt,
                          const void* dOT, long long lddot, const float* lse, const float* delta, void* dQ, long long lddq,
                          void* dK, long long lddk, void* dV, long long lddv, int B, int heads, int N, int d,
                          af_stream_t stream);

/* af_attention_bf16 on the long-sequence kernel (d in {40, 80}, Nk > 128 and a multiple of 128 / 64, no mask) with an
 * in-kernel clock64 timeline - a measurement aid (scripts/attn_tile_trace.py), results are those of af_attention_bf16.
 * trace: caller-owned device buffer of 512*64*8 + 512 + 2*64*8 int64: [first 512 CTAs (linear id)][key block < 64][8]
 * stamps of softmax warp 4 (loop top, S ready, S in registers, reference decided, P buffer free, exponentials issued, P
 * handed over); then the SM id of each of those CTAs; then [MMA issuer, TMA producer of CTA 0][64][8]. */
int af_attention_bf16_trace(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt, long long ldvt,
                            int kv_stride, void* O, long long* trace, int B, int heads, int Nq, int Nk, int d,
                            af_stream_t stream);

/* GroupNorm(32) over the channel concat [x0 | x1] of fp32 NHWC tensors, optional SiLU, bf16 output
 * [B, HW, C0+C1]; optional raw bf16 copy of the concat (operand of the 1x1 skip conv).
 * Replaces GroupNorm32+SiLU (util.py:217-219; openaimodel.py:205-207,229-231,693-695) and Normalize
 * (attention.py:71-72,325).
 * Statistics format (one per source tensor): stats[(b*slots + slot)*C + c] = (sum, sum of squares) over the pixels
 * of `slot` - written by the epilogue of the GEMM / conv that produced the tensor (af_epilogue.gn_stats) or by
 * af_groupnorm_stats.  af_groupnorm_finalize -> mean_rstd [B,32,2]; af_groupnorm_apply makes the one data pass.
 * af_groupnorm_silu = stats + finalize + apply with workspace af_groupnorm_workspace_bytes(B, C0+C1).
 * All reductions run in a fixed order (bit-reproducible).
 * Accuracy: af_groupnorm_finalize takes the variance in one pass in fp32, E[x^2] - E[x]^2, so its error grows with
 * (mean/std)^2 of the group.  Worst relative rstd error measured on a B200 at a 1000 W power limit
 * (tests/test_norm_gpu.py): 2e-6 for groups with mean/std below ~3, 1.8e-4 at mean/std = 30, 1.4e-3 at 100,
 * 1.5e-2 at 300.  Up to 100 the bf16 output stays within its rounding-level limit; beyond that, centre the tensor
 * first. */
size_t af_groupnorm_workspace_bytes(int B, int C);
int af_groupnorm_stats_slots(int B, int HW);
int af_groupnorm_stats(const float* x, int C, int B, int HW, float* stats, int slots, af_stream_t stream);
int af_groupnorm_finalize(const float* stats0, int C0, int slots0, const float* stats1, int C1, int slots1, int B,
                          int HW, float eps, float* mean_rstd, af_stream_t stream);
int af_groupnorm_apply(const float* x0, int C0, const float* x1, int C1, int B, int HW, const float* mean_rstd,
                       const float* gamma, const float* beta, int silu, void* y_bf16, void* raw_bf16,
                       af_stream_t stream);
int af_groupnorm_silu(const float* x0, int C0, const float* x1, int C1, int B, int HW, const float* gamma,
                      const float* beta, float eps, int silu, void* y_bf16, void* raw_bf16, float* workspace,
                      af_stream_t stream);

/* nn.LayerNorm(C) (attention.py:267-269) on fp32 rows -> bf16. */
int af_layernorm(const float* x, long long rows, int C, const float* gamma, const float* beta, float eps, void* y_bf16,
                 af_stream_t stream);
/* same, fp32 output (CLIP final_layer_norm: arc2face_models.py:248, modules.py:370). */
int af_layernorm_f32(const float* x, long long rows, int C, const float* gamma, const float* beta, float eps, float* y,
                     af_stream_t stream);

/* First / last convolutions of the UNet (4 latent channels), fp32 CUDA-core kernels that also convert
 * between the public NCHW layout and the internal NHWC one (openaimodel.py:527-533, :693-697).  af_conv_in also takes
 * Cin = 3: the VAE encoder's conv_in on RGB images (model.py:436-440). */
int af_conv_in(const float* x_nchw, const float* w /*[Cout,Cin,3,3]*/, const float* bias, float* y_nhwc, int B, int Cin,
               int H, int W, int Cout, af_stream_t stream);
int af_conv_out(const void* x_nhwc_bf16, const float* w_packed /*[Cout,3,3,C]*/, const float* bias, float* y_nchw,
                int B, int H, int W, int C, int Cout, af_stream_t stream);

/* NHWC fp32 [B,HW,Cp] -> NCHW fp32 [B,Cout,HW] (first Cout <= 4 of the Cp padded channels): public layout of the
 * UNet output after the last conv ran on the tensor cores with Cout padded 4 -> 8 (openaimodel.py:696,1052). */
int af_nhwc_to_nchw(const float* x_nhwc, float* y_nchw, int B, int HW, int Cp, int Cout, af_stream_t stream);

/* timestep_embedding (util.py:154-174): out[b] = [cos(t_b f) | sin(t_b f)], fp32. */
int af_timestep_embedding(const float* t, float* out, int B, int dim, af_stream_t stream);

/* y[M,N] = silu_out?( silu_in?(x)[M,K] . W[N,K]^T + b ), fp32, small M (time_embed, emb_layers). */
int af_linear_small(const float* x, const float* w, const float* bias, float* y, int M, int N, int K, int silu_in,
                    int silu_out, af_stream_t stream);

int af_cast_bf16(const float* x, void* y_bf16, long long n, af_stream_t stream);
/* y[b,o,p] = bias[o] + sum_c w[o,c] * (in_scale * x[b,c,p]) over NCHW fp32 tensors with at most 4 channels: the VAE's
 * post_quant_conv applied to z / scale_factor (ldm/models/autoencoder.py:331, ldm/models/diffusion/ddpm.py:1267). */
int af_channel_mix4(const float* x_nchw, const float* w, const float* bias, float in_scale, int B, int Cin, int Cout,
                    long long HW, float* y_nchw, af_stream_t stream);
/* Posterior of the VAE encoder (DiagonalGaussianDistribution, ldm/modules/distributions/distributions.py:24-44) fused
 * with get_first_stage_encoding's scale (ddpm.py): moments NHWC fp32 [B,HW,2*zc] = (mean | logvar) per pixel.
 * lv = clamp(logvar, -30, 20); z = out_scale * (mean + exp(0.5*lv) * noise), or out_scale * mean (the mode) when noise
 * is NULL; fp32 in the reference's operation order (no contraction, full-precision exp).  noise, z, mean and logvar
 * (= lv) are NCHW fp32 [B,zc,HW]; mean / logvar may be NULL. */
int af_vae_posterior(const float* moments_nhwc, int B, long long HW, int zc, const float* noise_nchw, float out_scale,
                     float* z_nchw, float* mean_nchw, float* logvar_nchw, af_stream_t stream);
/* Row softmax of materialised scores for the VAE's single-head AttnBlock (ldm/modules/diffusionmodules/model.py:
 * 188-193: softmax(q.k^T * c^-1/2, dim=2)): y[r][0..n) = softmax(scale * x[r][0..n)), fp32 in, bf16 out, n <= 16384. */
int af_softmax_rows(const float* x, long long ldx, long long rows, int n, float scale, void* y_bf16, long long ldo,
                    af_stream_t stream);
/* F.interpolate(scale_factor=2, mode="nearest") (openaimodel.py:120) fused with the bf16 cast. */
int af_upsample2x_cast(const float* x_nhwc, void* y_bf16, int B, int H, int W, int C, af_stream_t stream);

/* CFG combine + DDIM update (ddim.py:260,279,283,295), reference fp32 operation order.
 * coef_table rows of 8 floats [g, sqrt(1-a_t), sqrt(a_t), sqrt(a_prev), sqrt(1-a_prev-sigma^2), sigma, temperature, 0]
 * (the noise term is (sigma * noise) * temperature, ddim.py:286); row = *step_idx (device) or 0 when step_idx is NULL.
 * eps = [cond ; uncond] when has_uncond.  x and x_prev may be the same buffer. */
int af_cfg_ddim_update(const float* x, const float* eps, int has_uncond, const float* noise, const float* coef_table,
                       const int* step_idx, float* x_prev, float* pred_x0, long long n, af_stream_t stream);
int af_advance_step(int* step_idx, const float* t_table, float* t_buf, int B, int num_steps, af_stream_t stream);

/* ---- conditioning path: CLIP text transformer pieces and AdaFace token splicing (once per prompt) ---- */

/* Causal / full multi-head attention for short sequences (CLIP text: 12 heads x 64, L <= 77).  qkv bf16 [B*L, ldq]:
 * q at column 0, k at k_off, v at v_off; head h of q at h*64.  mult > 1 = CLIPAttentionMKV
 * (adaface/arc2face_models.py:87-173): token t contributes `mult` keys/values, key (t, r) of head h at column
 * k_off + (h*mult + r)*64, masked like token t.  scale multiplies q (head_dim^-1/2).  out bf16 [B*L, ldo]. */
int af_attention_small(const void* qkv, long long ldq, int k_off, int v_off, void* out, long long ldo, int B,
                       int heads, int L, int mult, float scale, int causal, af_stream_t stream);
/* out[r,:] = table[ids[r],:] (token_embedding lookup, exact copies; ids are int64 as torch.long). */
int af_gather_rows(const float* table, const long long* ids, float* out, long long rows, int dim, int vocab,
                   af_stream_t stream);
/* x[b,t,:] += pos[t,:] (CLIPTextEmbeddings position add, modules.py:213-221). */
int af_add_pos(float* x, const float* pos, long long rows, int L, int dim, af_stream_t stream);
/* first[r] = first position of `token` in ids[r,:] or -1 (embedding_manager.py:1359,1368). */
int af_find_first_token(const long long* ids, int rows, int L, long long token, int* first, af_stream_t stream);
/* dst[r, start[r]+k, :] = src[src_index ? src_index[r] : r, k, :], k < K, rows with start[r] < 0 untouched
 * (embedding_manager.py:1516-1562; adaface/util.py:107,184).  Exact row copies: bit-exact by construction. */
int af_splice_rows(float* dst, const float* src, const int* start, const int* src_index, int rows, int L, int K,
                   int dim, af_stream_t stream);
/* out = w0*a + w1*b (+ w2*c): weighted sum of the last hidden states (arc2face_models.py:236-246, modules.py:361-368),
 * evaluated as ((w0*a + w1*b) + w2*c) like (stack * w).sum(0). */
int af_weighted_sum(const float* a, const float* b, const float* c, float w0, float w1, float w2, float* out,
                    long long n, af_stream_t stream);

/* ---- Stage-1 distillation step (SURVEY.md section 8 row T1): backward kernels.  The reference gets these from
 * torch.autograd over the modules cited above (guided_denoise ddpm.py:2483-2532 -> UNetModel.forward with grad; UNet
 * weights frozen ddpm.py:783-786).  dgrad GEMMs / convolutions reuse af_gemm_bf16 / af_conv3x3_bf16 on transposed
 * weight packs; the entry points below are the remaining pieces. ---- */

/* Batched strided C[z] = epi(A[z][M,K] . B[z][N,K]^T), z = b0*nb1 + b1, bf16 operands, fp32 accumulate
 * (mma.sync tiles; attention backward per (sample, head): autograd of attention.py:198-242).
 * mode 0: alpha*acc | 1: exp2(acc - vec[row]) | 2: exp2(acc - vec[col]) | 3: alpha*P[row,col]*(acc - vec[row]) |
 * 4: alpha*P[row,col]*(acc - vec[col]).  Entries with row >= valid_rows or col >= valid_cols are written as 0.
 * All strides in elements; operand pitches / batch strides multiples of 8, K % 8 == 0, N even. */
typedef struct af_bgemm {
  const void* A; long long lda, sA0, sA1;
  const void* B; long long ldb, sB0, sB1;
  void* C; long long ldc, sC0, sC1; int c_dtype;
  const float* vec; long long sV0, sV1;
  const void* P; long long ldp, sP0, sP1;
  int M, N, K, nb0, nb1, mode, valid_rows, valid_cols;
  float alpha;
} af_bgemm;
int af_bgemm_bf16(const af_bgemm* g, af_stream_t stream);

/* GroupNorm(32)(+SiLU) backward w.r.t. the fp32 input: x [B,HW,C], mean_rstd [B,32,2] (af_groupnorm_finalize),
 * dy bf16 [B,HW,C] (gradient of the bf16 output), dres fp32 or NULL (added: gradient of a residual branch), dx fp32.
 * workspace: af_groupnorm_bwd_workspace_floats(B, C, HW) floats.  Deterministic. */
size_t af_groupnorm_bwd_workspace_floats(int B, int C, int HW);
int af_groupnorm_bwd(const float* x, int C, int B, int HW, const float* mean_rstd, const float* gamma, const float* beta,
                     int silu, const void* dy_bf16, const float* dres, float* dx, float* workspace, af_stream_t stream);
/* nn.LayerNorm backward: dx = LN'(x)^T dy (+ dres); dy bf16 or fp32 (dy_dtype); dgamma / dbeta (both or neither) are
 * ACCUMULATED with fp32 atomics (trainable CLIP text LayerNorms of SubjBasisGenerator.prompt2token_proj). */
int af_layernorm_bwd(const float* x, long long rows, int C, const float* gamma, float eps, const void* dy, int dy_dtype,
                     const float* dres, float* dx, float* dgamma, float* dbeta, af_stream_t stream);
/* GEGLU in its unfused training form (attention.py:32-39): proj bf16 [T,2F] = (value | gate) -> h bf16 [T,F]. */
int af_geglu_fwd(const void* proj, long long T, int F, void* h, af_stream_t stream);
int af_geglu_bwd(const void* proj, const void* dh, long long T, int F, void* dproj, af_stream_t stream);
/* quick_gelu: out = x*sigmoid(1.702x) (dy NULL) or its derivative times dy; bf16. */
int af_quick_gelu(const void* x, const void* dy, long long n, void* out, af_stream_t stream);
/* delta[b][h][q] = sum_c a[b,q,h*d+c] * b[b,q,h*d+c] (rowsum(dO o O) of the softmax backward); a, b bf16 [B*N, heads*d]. */
int af_rowdot_heads(const void* a, const void* b, int B, int N, int heads, int d, float* delta, af_stream_t stream);
/* backward of af_attention_small: dqkv bf16 in the layout of qkv, from dout bf16 [B*L, ldo]. */
int af_attention_small_bwd(const void* qkv, long long ldq, int k_off, int v_off, const void* dout, long long ldo,
                           void* dqkv, int B, int heads, int L, int mult, float scale, int causal, af_stream_t stream);
/* dgrad of UNetModel.out[2] (openaimodel.py:696): dout NCHW fp32 [B,Cout,H,W], w fp32 [Cout,C,3,3] -> dy bf16 NHWC. */
int af_conv_out_dgrad(const float* dout_nchw, const float* w, int B, int H, int W, int C, int Cout, void* dy_bf16,
                      af_stream_t stream);
/* backward of nearest x2 upsampling (openaimodel.py:120): in fp32 [B,2H,2W,C] -> out [B,H,W,C] (2x2 sums). */
int af_sumpool2x2(const float* in, int B, int H, int W, int C, float* out, af_stream_t stream);
/* operand of the stride-2 conv dgrad (openaimodel.py:155): in fp32 [B,H,W,C] -> out bf16 [B,2H,2W,C], zeros inserted. */
int af_zero_insert2x(const float* in, int B, int H, int W, int C, void* out_bf16, af_stream_t stream);
/* out bf16 [C][ldo] = in[R][C]^T (in fp32 or bf16), zero padded to ldo columns: weight-gradient GEMM operands. */
int af_transpose_to_bf16(const void* in, int in_dtype, int R, int C, long long ldo, void* out_bf16, af_stream_t stream);

/* Prodigy optimizer step over one flat fp32 parameter bucket (ldm/prodigy.py:97-256; the trainer's optimizer,
 * ddpm.py configure_optimizers).  Pass 1 updates exp_avg / exp_avg_sq / s (:182-188) and ADDS g.(p0-p) and sum|s| into
 * sums[0..1] (double; :179,:189 - the caller zeroes them and derives d, :212-216); pass 2 applies the decoupled weight
 * decay and the Adam-style update (:240-248) with the new d. */
int af_prodigy_moments(const float* p, const float* grad, const float* p0, float* s, float* exp_avg, float* exp_avg_sq,
                       long long n, float beta1, float beta2, float beta3, float d, float s_alpha, float coupled_decay,
                       double* sums, af_stream_t stream);
int af_prodigy_apply(float* p, const float* exp_avg, const float* exp_avg_sq, long long n, float dlr, float d_eps,
                     float decoupled_decay, af_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ADAFACE_B200_H */
