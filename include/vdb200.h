/* vdb200 — C ABI of the B200-native Versatile-Diffusion sampling hot path (libvdb200.so).
 *
 * The reference (SHI-Labs/Versatile-Diffusion) has no FFI/operator boundary: its hot path is eager
 * PyTorch inside lib/model_zoo (SURVEY.md §8b).  This header is the boundary a maintainer binds
 * instead: every entry point replaces the arithmetic of one reference call site (cited per function),
 * takes raw device pointers + explicit sizes + a cudaStream_t (passed as void*), allocates nothing,
 * keeps no global state besides a thread-local error string and a launch counter, and returns an
 * int status (0 = ok).  Python binding: versatile-diffusion_b200/vdb200/_lib.py (ctypes); the
 * reference-side stubs are shown in INTEGRATION.md.
 *
 * Conventions
 *   - activations: bf16, NHWC / token-major ([B, H, W, C] == [B*H*W, C]); latents/images fp32.
 *   - weights: bf16 [N, K] row-major (K contiguous); conv weights repacked to [Cout, (ky,kx,ci)].
 *   - all device pointers 16-byte aligned; leading dimensions in ELEMENTS.
 *   - `stream` is a cudaStream_t; kernels are stream-ordered and CUDA-graph capturable.
 */
#ifndef VDB200_H_
#define VDB200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { VDB_OK = 0, VDB_ERR_INVALID = 1, VDB_ERR_CUDA = 2, VDB_ERR_UNSUPPORTED = 3 };
enum { VDB_ACT_NONE = 0, VDB_ACT_SILU = 1, VDB_ACT_GELU = 2, VDB_ACT_QUICK_GELU = 3, VDB_ACT_GEGLU = 4,
       VDB_ACT_GELU_TANH = 5 /* GPT-2's tanh-form GELU, optimus_gpt2.py:99-100 */,
       VDB_ACT_TANH = 6 /* BertPooler's tanh, optimus_bert.py:364-376 */ };

/* ---- library state ------------------------------------------------------------------------- */
const char* vdb_version(void);
const char* vdb_last_error(void);        /* message of the last non-zero status on this thread */
long long vdb_launch_count(void);        /* kernels launched by this library since the last reset */
void vdb_reset_launch_count(void);
int vdb_num_sms(void);

/* ---- K4: CFG mix + DDIM update — DDIMSampler.p_sample_ddim, lib/model_zoo/ddim.py:144-171 ------
 * e = e_u + scale*(e_c - e_u); pred_x0 = (x - sqrt(1-a_t) e)/sqrt(a_t);
 * x_prev = sqrt(a_prev) pred_x0 + sqrt(1 - a_prev - sigma^2) e + sigma*noise*temperature.
 * coef: device fp32 {a_t, a_prev, sigma_t, sqrt_one_minus_a_t}[, more rows]; step_idx (device int,
 * may be NULL) selects the row, so one captured CUDA graph serves every step. e_uncond/noise/pred_x0
 * may be NULL (scale==1 path, eta==0, no pred_x0 wanted). x_prev may alias x (in place); x_prev_dup (may be
 * NULL) receives a second copy — the cond half of the next step's torch.cat([x]*2) (ddim.py:144).
 * fp32, bit-identical to the reference ops. */
int vdb_ddim_cfg_step(const float* e_uncond, const float* e_cond, const float* x, const float* noise,
                      const float* coef, const int* step_idx, float scale, float temperature, float* x_prev,
                      float* x_prev_dup, float* pred_x0, long long n, void* stream);
/* y = a*x + b*z, fp32 — VD_v2_0.q_sample (vd.py:221-224) for the img2img start (ddim.py:97-103) */
int vdb_axpby_f32(const float* x, const float* z, float a, float b, float* y, long long n, void* stream);
int vdb_add_int(int* p, int delta, void* stream); /* device-side step counter update */
/* y = c0*x0 + c1*x1 + c2*x2 + c3*x3 (x1..x3 may be NULL), fp32 — PLMS eps extrapolation (north-star addition: the
 * reference has no PLMS sampler; formula of Liu et al. 2022 / CompVis latent-diffusion plms.py) */
int vdb_lincomb4_f32(const float* x0, const float* x1, const float* x2, const float* x3, float c0, float c1, float c2,
                     float c3, float* y, long long n, void* stream);

/* ---- tcgen05 GEMM — nn.Linear / 1x1 conv call sites: attention.py:37-64,161-193,237,249;
 *      autokl_modules.py:150-202; HF CLIP q/k/v/out/fc1/fc2 (clip.py:58-61,92-100) ----------------
 * out[M,N] = act(alpha * ([A | A2] @ W^T + bias)) + resid.   A [M,K] (lda), optional A2 [M,K2] (lda2)
 * concatenated along K, W [N, K+K2] (ldw).  bias fp32 [N] (bias_bstride==0) or per-batch rows
 * [.., N] selected by row / rows_per_batch.  act = VDB_ACT_*; VDB_ACT_GEGLU expects W/bias rows packed
 * per 256-column tile as 128 value rows then their 128 gate rows and writes N/2 columns
 * (GEGLU.forward, attention.py:42-44).  out bf16 (out_f32==0) or fp32.  bn: 0 = auto, else force
 * tile N in {64,128,160,256}.  ksplit: 0 = auto, 1 = off; split-K needs workspace >= ksplit*M*N*4 B. */
int vdb_gemm_bf16(const void* A, long long M, long long K, long long lda, const void* A2, long long K2,
                  long long lda2, const void* W, long long N, long long ldw, const float* bias,
                  long long bias_bstride, long long rows_per_batch, const void* resid, long long ldr, void* out,
                  long long ldo, int out_f32, int act, float alpha, int bn, int ksplit, void* workspace,
                  size_t ws_bytes, void* stream);

/* ---- the same GEMM with a LayerNorm folded in — BasicTransformerBlock norm1/2/3, attention.py:206-208,214-218 -------------
 * CONSUMER (ln_stats != NULL):  out = act( LN(x) W0^T + b0 )  computed from the RAW x without ever forming LN(x):
 *     out[m,n] = act( rstd[m] * (x W^T - mean[m] * ln_colsum[n]) + bias[n] )
 *   with W = W0 * gamma (per input channel, rounded to bf16), ln_colsum[n] = sum_k float(W[n,k]), bias[n] = b0[n] + sum_k beta_k W0[n,k]
 *   prepared once by the caller.  mean / rstd come from ln_stats = [ln_parts][ln_rows][2] fp32 partial (sum, sum of squares) over
 *   disjoint column ranges of x's rows (written by a PRODUCER launch below, which reports ln_parts), ln_dim == K = the LayerNorm width,
 *   ln_eps its epsilon.
 *   ln_on_cols = 1: x is the W-side operand (out^T = W0 LN(x)^T, the transposed V^T projection): A holds the prepared weights, the
 *   statistics belong to the output COLUMNS, ln_colsum is indexed by the output ROW and ln_rowbias[m] (may be NULL) carries the beta term.
 *   act: VDB_ACT_NONE or VDB_ACT_GEGLU (packed as for vdb_gemm_bf16; ln_colsum packed like bias).  No residual.
 * PRODUCER (stats_out != NULL):  out = A W^T + bias + resid as vdb_gemm_bf16, and stats_out (room for [2 * ceil(N/64)][M][2] fp32)
 *   receives *stats_parts partial (sum, sum of squares) per output row (fp32 values before the bf16 rounding; one partial per N tile
 *   and epilogue warp, so *stats_parts = 2 * N tiles is known on the host when the call returns), N % 32 == 0.
 * Exactly one of ln_stats / stats_out; bf16 out, 16-byte aligned out / resid rows; needs the TMA-store epilogue (VDB_EPI_TMA != 0). */
int vdb_gemm_ln_bf16(const void* A, long long M, long long K, long long lda, const void* W, long long N, long long ldw,
                     const float* bias, const void* resid, long long ldr, void* out, long long ldo, int act,
                     const float* ln_stats, long long ln_rows, int ln_parts, int ln_dim, float ln_eps, const float* ln_colsum,
                     int ln_on_cols, const float* ln_rowbias, float* stats_out, int* stats_parts, int bn, void* stream);

/* ---- skinny GEMM on the CUDA cores for a small operand of <= 64 rows — the 0-D diffuser's Linear_MultiDim / FCBlock_MultiDim GEMMs
 *      (openaimodel.py:2084-2141, 2275-2354; M = batch rows) and the 32-row projections of its context blocks --------------------
 * small = [S, K1 (+K2)] bf16 rows (two sources concatenated along K, small2 may be NULL), big = [R, K1+K2] bf16 rows, fp32 accumulate.
 * transpose_out 0:  out[s, r] = small[s] . big[r] + bias[s * bias_bstride + r] + resid[s, r]     (activations x weights^T)
 * transpose_out 1:  out[r, s] = small[s] . big[r]                                               (no bias / residual: V^T projection)
 * The small operand must fit shared memory: vdb_gemm_skinny_fits(S, K) != 0 (S padded to 8 / 16 / 32 / 64 rows x K x 2 B <= 200 KB). */
int vdb_gemm_skinny_fits(int S, long long K);
int vdb_gemm_skinny_bf16(const void* small1, int S, long long K1, long long lds1, const void* small2, long long K2, long long lds2,
                         const void* big, long long R, long long ldb, const float* bias, long long bias_bstride,
                         const void* resid, long long ldr, void* out, long long ldo, int transpose_out, void* stream);

/* ---- tcgen05 implicit-GEMM 3x3 conv on NHWC — ResBlock convs openaimodel.py:203,229; Downsample
 *      :150-152; Upsample.conv :105; VAE autokl_modules.py:48-76,93-111 ---------------------------
 * mode 0: stride 1 pad 1; mode 1: stride 2 pad 1; mode 2: stride 2 with pad (0,1,0,1) (VAE).
 * mode 3 + 2*py + px: parity (py,px) of "nearest 2x upsample then 3x3 conv" (Upsample.forward, openaimodel.py:107-117;
 *      autokl_modules.py:54-58) evaluated on the SOURCE image with the 9 taps folded into 2x2: X = source [B,H,W,C],
 *      out = [B,H,W,N] (that parity sub-lattice), Wt = [N, 4*C] (ty,tx,c) pre-summed on the host; no skip inputs.
 *      vdb_interleave2x2_nhwc assembles the four parities into [B,2H,2W,N].
 * mode 7 + 2*py + px: the same parity conv, but `out` is the full [B,2H,2W,N] tensor and the tile is stored straight into pixels
 *      (2y+py, 2x+px) through the output tensor map (no interleave pass, no parity temporaries); bf16 out, no residual / skips /
 *      split-K, N % 32 == 0 (needs the TMA-store epilogue).
 * Wt [N, 9*C + Cs1 + Cs2], K order (ky,kx,c) then the 1x1 skip_connection columns whose inputs
 * skip1/skip2 (raw NHWC at output resolution; the two halves of torch.cat([h, hs.pop()]),
 * vd.py:372) are accumulated into the same TMEM tile (ResBlock.skip_connection, openaimodel.py:240).
 * bias/resid/out/act as vdb_gemm_bf16 with rows_per_batch = Hout*Wout. C, Cs1, Cs2 multiples of 64. */
int vdb_conv3x3_bf16(const void* X, int B, int H, int W, int C, int mode, const void* Wt, int N, long long ldw,
                     const void* skip1, int Cs1, const void* skip2, int Cs2, const float* bias,
                     long long bias_bstride, const void* resid, long long ldr, void* out, long long ldo,
                     int out_f32, int act, int bn, int ksplit, void* workspace, size_t ws_bytes, void* stream);

/* ---- tcgen05/TMEM flash attention — CrossAttention.forward, attention.py:178-192 -----------------
 * O = softmax(Q K^T * scale) V per (batch, head), fp32 online softmax, nothing materialised.
 * Q [B*Nq, ldq] head h at columns q_col0 + h*DK; K [B*Nk, ldk] at k_col0 + h*DK;
 * Vt [H*DVP, ldv] row h*DVP + c, column b*Nk + j; out [B*Nq, ldo] head h at columns h*d_head.
 * DK = vdb_attention_dk_pad(d_head), DVP = vdb_attention_dv_pad(d_head): (64, 48) up to d_head 48, (64, 64) up to 64,
 * (128, 80) up to 80, (192, 160) up to 160 (d_head a multiple of 8); pad columns/rows must be
 * zero (the projection weights are zero-padded at pack time). causal != 0: CLIP text mask.
 * Batch b starts at row b*q_bstride of Q/out and at row (K) / column (Vt) b*kv_bstride; kv_bstride must be a
 * multiple of 8 (TMA: 16-byte aligned innermost coordinate), so ragged contexts (77, 257 tokens) are stored
 * padded to 80 / 264 per batch item; the pad keys are masked by Nk. 0 = dense (stride = count). */
int vdb_attention_dk_pad(int d_head);
int vdb_attention_dv_pad(int d_head);
int vdb_attention_bf16(const void* Q, long long ldq, int q_col0, const void* K, long long ldk, int k_col0,
                       const void* Vt, long long ldv, void* out, long long ldo, int B, int H, int Nq, int Nk,
                       int q_bstride, int kv_bstride, int d_head, float scale, int causal, void* stream);
/* The same attention with a key count per batch item — BertSelfAttention with the padding mask of
 * BertForLatentConnector_XX.forward (optimus_bert.py:1349-1439), whose keys are a prefix [CLS] .. [SEP] of every padded row.
 * kv_len: device int [B]; batch item b attends to keys j < kv_len[b] only (values clamped to [1, Nk]).  The reference adds
 * -10000 to the scores of the pad keys instead; with at least one real key in the row ([CLS] always is) exp(s - 10000 - max)
 * is exactly 0 in fp32 for any score range a trained BERT produces, so leaving those keys out is the same softmax.  Runs the
 * single-tile kernel only, d_head 49..64 (BERT's 64); with every kv_len[b] == Nk the result equals vdb_attention_bf16's bit for bit. */
int vdb_attention_keylen_bf16(const void* Q, long long ldq, int q_col0, const void* K, long long ldk, int k_col0,
                              const void* Vt, long long ldv, void* out, long long ldo, int B, int H, int Nq, int Nk,
                              int q_bstride, int kv_bstride, int d_head, float scale, int causal, const int* kv_len,
                              void* stream);

/* ---- GroupNorm(32) [+SiLU] [+channel concat] on NHWC — normalization()/Normalize():
 *      diffusion_utils.py:168-191 (eps 1e-5), attention.py:76-77 & autokl_modules.py:38-39 (1e-6) ----
 * y[B,HW,C1+C2] = act(GN32(cat(x1,x2))).  scratch: ZERO-INITIALISED device buffer of
 * vdb_groupnorm_scratch_floats(B,HW) floats (partial sums, finalised mean/rstd, per-batch arrival counters); it may
 * be reused by later calls on the same stream (the kernels leave the counters at zero). Deterministic: no float atomics. */
int vdb_groupnorm_nsplit(int B, int HW);
long long vdb_groupnorm_scratch_floats(int B, int HW);
int vdb_groupnorm_nhwc(const void* x1, int C1, const void* x2, int C2, int B, int HW, int groups, const float* gamma,
                       const float* beta, float eps, int act, float* scratch, void* y, void* stream);

/* ---- LayerNorm over the last dim — BasicTransformerBlock.norm1/2/3 attention.py:206-208 ---------- */
int vdb_layernorm(const void* x, long long rows, int C, const float* gamma, const float* beta, float eps, void* y,
                  void* stream);

/* ---- nearest 2x upsample NHWC — Upsample.forward openaimodel.py:114, autokl_modules.py:54 -------- */
int vdb_upsample2x_nhwc(const void* x, int B, int H, int W, int C, void* y, void* stream);

/* ---- CLIP image preprocessing on the device — replaces the host PIL round trip of CLIPImageContextEncoder._encode,
 *      clip.py:88-94 (ToPILImage + CLIPProcessor: bicubic resize of the shortest side to 224, centre crop, rescale, normalise).
 *      Bit-exact with torchvision.ToPILImage + Pillow's 8-bit two-pass bicubic resampling; the int32 coefficient tables
 *      (bounds [out,2] = first tap, tap count; kk [out,ksize], 22 fractional bits) come from the host.  mean3 / std3 are HOST arrays. */
int vdb_clip_to_u8_hwc(const float* x, int n, int H, int W, void* y /* u8 [n,H,W,3] */, void* stream);
int vdb_resample_h_u8(const void* x /* u8 [n,H,Win,3] */, int n, int H, int Win, int Wout, const int* bounds, const int* kk,
                      int ksize, void* y /* u8 [n,H,Wout,3] */, void* stream);
int vdb_resample_v_crop_norm(const void* x /* u8 [n,Hin,W,3] */, int n, int Hin, int W, const int* bounds, const int* kk,
                             int ksize /* 0: no vertical resize */, int top, int left, int S, const float* mean3,
                             const float* std3, float* y /* fp32 [n,3,S,S] */, void* stream);

/* [4 parities (py,px)][B,H,W,C] bf16 -> [B,2H,2W,C]: out[b,2y+py,2x+px,:] = src[py*2+px][b,y,x,:] (see conv mode 3..6). */
int vdb_interleave2x2_nhwc(const void* src, int B, int H, int W, int C, void* y, void* stream);

/* ---- im2col for tiny-Cin 3x3 convs (latent 4ch / RGB 3ch inputs): fp32 NHWC -> bf16 [B*H*W, Kpad]
 *      (x*in_scale + in_shift applied first: AutoencoderKL.encode's x*2-1, autokl.py:34) ----------- */
int vdb_im2col3x3_small(const float* x, int B, int H, int W, int Cin, int Kpad, float in_scale, float in_shift,
                        void* y, void* stream);

/* ---- fp32 NCHW <-> NHWC permute with y = x*mul + add [clamped to [0,1]] (autokl.py:47) ------------ */
int vdb_permute_f32(const float* x, int B, int C, long long HW, int to_nhwc, float mul, float add, int clamp01,
                    float* y, void* stream);
/* DiagonalGaussianDistribution.sample (distributions.py:24-37) fused with the latent scale of vae_encode
 * (vd.py:282-289): z = (mean + exp(0.5*clamp(logvar,-30,20)) * noise) * post_mul on NHWC fp32 moments [npix,2C] */
int vdb_gaussian_sample(const float* moments, const float* noise, int C, long long npix, float post_mul, float* z,
                        void* stream);
int vdb_cast_f32_bf16(const float* x, void* y, long long n, void* stream);
/* tiny 1x1 conv on fp32 NHWC: y = W (x*pre_mul) + b — quant_conv / post_quant_conv, autokl.py:26-27,36,45 and
 * the 1/latent_scale_factor of VD_v2_0.vae_decode, vd.py:291-296 */
int vdb_pointwise_small(const float* x, long long npix, int Cin, int Cout, const float* Wm, const float* bias,
                        float pre_mul, float* y, void* stream);
int vdb_cast_bf16_f32(const void* x, float* y, long long n, void* stream);

/* ---- timestep_embedding [cos|sin] — diffusion_utils.py:131-151 ---------------------------------
 * ts: device int64 [B], or a table indexed by *step_idx (broadcast to all B rows) when step_idx != NULL.
 * neg_log_period = (float)(-ln(max_period)). */
int vdb_timestep_embedding(const long long* ts, const int* step_idx, int B, int dim, float neg_log_period,
                           float* out, void* stream);

/* ---- skinny linear (M <= 16) — time_embed openaimodel.py:2629-2633, ResBlock.emb_layers :217-223 --
 * out[M,N] = act_out(act_in(x)[M,K] @ W[N,K]^T + bias); x/out fp32, W bf16; act 0 none, 1 SiLU. */
int vdb_linear_small(const float* x, int M, int K, const void* Wt, int N, const float* bias, int act_in, int act_out,
                     float* out, void* stream);

/* ---- CLIP context-encoder front/back ends — CLIPTextContextEncoder.encode clip.py:53-62, CLIPImageContextEncoder
 *      ._encode / ._encode_wmask clip.py:88-143 (the arithmetic of transformers.CLIPModel around the encoder layers,
 *      which run on vdb_layernorm / vdb_gemm_bf16 / vdb_attention_bf16).  Token streams are bf16 [B, Lp, C] with
 *      Lp = L rounded up to a multiple of 8 and zero pad rows. ------------------------------------------------- */
/* x[b,n] = token_embedding[tokens[b,n]] + position_embedding[n] */
int vdb_clip_text_embed(const long long* tokens, const float* tok_emb, const float* pos_emb, int B, int L, int Lp, int C,
                        void* x, void* stream);
/* PxP patches of NCHW fp32 pixels -> bf16 [B*(HW/P)^2, Kpad] rows in the patch_embedding conv's (c,py,px) order */
int vdb_patchify(const float* pixels, int B, int Cin, int HW, int P, int Kpad, void* y, void* stream);
/* [class_embedding ; patch embeddings] + position_embedding, optional per-token scale (masked variant) */
int vdb_vit_assemble(const void* patches, const float* cls, const float* pos, const float* tok_scale, int B, int L, int Lp,
                     int C, void* x, void* stream);
/* out[b,n,:] = z[b,n,:] / ||z[b, idx[b], :]|| [* row_scale[b,n]], fp32 [B,L,C] (idx NULL = token 0) */
int vdb_scale_by_row_norm(const void* z, const int* idx, const float* row_scale, int B, int L, int Lp, int C, float* out,
                          void* stream);

/* ---- row softmax (VAE AttnBlock, autokl_modules.py:186-188) ------------------------------------- */
int vdb_softmax_rows(const void* x, long long rows, int n, long long ld, float scale, void* y, void* stream);

/* ---- per-position affine + activation (text-latent flow, SURVEY §8f rank 4): y[r,i] = act(x[r,i] * gamma[i] + beta[i]) on bf16
 *      rows with fp32 parameters — the affine half of FCBlock's GroupNorm32 (openaimodel.py:2100-2112), whose gamma / beta are
 *      indexed by the FLATTENED channel c*sdim + s while vdb_groupnorm_nhwc normalises per channel c.  act 0 none, 1 SiLU. ---- */
int vdb_affine_act_rows(const void* x, long long rows, int n, const float* gamma, const float* beta, int act, void* y, void* stream);

/* ---- load-time weight repack (SURVEY §8b `vdb_pack_conv_weight`): checkpoint tensors in the reference's layouts (fp32,
 *      contiguous: Conv2d [Cout,Cin,kh,kw], Linear [out,in]) -> the bf16 K-major layouts the kernels above consume, so a
 *      binder that keeps the reference's own nn.Modules needs none of this repo's Python.  All device pointers. ------------ */
/* Conv2d weight [Cout, Cin, kh, kw] -> out[n, col0 + (ky*kw + kx)*Cin + ci] (row stride ldo): 3x3 convs of ResBlock.in_layers[2] /
 * out_layers[3] / Downsample.op / Upsample.conv (openaimodel.py:89-274) with col0 = 0, ldo = 9*Cin [+ Cskip]; a channel-changing
 * ResBlock's 1x1 skip_connection (:233-240) is appended as extra K columns with kh = kw = 1, col0 = 9*Cout_of_conv1. */
int vdb_pack_conv_weight(const float* w, int Cout, int Cin, int kh, int kw, void* out, long long ldo, long long col0, void* stream);
/* GEGLU.proj (attention.py:37-45) weight [2*n2, K] + bias [2*n2] -> rows interleaved per 256-row tile (128 value rows, then
 * their 128 gate rows) as the ACT_GEGLU epilogue of vdb_gemm_bf16 expects; n2 % 128 == 0. */
int vdb_pack_geglu(const float* w, const float* b, int n2, int K, void* w_out, float* b_out, void* stream);
/* CrossAttention.to_q / to_k / to_v weight [H*d, K] (attention.py:152-168) -> [H*dpad, K] with zero rows after each head's d
 * rows; dpad = vdb_attention_dk_pad(d) for q / k, vdb_attention_dv_pad(d) for v. */
int vdb_pad_heads(const float* w, int H, int d, int dpad, int K, void* out, void* stream);

/* ---- Optimus GPT-2 text decode with a KV cache — optimus_vae_next.decode / sample_single_sequence_conditional
 *      (lib/model_zoo/optimus.py:662-688, 745-763) on GPT2ForLatentConnector_XX (optimus_models/optimus_gpt2.py:813-1112).
 *      The reference re-runs the whole prefix per token; these kernels keep a per-layer bf16 KV cache [n, H, 32, 64] instead.
 *      `step` is a device int: the index t (0 = <BOS>) of the token being processed, so one captured graph serves every step
 *      (advance it with vdb_add_int). Sequences hold at most 30 tokens (max_length of optimus.py:751). -------------------- */
/* Single-query attention of token t (Attention.forward / _attn, optimus_gpt2.py:151-209), d_head 64, any H:
 * appends k, v of qkv[row] = [q | k | v] (each H*64, the c_attn output) at slot t of kcache / vcache, then attends over
 * key 0 = the latent memory mem[row, h*64 ..] (a layer's slice of linear(z), used as past key AND value, :887-893) and the
 * cached tokens 0..t; out[row, h*64 ..] = softmax(q k^T * scale) v (fp32 softmax).  ldqkv, ldmem multiples of 8. */
int vdb_kv_decode_attention(const void* qkv, long long ldqkv, const void* mem, long long ldmem, void* kcache, void* vcache,
                            const int* step, int n, int H, float scale, void* out, long long ldo, void* stream);
/* One CTA per row: p = softmax(logits[row, :V] / *temperature) (fp32, fixed-order sums), token = smallest i with
 * cumsum(p)[i] > u (torch.multinomial's draw, optimus.py:678, without the top_p = 1.0 filter, which only drops tokens whose
 * fp32 cumulative sum rounds above 1).  u = uniforms[row * ldu + t] when uniforms != NULL, else Philox4x32-10 keyed by *seed
 * with counter (row, t).  A row whose token t is eos stays at eos; a token landing at index max_len-1 becomes eos (:680-685).
 * forced != NULL ([n, ldt] int32): take forced[row, t+1] instead of sampling (teacher forcing).  Writes tokens[row, t+1] and,
 * when x_next != NULL, x_next[row] = bf16(wte[token] + wpe[t+2] + emb_add[row]) (GPT2Model_XX.forward, :941-951; positions
 * start at 1 behind the memory slot).  wte bf16 [>= vocab, C], wpe / emb_add fp32. */
int vdb_sample_tokens(const float* logits, long long ldl, int V, int n, const float* temperature, const int* step,
                      const unsigned long long* seed, const float* uniforms, int ldu, const int* forced, int eos, int max_len,
                      int* tokens, int ldt, const void* wte, const float* wpe, const float* emb_add, long long ld_emb, int C,
                      void* x_next, long long ldx, void* stream);
/* x[row] = bf16(wte[tokens[row, t]] + wpe[t + pos_offset] + emb_add[row]), t = *step (0 when step == NULL): the <BOS> input. */
int vdb_token_embed(const int* tokens, int ldt, const int* step, int pos_offset, const void* wte, const float* wpe,
                    const float* emb_add, long long ld_emb, int n, int C, void* x, long long ldx, void* stream);

/* ---- Optimus BERT text encode — optimus_vae_next.encode (lib/model_zoo/optimus.py:729-743) on BertForLatentConnector_XX
 *      (optimus_models/optimus_bert.py:1349-1439).  The 12 post-LN layers run on vdb_gemm_bf16 / vdb_attention_keylen_bf16 /
 *      vdb_layernorm, the pooler on the VDB_ACT_TANH epilogue. ---------------------------------------------------------- */
/* BertEmbeddings.forward (optimus_bert.py:144-175) with positions 0.. and token type 0: for ids int32 [n, L] (row-major),
 * y[b*L + j] = bf16(LayerNorm(word_emb[ids[b, j]] + pos_emb[j] + type_emb[0]) * gamma + beta), fp32 throughout, the fp32
 * tables read in place.  C % 128 == 0, C <= 1024, L <= max_pos; ids outside [0, vocab) are clamped. */
int vdb_bert_embed_ln(const int* ids, int n, int L, const float* word_emb, int vocab, const float* pos_emb, int max_pos,
                      const float* type_emb, const float* gamma, const float* beta, float eps, int C, void* y, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VDB200_H_ */
