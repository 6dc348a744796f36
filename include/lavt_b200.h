/* lavt_b200.h -- C ABI of the B200-native (sm_100a) LAVT-RS hot path.
 *
 * The reference (Yxxxb/LAVT-RS) has no FFI layer: its hot path is Python modules calling PyTorch ops.
 * Each entry point below replaces the PyTorch op sequence of one reference function (cited per
 * function as file:line relative to the reference root).  The Python host in lavt_rs_b200/lib/ binds
 * them with ctypes (lavt_rs_b200/_cabi.py) and keeps the reference's module / state-dict API.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless stated otherwise; `stream` is a cudaStream_t passed as void*
 *   - activations: channels-last, tokens x C row-major; "bf16" = __nv_bfloat16, residual stream = fp32
 *   - weights: nn.Linear layout [out, in] (K-major), bf16
 *   - return value: 0 = ok, non-zero = error (LAVT_ERR_*); lavt_last_error() gives the message.
 *     There is NO CPU fallback: unsupported shapes / non-sm_100 devices are errors.
 */
#ifndef LAVT_B200_H_
#define LAVT_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LAVT_ABI_VERSION 4

#define LAVT_ERR_SHAPE 1
#define LAVT_ERR_CUDA 2
#define LAVT_ERR_ARCH 3

enum { LAVT_ACT_NONE = 0, LAVT_ACT_GELU = 1, LAVT_ACT_RELU = 2, LAVT_ACT_TANH = 3, LAVT_ACT_SIGMOID = 4 };

/* Window geometry of one Swin block on a (B,D,H,W,C) channels-last tensor.
 * (wd,wh,ww)/(sd,sh,sw) are the EFFECTIVE window/shift after get_window_size clamping
 * (lib/video_swin_transformer.py:70-83); (Wd,Wh,Ww) is the configured window that sizes the
 * relative_position_bias_table (:107-127). nw* = ceil(dim / w*). N = wd*wh*ww. */
typedef struct lavt_win_geom {
  int32_t B, D, H, W;
  int32_t wd, wh, ww;
  int32_t sd, sh, sw;
  int32_t nwd, nwh, nww;
  int32_t N;
  int32_t Wd, Wh, Ww;
} lavt_win_geom_t;

/* Fused GEMM epilogue:
 *   pre = acc[m,n] * cscale[n] + bias[n]
 *   out[orow(m), n] = act(pre) * mul'[m,n] * rscale[orow(m) / rscale_rows] + resid[orow(m), n],   out_pre[orow(m), n] = pre
 * mul' = mul, or GELU'(mul) with mul_act = LAVT_ACT_GELU: the fc2 input gradient times the derivative of the saved fc1
 * pre-activation in one launch (adjoint of Mlp, lib/video_swin_transformer.py:30-36); out_pre keeps the pre-activation of a
 * training-mode forward next to the activated output (fc1: both tensors from one launch).
 * orow = m, or (win != NULL) the token row that window-row m maps back to (window_reverse +
 * reverse cyclic shift + crop, lib/video_swin_transformer.py:238-247); pad rows are dropped. */
typedef struct lavt_epilogue {
  const float* cscale;   /* [N] or NULL */
  const float* bias;     /* [N] or NULL */
  int32_t act;           /* LAVT_ACT_* */
  int32_t ldm;           /* row pitch of mul (elements) */
  const void* mul;       /* bf16 [M, ldm] or NULL */
  const float* resid;    /* fp32 [rows_out, ldo] or NULL */
  float* out_f32;        /* fp32 [rows_out, ldo] or NULL */
  void* out_bf16;        /* bf16 [rows_out, ldo] or NULL */
  int32_t ldo;           /* row pitch of resid / out / out_pre (elements) */
  int32_t mul_act;       /* 0: multiply by mul; LAVT_ACT_GELU: multiply by GELU'(mul) */
  const lavt_win_geom_t* win; /* HOST pointer or NULL */
  const float* rscale;   /* fp32 per-sample scale of the whole branch, or NULL: DropPath in training (timm drop_path as used at
                            lib/video_swin_transformer.py:266,271: 0 or 1/keep_prob per clip); sample = output row / rscale_rows */
  int32_t rscale_rows;
  int32_t pre_mode;      /* 0: out_pre = pre;  1 (act = LAVT_ACT_GELU only): out_pre = GELU'(pre), the factor the backward of fc1 needs */
  void* out_pre;         /* bf16 [rows_out, ldo] or NULL: the value BEFORE the activation (tcgen05 GEMM / conv entry points only) */
} lavt_epilogue_t;

const char* lavt_last_error(void);
int lavt_abi_version(void);
/* 0 if the current device is sm_100 (B200), LAVT_ERR_ARCH otherwise. */
int lavt_check_device(void);

/* C[M,N] = A[M,K] (bf16, pitch lda) x Wt[N,K]^T (bf16, pitch ldw), fp32 accumulate on tcgen05 tensor
 * cores, fused epilogue.  Replaces nn.Linear / Conv1d(k=1) call sites:
 *   qkv / proj  lib/video_swin_transformer.py:144,166 (lib/backbone.py:125,139)
 *   fc1 / fc2   :30-36          PatchMerging.reduction :309     PatchEmbed3D.proj :627
 *   PWAM vis_project / f_query / W / project_mm :900-973        LanguageGate res_gate :519-525
 * Requires N % 32 == 0, K % 8 == 0 (tile remainders are handled by TMA zero fill and a column guard in the epilogue). */
int lavt_gemm_bf16(const void* A, int64_t lda, const void* Wt, int64_t ldw, int32_t M, int32_t N, int32_t K,
                   const lavt_epilogue_t* epi, void* stream);

/* 3x3 / pad 1 / stride 1 convolution as an implicit GEMM over NHWC bf16 input (pixel pitch ldx >= Cin):
 *   out[pix, co] = epilogue( sum_{ky,kx,ci} x[img, h+ky-1, w+kx-1, ci] * Wt[co, (ky*3+kx)*Cin + ci] )
 * Replaces conv{1,2}_{4,3,2} + BatchNorm2d(eval, folded into cscale/bias) + ReLU of
 * SimpleDecoding.forward, lib/mask_predictor.py:56-87.  Requires Cin % 8 == 0, Cout % 32 == 0. */
int lavt_conv3x3_bf16(const void* x_nhwc, int64_t ldx, int32_t n_img, int32_t H, int32_t W, int32_t Cin,
                      const void* Wt, int32_t Cout, const lavt_epilogue_t* epi, void* stream);

/* 3x3x3 / pad 1 / stride 1 Conv3d as an implicit GEMM over NDHWC bf16 input (position pitch ldx >= Cin), 5-D TMA boxes:
 *   out[pos, co] = epilogue( sum_{kz,ky,kx,ci} x[clip, d+kz-1, h+ky-1, w+kx-1, ci] * Wt[co, ((kz*3+ky)*3+kx)*Cin + ci] )
 * Replaces the Conv3d(3,3,3) layers of SepTPWAM (temporal_vis_project / f_query_t / W_t / project_mm_t,
 * lib/video_swin_transformer.py:1334-1336, 1376-1379, 1435-1438, 1459-1461) under the README video flags
 * (--sep_t_pwam --conv3d_kernel_size_t 3-3-3 ...).  Requires Cin % 8 == 0, Cout % 32 == 0. */
int lavt_conv3d_bf16(const void* x_ndhwc, int64_t ldx, int32_t n_clip, int32_t D, int32_t H, int32_t W, int32_t Cin,
                     const void* Wt, int32_t Cout, const lavt_epilogue_t* epi, void* stream);

/* ---- LayerNorm fused with the gathers that feed the GEMMs (fp32 rows in, bf16 and/or fp32 rows out) ---- */

/* out[m,:] = LN(x[m,:]) * gamma + beta over C channels.  norm2 before the MLP (lib/video_swin_transformer.py:250),
 * patch_embed.norm (:630), per-stage output norm{i} (:871).  C % 4 == 0, C <= 3072. out_bf16 / out_f32 may be NULL (not both). */
int lavt_layernorm_rows(const float* x, int64_t ldx, int64_t M, int32_t C, const float* gamma, const float* beta,
                        float eps, void* out_bf16, float* out_f32, void* stream);

/* LN1 + zero pad + cyclic shift + window_partition as one gather (lib/video_swin_transformer.py:218-234):
 * out[(b*nW + w)*N + t, :] = LN(x[token(w,t)]) or 0 for a pad row.  x is (B,D,H,W,C) fp32. */
int lavt_layernorm_window_gather(const float* x, int32_t C, const lavt_win_geom_t* geom, const float* gamma,
                                 const float* beta, float eps, void* out_bf16, void* stream);

/* PatchMerging gather + LN(4C) (lib/video_swin_transformer.py:298-308): (B,D,H,W,C) fp32 ->
 * (B,D,ceil(H/2),ceil(W/2),4C) bf16, channel blocks ordered (0,0),(1,0),(0,1),(1,1); odd H/W zero padded. */
int lavt_patch_merge_layernorm(const float* x, int32_t B, int32_t D, int32_t H, int32_t W, int32_t C,
                               const float* gamma, const float* beta, float eps, void* out_bf16, void* stream);

/* PatchEmbed3D im2col (lib/video_swin_transformer.py:616-628): pixels x[b,c,t,h,w] fp32 addressed through element
 * strides (stride_b, stride_c, stride_t; rows of W contiguous floats), so both the backbone's (B,3,T,H,W) input and
 * LAVTVideo's un-permuted (B,T,3,H,W) input (lib/_utils.py:97) are read in place ->
 * (B*T*ceil(H/4)*ceil(W/4), 64) bf16 rows, column = c*16 + ph*4 + pw, columns 48..63 zero (GEMM K = 64). */
int lavt_patch_embed_im2col(const float* x, int64_t stride_b, int64_t stride_c, int64_t stride_t, int32_t B, int32_t T,
                            int32_t H, int32_t W, void* out_bf16, void* stream);

/* ---- window attention core (lib/video_swin_transformer.py:147-165) ----
 * qkv: bf16 [B*nW*N, 3C] in window order, q already scaled by head_dim^-0.5 * log2(e) (the softmax is evaluated in
 * base 2; fold the factor into the qkv GEMM epilogue via cscale); table_t: fp32 [nH, L] = the module's
 * relative_position_bias_table [L, nH] transposed; out: bf16 [B*nW*N, C].  head_dim must be 32. */
int lavt_window_attention(const void* qkv, const float* table_t, int32_t L, int32_t nH, const lavt_win_geom_t* geom,
                          void* out_bf16, void* stream);
/* Same, and lse fp32 [B*nW*N, nH] = log2-sum-exp2 of every score row (what the backward needs besides qkv and out; written by the
 * tcgen05 kernels only, i.e. for windows of 16 tokens or more -- lavt_window_attention_has_lse tells whether this geometry gets it: 1 / 0). */
int lavt_window_attention_lse(const void* qkv, const float* table_t, int32_t L, int32_t nH, const lavt_win_geom_t* geom, void* out_bf16,
                              float* lse, void* stream);
int lavt_window_attention_has_lse(const lavt_win_geom_t* geom, int32_t L, int32_t nH);
/* Kernel selection for lavt_window_attention (process-wide; initial value from the LAVT_ATTN_IMPL environment variable, "tc2" / "tc3"):
 *   0 = auto: attn_tc3.cu (row-parallel tcgen05 / TMEM kernel) for windows whose (h, w) extent is the full 7 x 7 or 12 x 12, the
 *       key-chunked one-pass tcgen05 kernel (attn_tc2.cu) for every other window of 16 ... 1152 tokens, the mma.sync kernel
 *       (attn_window.cu) for windows of fewer than 16 tokens
 *   3 = attn_tc2.cu wherever it applies (A/B runs), else as auto
 *   4 = same as auto (attn_tc3.cu where it applies)
 * Any other value, including the retired 1 (mma.sync only) and 2 (round-1 tcgen05 kernel), means auto.  Returns the previous setting. */
int lavt_set_attention_impl(int32_t impl);

/* ---- PWAM (lib/video_swin_transformer.py:919-1009) ---- */
/* InstanceNorm1d statistics over the n tokens of each clip: x fp32 [B,n,C] -> stats fp32 [B,2,C] = (mean, rstd).
 * (the pre-norm projections q_pre / lang_pre are kept in fp32: they are never tensor-core operands) */
int64_t lavt_instnorm_workspace_floats(int32_t B, int64_t n, int32_t C);
int lavt_instnorm_stats(const float* x, int32_t B, int64_t n, int32_t C, float eps, float* stats,
                        float* workspace, void* stream);
/* k, v = (W l + b) * l_mask : l fp32 [B,Lin,Nl], mask fp32 [B,Nl], weights fp32 [C,Lin] -> k, v fp32 [B,Nl,C] */
int lavt_pwam_kv(const float* l, const float* mask, const float* wk, const float* bk, const float* wv, const float* bv,
                 float* k, float* v, int32_t B, int32_t Nl, int32_t Lin, int32_t C, void* stream);
/* LangProject of the --fuse simple ablation (lib/video_swin_transformer.py:1012-1039): per clip, masked mean of the word features ->
 * Linear(Lin -> C) -> ReLU -> Linear(C -> C).  l fp32 [B,Lin,Nl], mask fp32 [B,Nl], w0 [C,Lin], w2 [C,C].  The sentence vector is
 * written as stats fp32 [B,2,C] = (-lang, 1): lavt_pwam_mul_norm over an all-zero lang tensor then yields vis * lang. */
int lavt_lang_project(const float* l, const float* mask, const float* w0, const float* b0, const float* w2, const float* b2, float* stats,
                      int32_t B, int32_t Nl, int32_t Lin, int32_t C, void* stream);
/* o = softmax_words(C^-0.5 * IN(q_pre) k^T + (1e4 mask - 1e4)) v ; q_pre fp32, o bf16 [B,n,C] */
int lavt_pwam_attend(const float* qpre, const float* stats, const float* k, const float* v, const float* mask,
                     void* o_bf16, int32_t B, int64_t n, int32_t C, int32_t Nl, int32_t heads, void* stream);
/* out = vis * IN(lang_pre) (vis, out bf16; lang_pre fp32 [B,n,C]) -- the A operand of project_mm */
int lavt_pwam_mul_norm(const void* vis_bf16, const float* lang, const float* stats, void* out_bf16, int32_t B,
                       int64_t n, int32_t C, void* stream);

/* out = InstanceNorm(a) + InstanceNorm(b) with precomputed statistics (fp32 [B,n,C]; out may alias a): SepTPWAM sums its
 * temporal and spatial branches after their InstanceNorm3d (lib/video_swin_transformer.py:1513-1524, 1556-1561) */
int lavt_instnorm_sum2(const float* a, const float* stats_a, const float* b, const float* stats_b, float* out, int32_t B,
                       int64_t n, int32_t C, void* stream);

/* ---- text side: BertModel(text, attention_mask)[0] (lib/_utils.py:52-54, 98-100; bert/modeling_bert.py = HF v3.0.2) ----
 * The dense layers are lavt_gemm_bf16 calls and the LayerNorms lavt_layernorm_rows (eps 1e-12); these are the rest. */
/* BertEmbeddings: out[b*Nl+t, :] = word[ids[b,t]] + pos[t] + type0  (fp32 rows; the embedding LayerNorm follows) */
int lavt_bert_embed(const int64_t* ids, const float* word, const float* pos, const float* type0, float* out, int32_t B, int32_t Nl,
                    int32_t H, int32_t vocab, void* stream);
/* BertSelfAttention core per (sentence, head), head_dim 64, Nl <= 128: softmax(q k^T + (1 - mask) * -10000) v.
 * qkv bf16 [B*Nl, 3H] = q | k | v with q pre-scaled by 64^-0.5 * log2(e); mask fp32 [B, Nl]; out bf16 [B*Nl, H] */
int lavt_bert_attention(const void* qkv_bf16, const float* mask, void* out_bf16, int32_t B, int32_t Nl, int32_t H, int32_t heads,
                        void* stream);
/* Split-precision operand of the text encoder's GEMMs: x fp32 [M,K] (pitch ldx) -> out bf16 [M,3K] = hi | lo | hi with hi = bf16(x),
 * lo = bf16(x - hi).  Against weights stored [W_hi | W_hi | W_lo] one lavt_gemm_bf16 launch accumulates hi W_hi + lo W_hi + hi W_lo in
 * fp32 on the tensor cores (relative error ~1e-5): BERT's 12 layers no longer dominate the logit error of the whole model. */
int lavt_split3_bf16(const float* x, int64_t ldx, void* out_bf16, int64_t M, int32_t K, void* stream);
/* lavt_bert_attention with fp32 qkv [B*Nl, 3H] / out [B*Nl, H] (same pre-scaled q convention) */
int lavt_bert_attention_f32(const float* qkv, const float* mask, float* out, int32_t B, int32_t Nl, int32_t H, int32_t heads, void* stream);
/* (B, Nl, C) fp32 -> (B, C, Nl) fp32: l_feats = last_hidden_state.permute(0, 2, 1) (lib/_utils.py:54) */
int lavt_rows_to_channels_first(const float* in, float* out, int32_t B, int32_t Nl, int32_t C, void* stream);

/* ---- fp32 validation twins (csrc/fp32_ref_kernels.cu) ----
 * north_star tolerance: "1e-4 in fp32 with fp32 accumulate".  The production contractions take bf16 operands; these twins take fp32
 * operands, accumulate in fp32 on the CUDA cores and share the production epilogue (lavt_epilogue_t, incl. the window-reverse scatter)
 * and index math, so a Swin block replays at fp32 accuracy on the device (lavt_rs_b200.engine.set_precision("fp32")).  Validation only:
 * slow, never selected by default.
 * lavt_gemm_f32_ref: out = epilogue(A[M,K] Wt[N,K]^T), any M / N / K.
 * lavt_window_attention_f32_ref: qkv fp32 [rows, 3C] (q pre-scaled by 32^-0.5 * log2 e, as in the bf16 path) -> out fp32 [rows, C].
 * lavt_layernorm_window_gather_f32: lavt_layernorm_window_gather with an fp32 result. */
int lavt_gemm_f32_ref(const float* A, int64_t lda, const float* Wt, int64_t ldw, int32_t M, int32_t N, int32_t K, const lavt_epilogue_t* epi,
                      void* stream);
int lavt_window_attention_f32_ref(const float* qkv, const float* table_t, int32_t L, int32_t nH, const lavt_win_geom_t* geom, float* out,
                                  void* stream);
int lavt_layernorm_window_gather_f32(const float* x, int32_t C, const lavt_win_geom_t* geom, const float* gamma, const float* beta, float eps,
                                     float* out_f32, void* stream);

/* ---- VLT fuse-and-classify head (lib/vlt.py:12-485; models vlt / lavt_vlt, lib/segmentation.py:299-433) ----
 * The head's convolutions and Linear / Conv1d layers run on lavt_gemm_bf16 / lavt_conv3x3_bf16 (eval BatchNorm folded into the
 * epilogue); these are the memory-bound pieces between them.
 * lavt_rows_affine_act: out[r, c] = act((x[r, c] + add[r, c]) * v[r / rows_per_image, c] * s[c] + t[c]); add (bf16) / v / s / t may be NULL.
 *   x bf16 or fp32 rows (pitch ldx), out bf16 and / or fp32 (pitch ldo).  x_c4 + vis_reduce_chann_1(x_c4), times the sentence vector,
 *   joint_threshold BatchNorm + ReLU in one pass (:140-145), and the ReLU after lang_proj (:101-104).
 * lavt_avgpool2_nhwc: nn.AvgPool2d(2) (:61, :151) over NHWC bf16 (pixel pitches ldi / ldo), even H and W.
 * lavt_append_coords: vlt_concat_coords (:267-292): out NHWC bf16 [n,H,W,C+8] = in | x x x y y y 0 0 with x, y in [-1, 1].
 * lavt_rows_add_table: out[r, :] = x[r, :] + table[r % period, :] -- PositionalEncoding (:204-222) on batch-major rows.
 * lavt_mha_small: the attention core of nn.MultiheadAttention with head_dim 32 (:256, :262, :351): out[b, i, h*32:] =
 *   softmax_j(q[b,i,h] . k[b,j,h] / sqrt(32) + (key_mask[b,j] == 0 ? -inf : 0)) v[b,j,h]; q [B,Lq] rows of pitch ldq etc., S <= 1024 keys.
 * lavt_gate_transpose: out NHWC bf16 [B,S,Q] = gate[b*Q+q] * x[b*Q+q, s] -- gates * y of QueryBalancingModule (:405) and the
 *   permute/view of q_to_spatial's output (:180-182) in one pass. */
int lavt_rows_affine_act(const void* x, int32_t x_is_bf16, int64_t ldx, const void* add_bf16, int64_t lda, const float* v, int64_t rows_per_image,
                         const float* s, const float* t, int32_t act, void* out_bf16, float* out_f32, int64_t ldo, int64_t rows, int32_t C,
                         void* stream);
int lavt_avgpool2_nhwc(const void* in_bf16, int64_t ldi, void* out_bf16, int64_t ldo, int32_t n_img, int32_t H, int32_t W, int32_t C, void* stream);
int lavt_append_coords(const void* in_bf16, int64_t ldi, void* out_bf16, int32_t n_img, int32_t H, int32_t W, int32_t C, void* stream);
int lavt_rows_add_table(const void* x, int32_t x_is_bf16, int64_t ldx, const float* table, int64_t period, void* out_bf16, float* out_f32,
                        int64_t ldo, int64_t rows, int32_t C, void* stream);
int lavt_mha_small(const void* q_bf16, int64_t ldq, const void* k_bf16, int64_t ldk, const void* v_bf16, int64_t ldv, const float* key_mask,
                   void* out_bf16, int64_t ldo, int32_t B, int32_t Lq, int32_t S, int32_t heads, void* stream);
int lavt_gate_transpose(const float* x, int64_t ldx, const float* gate, int64_t ldg, void* out_bf16, int32_t B, int32_t Q, int32_t S, void* stream);

/* ---- decoder glue (lib/mask_predictor.py:56-99, lib/_utils.py:106) ---- */
/* out NHWC bf16 [n,H,W,C1+C2] = cat[bilinear(prev [n,ph,pw,C1] -> HxW, align_corners=True), skip [n,H,W,C2]];
 * C2 = 0 (skip NULL) is a plain upsample: nn.Upsample(scale_factor=2, bilinear, align_corners=True) of lib/vlt.py:48,75,437-452 */
int lavt_upsample_concat(const void* prev_bf16, int32_t ph, int32_t pw, int32_t C1, const void* skip_bf16, int32_t C2,
                         void* out_bf16, int32_t n_img, int32_t H, int32_t W, void* stream);
/* conv3x3 + folded BN + ReLU of cat[bilinear(Y [n,h,w,C_Y] -> HxW, align_corners=True), skip], evaluated on the coarse grid:
 * out bf16 [n,H,W,hid] = ReLU(addend + s[co] * sum_tap sum_corner beta * Z[n, corner, tap*hid + co]), Z bf16 [n,h,w,9*hid] = Y . W_tap
 * (row tap*hid + co of the weight holds w[co, :C_Y, ky, kx], tap = ky*3+kx; zero padding on the fine grid).  addend = P fp32 [n,H,W,hid]
 * (the skip half of the conv with the BN folded in) or, with P NULL, b fp32 [hid]. */
int lavt_upconv_blend(const void* z_bf16, int32_t h, int32_t w, int32_t hid, const float* P, const float* s, const float* b, void* out_bf16,
                      int32_t n_img, int32_t H, int32_t W, void* stream);
/* conv1_1: logits[pix, 0:2] = y[pix, :] . w[0:2, :] + b */
int lavt_conv1x1_logits(const void* y_bf16, const float* w, const float* b, float* out, int64_t npix, int32_t C, void* stream);
/* (n,h,w,2) fp32 -> (n,2,H,W) fp32 NCHW, bilinear align_corners=True */
int lavt_upsample_logits(const float* in, float* out, int32_t n_img, int32_t h, int32_t w, int32_t H, int32_t W, void* stream);
/* layout converters for the NCHW tensors of the reference's backbone / classifier API */
int lavt_nhwc_to_nchw(const float* in, float* out, int32_t n_img, int32_t P, int32_t C, void* stream);
int lavt_nchw_to_nhwc_bf16(const float* in, void* out_bf16, int32_t n_img, int32_t P, int32_t C, void* stream);

/* ================================================================================================
 * Backward pass (training step, BASELINE config 4).  The reference differentiates its forward with autograd
 * (train.py:330-360: loss.backward()); these are the adjoints of the forward entry points above.  Conventions: the
 * gradient on the residual stream is fp32 [tokens, C]; gradients that feed a GEMM are bf16 rows; parameter gradients
 * are fp32 and ACCUMULATED (+=) so that the caller zeroes them once per step (optimizer.zero_grad(), train.py:352).
 * ================================================================================================ */

/* dst[M, ldd] (+)= A[M,K] x Bt[N,K]^T with the K axis split over work items (weight gradients: dW = dY^T X has few output
 * tiles and K = all tokens).  A = dY^T [out, tokens], Bt = X^T [in, tokens] (lavt_transpose_bf16).  b_koff (a multiple of 8)
 * shifts the K coordinate of Bt (taps of a convolution weight gradient over a zero-padded pixel axis).  Adjoint of every nn.Linear /
 * Conv1d(k=1) / Conv2d weight on the path w.r.t. its weight. */
int64_t lavt_gemm_splitk_workspace_floats(int32_t M, int32_t N, int32_t K);
int lavt_gemm_bf16_splitk(const void* A, int64_t lda, const void* Bt, int64_t ldb, int32_t M, int32_t N, int32_t K, int32_t b_koff,
                          float* workspace, int64_t workspace_floats, float* dst, int64_t ldd, int32_t accumulate, void* stream);
/* Small-M forward GEMM (the text encoder's dense layers, bert/modeling_bert.py: 160 rows at 8 clips x 20 tokens): the same product as
 * lavt_gemm_bf16 computed as a split-K launch that fills the GPU (work item = (tile, k range), fp32 partials in ``workspace``, size from
 * lavt_gemm_splitk_workspace_floats) followed by one reduce + epilogue kernel (column scale, bias, GELU, fp32 residual; bf16 and / or fp32 out).
 * Identity row map only. */
int lavt_gemm_bf16_smallm(const void* A, int64_t lda, const void* Wt, int64_t ldw, int32_t M, int32_t N, int32_t K,
                          const lavt_epilogue_t* epi, float* workspace, int64_t workspace_floats, void* stream);

/* dst[n_out, n_in] (+)= dy[tokens, n_out]^T x[tokens, n_in] straight from the ROW-MAJOR activations: TMA boxes of 64 tokens x 64
 * channels land in shared memory as MN-major tcgen05 operands, so no transposed copies are made (split-K over the token axis,
 * workspace as for lavt_gemm_bf16_splitk with M = n_out, N = n_in, K = tokens).  n_out % 8 == 0, n_in % 32 == 0. */
int lavt_gemm_bf16_wgrad(const void* dy, int64_t lddy, const void* x, int64_t ldx, int64_t tokens, int32_t n_out, int32_t n_in,
                         float* workspace, int64_t workspace_floats, float* dst, int64_t ldd, int32_t accumulate, void* stream);
/* conv3x3 (pad 1, stride 1) WEIGHT gradient in one launch, no im2col and no padded / transposed copies:
 *   dw_taps[co, (ky*3+kx)*Cin + ci] (+)= sum_{img,h,w} dz[img,h,w,co] * x[img,h+ky-1,w+kx-1,ci]
 * dz, x: NHWC bf16 (contiguous).  Both operands are 4-D TMA boxes of 64 channels x (TH x TW = 64 pixels) that land in shared memory as
 * MN-major tcgen05 operands; the tap is a coordinate offset of the x box and the zero padding is TMA's out-of-bounds fill.  Split-K
 * over the pixel tiles.  Cin % 64 == 0.  Adjoint of lavt_conv3x3_bf16 w.r.t. its weights (lib/mask_predictor.py:56-87). */
int64_t lavt_conv3x3_wgrad_workspace_floats(int32_t n_img, int32_t H, int32_t W, int32_t Cin, int32_t Cout);
int lavt_conv3x3_wgrad(const void* dz_nhwc, const void* x_nhwc, int32_t n_img, int32_t H, int32_t W, int32_t Cin, int32_t Cout,
                       float* workspace, int64_t workspace_floats, float* dw_taps, int32_t accumulate, void* stream);
/* the same for Conv3d(3,3,3): dw_taps[co, ((kz*3+ky)*3+kx)*Cin + ci] over NDHWC operands, 5-D TMA boxes (SepTPWAM, adjoint of lavt_conv3d_bf16) */
int64_t lavt_conv3d_wgrad_workspace_floats(int32_t n_clip, int32_t D, int32_t H, int32_t W, int32_t Cin, int32_t Cout);
int lavt_conv3d_wgrad(const void* dz_ndhwc, const void* x_ndhwc, int32_t n_clip, int32_t D, int32_t H, int32_t W, int32_t Cin, int32_t Cout,
                      float* workspace, int64_t workspace_floats, float* dw_taps, int32_t accumulate, void* stream);
/* out[N, M] (pitch ldo) = in[M, N]^T (pitch ldi), bf16 */
int lavt_transpose_bf16(const void* in, int64_t ldi, void* out, int64_t ldo, int64_t M, int32_t N, void* stream);
/* dst[n] += sum_m x[m, n]  (bias gradients); x is bf16 (is_bf16 != 0) or fp32 */
int lavt_colsum_accumulate(const void* x, int32_t is_bf16, int64_t ldx, int64_t M, int32_t N, float* dst, void* stream);
/* out bf16 [M, C] = x[src(m)]: src = m, or (geom != NULL) the token of window row m, pad rows -> 0.  Adjoint of the proj
 * epilogue's window_reverse + un-shift + crop scatter (lib/video_swin_transformer.py:238-247). */
int lavt_cast_rows_bf16(const float* x, int64_t ldx, int64_t M, int32_t C, const lavt_win_geom_t* geom, void* out_bf16, void* stream);
/* same with a per-sample scale: out = x[src(m)] * rscale[src(m) / rscale_rows] (adjoint of the epilogue's rscale: DropPath backward) */
int lavt_cast_rows_scaled_bf16(const float* x, int64_t ldx, int64_t M, int32_t C, const lavt_win_geom_t* geom, const float* rscale,
                               int32_t rscale_rows, void* out_bf16, void* stream);
/* The same cast with the column sums of the (scaled, fp32) values added into colsum[C] (+=): the bias gradient of the Linear layer whose
 * output gradient the rows are (Mlp.fc2 / WindowAttention3D.proj of a Swin block under autograd) without a second pass; C <= 1024. */
int lavt_cast_rows_colsum_bf16(const float* x, int64_t ldx, int64_t M, int32_t C, const lavt_win_geom_t* geom, const float* rscale,
                               int32_t rscale_rows, void* out_bf16, float* colsum, void* stream);
/* exact-erf GELU on a saved bf16 pre-activation and its derivative (Mlp.act, lib/video_swin_transformer.py:33) */
/* Adjoint of lavt_lang_project (--fuse simple in training mode; reference lib/video_swin_transformer.py:1012-1039 under autograd):
 * ds fp32 [B,C] = gradient of the sentence vector (sum over the pixels of d a2 * vis: row 0 of lavt_pwam_mul_norm_bwd's reductions);
 * dw0 [C,Lin], db0 [C], dw2 [C,C], db2 [C] and dl [B,Lin,Nl] accumulate (+=; any may be NULL except the workspace of
 * B * (2 C + 2 Lin) floats). */
int lavt_lang_project_bwd(const float* l, const float* mask, const float* w0, const float* b0, const float* w2, const float* ds, float* dw0,
                          float* db0, float* dw2, float* db2, float* dl, float* workspace, int32_t B, int32_t Nl, int32_t Lin, int32_t C, void* stream);
int lavt_gelu_fwd(const void* x_bf16, void* y_bf16, int64_t count, void* stream);
int lavt_gelu_bwd(const void* dy_bf16, const void* x_bf16, void* dx_bf16, int64_t count, void* stream);
/* LayerNorm backward, adjoints of lavt_layernorm_rows / _window_gather / lavt_patch_merge_layernorm:
 * dx[token] = dres[token] + LN'(dy[row]) (dres may be NULL or alias dx); dgamma / dbeta accumulate. */
int lavt_layernorm_rows_bwd(const float* x, int64_t ldx, int64_t M, int32_t C, const void* dy_bf16, int64_t lddy, const float* gamma, float eps,
                            const float* dres, float* dx, float* dgamma, float* dbeta, void* stream);
int lavt_layernorm_window_gather_bwd(const float* x, int32_t C, const lavt_win_geom_t* geom, const void* dy_bf16, const float* gamma,
                                     float eps, const float* dres, float* dx, float* dgamma, float* dbeta, void* stream);
int lavt_patch_merge_layernorm_bwd(const float* x, int32_t B, int32_t D, int32_t H, int32_t W, int32_t C, const void* dy_bf16,
                                   const float* gamma, float eps, float* dx, float* dgamma, float* dbeta, void* stream);
/* Adjoint of lavt_window_attention: qkv / out as saved by the forward, dout = gradient of out; dqkv bf16 [rows, 3C] = gradient
 * of the UNSCALED qkv projection; dtable_t fp32 [nH, L] accumulates the relative_position_bias_table gradient (transposed), or NULL.
 * lse: the row statistics saved by lavt_window_attention_lse, or NULL (then they are recomputed in a first pass; mma.sync kernel only).
 * Windows of any size up to 8 x 12 x 12 = 1152 tokens; lavt_window_attention_bwd_kernel tells which kernel a geometry gets.
 * workspace: fp32 scratch of at least lavt_window_attention_bwd_workspace_floats(geom, L, nH) floats, owned by the caller and
 * not read across calls (NULL / 0 where that query returns 0).  Nothing is allocated inside the call. */
int lavt_window_attention_bwd(const void* qkv, const void* out, const void* dout, const float* table_t, int32_t L, int32_t nH,
                              const lavt_win_geom_t* geom, const float* lse, void* dqkv, float* dtable_t, float* workspace,
                              int64_t workspace_floats, void* stream);
/* fp32 workspace lavt_window_attention_bwd needs for this geometry when lse is given: 0 except on attn_bwd_tc2.cu for windows of more
 * than 128 tokens (one [N rounded up to 128, 32] dQ scratch per CTA of the persistent grid) */
int64_t lavt_window_attention_bwd_workspace_floats(const lavt_win_geom_t* geom, int32_t L, int32_t nH);
/* The kernel lavt_window_attention_bwd runs for this geometry under the current selection (host arithmetic, no device call):
 * 1 = mma.sync (attn_bwd.cu), 2 = attn_bwd_tc.cu, 3 = attn_bwd_tc2.cu, 0 = none (the call fails with LAVT_ERR_SHAPE). */
int lavt_window_attention_bwd_kernel(const lavt_win_geom_t* geom, int32_t L, int32_t nH, int32_t has_lse);
/* Kernel selection for lavt_window_attention_bwd (process-wide; initial value from LAVT_ATTN_BWD_IMPL = mma | tc | tc2):
 *   0 = auto: attn_bwd_tc.cu (tcgen05 / TMEM) for 7 x 7 windows with an even number of frames when lse is given, else the mma.sync
 *       kernel (attn_bwd.cu) where Q / K / V / dO and the table fit its shared memory, else attn_bwd_tc2.cu (tcgen05 / TMEM, key tiles
 *       outer, any window of 16 ... 1152 tokens with lse: the full and large clamped 8 x 12 x 12 windows)
 *   1 = mma.sync kernel only      2 = same as auto
 *   3 = attn_bwd_tc2.cu wherever it applies (A/B runs and tests), else as auto
 * Any other value means auto.  Returns the previous setting. */
int lavt_set_attention_bwd_impl(int32_t impl);

/* ---- PWAM + LanguageGate backward (adjoints of lavt_pwam_* above; reference lib/video_swin_transformer.py:919-1009, 519-525) ---- */
/* Per pixel: recompute q^ = IN(q_pre) and the masked word softmax P, dP = dO v^T, dS = P (dP - sum P dP).  Outputs:
 * dqhat fp32 [B,n,C] = C^-0.5 dS k; qs bf16 [B*n, C] = C^-0.5 q^; p_bd / ds_bd bf16 [B*n, B*heads*NlPad]: row (b, pixel) carries
 * P / dS of fusion head h in columns (b*heads + h)*NlPad + j and zeros elsewhere, so that dv = p_bd^T dO and dk = ds_bd^T qs
 * are ordinary weight-gradient GEMMs (lavt_gemm_bf16_splitk); sums fp32 [B,2,C] += (sum_n dqhat, sum_n dqhat * q^). */
int lavt_pwam_attend_bwd(const float* qpre, const float* stats, const float* k, const float* v, const float* mask, const void* do_bf16,
                         float* dqhat, void* qs_bf16, void* p_bd, void* ds_bd, float* sums, int32_t B, int64_t n, int32_t C, int32_t Nl,
                         int32_t NlPad, int32_t heads, void* stream);
/* a2 = vis * IN(lang_pre), vis = GELU(vis_pre): dvispre bf16 = da2 * IN(lang_pre) * GELU'(vis_pre); sums [B,2,C] += the
 * InstanceNorm reductions of g = da2 * vis (sum g, sum g * lang) */
int lavt_pwam_mul_norm_bwd(const void* da2, const void* vis, const void* vispre, const float* langpre, const float* stats, void* dvispre,
                           float* sums, int32_t B, int64_t n, int32_t C, void* stream);
/* InstanceNorm backward from the reductions: out bf16 = rstd * (g - S1/n - x^ S2/n); g = g_f32, or ga * gb (bf16) if g_f32 is NULL */
int lavt_instnorm_bwd(const float* g_f32, const void* ga_bf16, const void* gb_bf16, const float* xpre, const float* stats, const float* sums,
                      void* out_bf16, int32_t B, int64_t n, int32_t C, void* stream);
/* InstanceNorm reductions of an fp32 gradient: sums [B,2,C] += (sum_n g, sum_n g * IN(xpre)) -- SepTPWAM's summed branches */
int lavt_instnorm_bwd_reduce(const float* g, const float* xpre, const float* stats, float* sums, int32_t B, int64_t n, int32_t C,
                             void* stream);
/* Adjoint of lavt_pwam_kv: dkbuf / dvbuf fp32 [B*heads*NlPad, C] (the GEMM outputs above) -> dwk, dbk, dwv, dbv, dl (all +=) */
int lavt_pwam_kv_bwd(const float* dkbuf, const float* dvbuf, const float* mask, const float* l, const float* wk, const float* wv, float* dwk,
                     float* dbk, float* dwv, float* dbv, float* dl, int32_t B, int32_t Nl, int32_t NlPad, int32_t Lin, int32_t C,
                     int32_t heads, void* stream);
/* Elementwise pieces of the LanguageGate x' = x + tanh(relu(r G0^T) G2^T) * r and of GELU with fp32 sides (count % 8 == 0):
 *   mode 0: out_f32 = f + tanh(a) * b                             (forward: a = gate pre-activation, b = r, f = x)
 *   mode 1: out_bf16 = f * b * (1 - tanh(a)^2); out_f32 = f2 + f * tanh(a)   (f = dx', f2 = gradient of r so far or NULL)
 *   mode 2: out_bf16 = a * [b > 0]                                (ReLU backward: a = dg1, b = g1)
 *   mode 3: out_bf16 = GELU(a), out_f32 = the same                (a = bf16 pre-activation)
 *   mode 4: out_bf16 = f * GELU'(a)                               (f = fp32 gradient)
 *   mode 5: out_bf16 = out_f32 = GELU(a) + f                      (SepTPWAM: sum of the temporal and spatial GELU'd branches)
 *   mode 6: out_f32 = f + f2                                      (--version no_gate: x' = x + r; a = any bf16 tensor of that size)
 *   mode 7 / 8: modes 0 / 1 with a sigmoid instead of a tanh gate (--lg_act_layer sigmoid, reference lib/backbone.py:552-554) */
int lavt_gate_elementwise(int32_t mode, const void* a_bf16, const void* b_bf16, const float* f, const float* f2, void* out_bf16,
                          float* out_f32, int64_t count, void* stream);

/* ---- SimpleDecoding in training mode + loss (lib/mask_predictor.py:56-99 with BatchNorm2d batch statistics; losses.py:7-11) ---- */
/* t bf16 [npix, C] = relu((z - mean) * rstd * gamma + beta); z fp32 conv output, stats fp32 [2, C] = (mean, rstd) over all pixels
 * (lavt_instnorm_stats with B = 1) */
int lavt_bn_relu_apply(const float* z, const float* stats, const float* gamma, const float* beta, void* t_bf16, int64_t npix, int32_t C,
                       void* stream);
/* BatchNorm + ReLU backward, two phases around the (optionally cross-GPU) reduction: sums fp32 [2, C] += (sum dy, sum dy * z^) with
 * dy = dt * [t > 0] (these are d beta, d gamma); then dz bf16 = gamma * rstd * (dy - sums[0]/n_stat - z^ sums[1]/n_stat) */
int lavt_bn_relu_bwd_reduce(const void* dt_bf16, const void* t_bf16, const float* z, const float* stats, float* sums, int64_t npix, int32_t C,
                            void* stream);
int lavt_bn_relu_bwd_apply(const void* dt_bf16, const void* t_bf16, const float* z, const float* stats, const float* gamma, const float* sums,
                           void* dz_bf16, int64_t npix, int64_t n_stat, int32_t C, void* stream);
/* NHWC bf16 [n,H,W,C] (pixel pitch ldi) -> [C, ldo] with column (img*(H+2) + h+1)*Wp + w+1 - dshift (Wp >= W+2, a multiple of 8;
 * dshift in {-1,0,1}); the caller zeroes the buffer (borders).  In this layout tap (ky,kx) of a 3x3 conv is the column offset
 * (ky-1)*Wp + (kx-1): the conv weight gradient is nine lavt_gemm_bf16_splitk calls, A = dz^T (dshift 0), Bt = the copy of x^T
 * written with dshift = kx-1, b_koff = (ky-1)*Wp (TMA needs 16-byte aligned inner coordinates, hence the three shifted copies).
 * D > 0: the n_img frames are clips of D frames, each clip padded with a zero frame on either side (frame index -> clip*(D+2) + d+1):
 * the 27 taps of a Conv3d(3,3,3) weight gradient (SepTPWAM) add (kz-1)*(H+2)*Wp to b_koff.  D = 0: 2-D. */
int lavt_nhwc_pad_transpose(const void* in_bf16, int64_t ldi, void* out_bf16, int64_t ldo, int32_t n_img, int32_t H, int32_t W, int32_t C,
                            int32_t Wp, int32_t dshift, int32_t D, void* stream);
/* adjoint of the upsample half of lavt_upsample_concat: dprev bf16 [n,ph,pw,C1] from dcat bf16 [n,H,W,Ct] (channels 0..C1) */
int lavt_upsample_concat_bwd(const void* dcat_bf16, int32_t Ct, void* dprev_bf16, int32_t ph, int32_t pw, int32_t C1, int32_t n_img, int32_t H,
                             int32_t W, void* stream);
/* adjoint of lavt_conv1x1_logits: dy bf16 [npix, C]; dw fp32 [2, C] and db fp32 [2] accumulate */
int lavt_conv1x1_logits_bwd(const float* dlogits, const void* y_bf16, const float* w, void* dy_bf16, float* dw, float* db, int64_t npix,
                            int32_t C, void* stream);
/* adjoint of lavt_upsample_logits: dout fp32 (n,2,H,W) -> din fp32 (n,h,w,2) */
int lavt_upsample_logits_bwd(const float* dout, float* din, int32_t n_img, int32_t h, int32_t w, int32_t H, int32_t W, void* stream);
/* weighted 2-class cross-entropy over logits fp32 (n,2,H,W) and target int64 (n,H,W) (losses.py:7-11: weights 0.9 / 1.1).
 * phase 0: acc[0] += sum w[t] * nll, acc[1] += sum w[t] (loss = acc[0] / acc[1]);
 * phase 1: dlogits = gscale * w[t] * (softmax - onehot) / acc[1] */
int lavt_cross_entropy(const float* logits, const int64_t* target, float w0, float w1, float* acc, float* dlogits, float gscale, int32_t n_img,
                       int32_t H, int32_t W, int32_t phase, void* stream);

/* ---- optimizer (train.py:688-699: torch.optim.AdamW over the reference's parameter groups + polynomial LR decay) ---- */
typedef struct lavt_adamw_tensor {
  float* p;          /* parameter (fp32, updated in place) */
  const float* g;    /* gradient */
  float* m;          /* exp_avg */
  float* v;          /* exp_avg_sq */
  float* vmax;       /* max_exp_avg_sq (AMSGrad) or NULL */
  int64_t n;         /* elements */
  float bc1, bc2;    /* bias corrections 1 - beta_k^step of THIS tensor (torch keeps one step counter per parameter) */
} lavt_adamw_tensor_t;
/* elements handled per thread block; block_prefix[i] = sum_{j<i} ceil(n_j / chunk), n_blocks = block_prefix[n_tensors] */
int lavt_adamw_chunk_elems(void);
/* One AdamW step for all tensors of a parameter group in one launch (table / prefix are DEVICE arrays).  torch.optim.AdamW
 * semantics: p *= 1 - lr*wd; m, v moment updates; p -= lr/bc1 * m / (sqrt(v or vmax)/sqrt(bc2) + eps), bc_k = 1 - beta_k^step. */
int lavt_adamw_step(const lavt_adamw_tensor_t* table_dev, const int32_t* block_prefix_dev, int32_t n_tensors, int32_t n_blocks,
                    float lr, double beta1, double beta2, float eps, float weight_decay, void* stream);

/* ---- input / output edges of the inference scripts (SURVEY.md section 8f-2) ---- */
/* T.ToTensor() + T.Normalize(mean, std) (train.py:54-60): uint8 HWC frames [n,H,W,3] (already resized) -> fp32 [n,3,H,W];
 * mean3_host / std3_host are HOST arrays of 3 floats */
int lavt_normalize_u8(const uint8_t* frames_hwc, float* out_nchw, int32_t n_img, int32_t H, int32_t W, const float* mean3_host,
                      const float* std3_host, void* stream);
/* F.interpolate(logits, (out_h, out_w), bilinear, align_corners=True).argmax(1) * 255 (test_ytvos.py:249-253, 274-279):
 * fp32 [n,2,H,W] -> uint8 [n,out_h,out_w] */
int lavt_logits_to_mask(const float* logits_nchw, uint8_t* mask, int32_t n_img, int32_t H, int32_t W, int32_t out_h, int32_t out_w,
                        void* stream);

/* ---- GA-CD fusion (lib/bcam.py:78-127; the --gacd ablation of the 2-D image backbone, lib/backbone.py:578-582) ----
 * Everything after mm_gen: xm fp32 [B,n,C] = relu(Linear(ls * x)), lang_stats = the (-ls, 1) block written by lavt_lang_project.
 * One query vector per image, so the collection / diffusion attentions reduce to per-token dot products with u_c = Wc^T q, u_d = Wd^T q,
 * a softmax over the tokens and out[n] = xm[n] + sigmoid(s_d[n]) (Wv sum_n softmax(s_c)[n] xm[n] + bv).  Weights fp32 [C,C] / [C]. */
int64_t lavt_gacd_workspace_floats(int32_t B, int64_t n, int32_t C);
int lavt_gacd_fuse(const float* xm, const float* lang_stats, const float* wq, const float* bq, const float* wc, const float* bc,
                   const float* wd, const float* bd, const float* wv, const float* bv, float* workspace, float* out_f32,
                   void* out_bf16, int32_t B, int64_t n, int32_t C, void* stream);

/* ---- BCAM fusion (lib/bcam.py:8-75; the --bcam ablation of the 2-D image backbone, lib/backbone.py:573-577) ----
 * All contractions of the module are lavt_gemm_bf16 calls; these are the kernels between them.
 * lavt_bcam_words: lr = lang_reduce(l^T) (lib/bcam.py:47): l fp32 [B,Lin,Nl], w fp32 [C,Lin] -> lr bf16 [B,Nlp,C] (rows >= Nl zero) and
 *   its transpose lrT bf16 [B,C,Nlp] (the K-major operands of sim = q lr^T and out = sim lr, :52-56).
 *   With act = LAVT_ACT_GELU and mask fp32 [B,Nl] (else LAVT_ACT_NONE / NULL) the same kernel is EFN's lang = gelu(lang_project(l)) * l_mask
 *   (lib/bcam.py:186-187).
 * lavt_bcam_softmax_rows: p[r, 0:cols] = softmax(s[r, 0:cols] + (1e4 mask[r / rows_per_mask, :] - 1e4)) as bf16, p[r, cols:ldp] = 0
 *   (mask may be NULL): the word softmax (:54-55) and the hw x hw relation map (:62); cols <= 16384.
 * lavt_bcam_transpose_pad: in bf16 [B*n, ldi] (C channels) -> out bf16 [B, C, ldo], columns n..ldo zero: query3 as the K-major
 *   operand of out2 = rel_map query3 (:63-64). */
int lavt_bcam_words(const float* l, const float* w, const float* bias, const float* mask, int32_t act, void* lr_bf16, void* lrT_bf16,
                    int32_t B, int32_t Nl, int32_t Nlp, int32_t Lin, int32_t C, void* stream);
int lavt_bcam_softmax_rows(const float* s, int64_t lds, const float* mask, int64_t rows_per_mask, void* p_bf16, int64_t ldp, int64_t rows,
                           int32_t cols, void* stream);
int lavt_bcam_transpose_pad(const void* in_bf16, int64_t ldi, void* out_bf16, int64_t ldo, int32_t B, int64_t n, int32_t C, void* stream);

/* ---- EFN fusion (lib/bcam.py:160-269; the --efn ablation of the 2-D image backbone, lib/backbone.py:583-588) ----
 * The contractions are lavt_gemm_bf16 calls (the k = 3 Conv1d of EFNAttention.W, :231-233, as three row-shifted accumulating GEMMs; the
 * dim = -2 softmax of :255 as the row softmax of the transposed product); word side / softmaxes / K-major copies are the lavt_bcam_* kernels.
 * lavt_efn_sentence_bias: sb fp32 [B,C] = bias + w sent, sent = masked mean of l fp32 [B,Lin,Nl] (:179-180), w fp32 [C,Lin] with row pitch
 *   ldw: the language half of project's Conv1d over cat[x, sentence] (:183-185) as a per-image bias of the GEMM over x.
 * lavt_efn_norm_pool: out bf16 [B, rows_out, C] = AvgPool2d(2) (pool != 0; n = h*h tokens as a square image, :243-249) of the InstanceNorm of
 *   pre fp32 [B,n,C] with stats fp32 [B,2,C] = (mean, rstd) from lavt_instnorm_stats; rows beyond the n/4 (or n) produced are zero.
 * lavt_efn_norm_upsample: out (fp32 and / or bf16) [B,n,C] = nn.Upsample(scale_factor=2, bilinear) (up != 0, :263-266) of the InstanceNorm of
 *   pre fp32 [B, n/4, C]; up == 0: the InstanceNorm alone.
 * lavt_efn_word_attend: k_pre fp32 [B*n, C] = f_key(L), L = softmax_words(score + (1e4 mask - 1e4)) lang^T (:189-194, :241), evaluated as
 *   sum_j p[i, j] g[b, j, :] with g fp32 [B, g_rows, C] = f_key(lang^T) (bias included) and score fp32 [B*n, lds]: everything stays fp32
 *   because the few words carry all of the token-to-token variation and an InstanceNorm follows.  Nl <= 128. */
int lavt_efn_word_attend(const float* score, int64_t lds, const float* mask, const float* g, int64_t g_rows, float* out, int32_t B, int64_t n,
                         int32_t Nl, int32_t C, void* stream);
int lavt_efn_sentence_bias(const float* l, const float* mask, const float* w, int64_t ldw, const float* bias, float* sb, int32_t B, int32_t Nl,
                           int32_t Lin, int32_t C, void* stream);
int lavt_efn_norm_pool(const float* pre, const float* stats, void* out_bf16, int32_t B, int64_t n, int32_t h, int32_t pool, int64_t rows_out,
                       int32_t C, void* stream);
int lavt_efn_norm_upsample(const float* pre, const float* stats, float* out_f32, void* out_bf16, int32_t B, int64_t n, int32_t h, int32_t up,
                           int32_t C, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LAVT_B200_H_ */
