// Internal dispatch entry points (one per kernel family); called from cabi.cu.
#pragma once
#include "common.cuh"
#include "geom.cuh"

namespace lavt {

enum { MODE_IDENTITY = 0, MODE_WINDOW = 1, MODE_MERGE = 2 };

struct LnParams {
  const float* x;            // source rows, fp32, pitch ldx
  long long ldx;
  const float* gamma;        // [Cn]
  const float* beta;         // [Cn]
  __nv_bfloat16* out_bf16;   // [M, Cn] or nullptr
  float* out_f32;            // [M, Cn] or nullptr
  long long M;               // output rows
  int C;                     // source channels per token
  float eps;
  WinGeom win;               // MODE_WINDOW
  int mB, mD, mH, mW;        // MODE_MERGE: source grid (B,D,H,W)
};
int ln_rows_dispatch(int mode, const LnParams& p, cudaStream_t st);
int im2col_patch4_dispatch(const float* x, long long sB, long long sC, long long sT, __nv_bfloat16* out, int B, int T, int H,
                           int W, cudaStream_t st);
long long colstats_workspace_floats(int B, long long n, int C);
int colstats_dispatch(const float* x, float* stats, float* workspace, int B, long long n, int C, float eps, cudaStream_t st);
int instnorm_sum2_dispatch(const float* a, const float* sa, const float* b, const float* sb, float* out, int B, long long n,
                           int C, cudaStream_t st);
int pwam_mul_dispatch(const __nv_bfloat16* vis, const float* lang, const float* stats, __nv_bfloat16* out, int B,
                      long long n, int C, cudaStream_t st);

struct AttnParams {
  const __nv_bfloat16* qkv;   // [rows, 3C]: q | k | v, each [nH][32]
  const float* table_t;       // [nH, L] relative_position_bias_table, transposed (coalesced per-head reads)
  __nv_bfloat16* out;         // [rows, C]
  int C, nH, L;
  WinGeom win;
  float* lse;                 // [rows, nH] log2-sum-exp2 of every score row, or nullptr (training: saved for the backward; tcgen05 kernel only)
};
int window_attn_dispatch(const AttnParams& p, cudaStream_t st);
int attn_impl_setting(int set);   // set < 0: query only; returns the previous value (0 = auto, 3 = prefer attn_tc2.cu, 4 = attn_tc3.cu where it applies = auto)
// The kernel window_attn_dispatch runs for p (host arithmetic only, no device call): attn_tc3.cu, attn_tc2.cu or the mma.sync
// fallback of attn_window.cu (windows of fewer than 16 tokens; the only choice that writes no lse)
enum class AttnKernel { TC3, TC2, MMA };
AttnKernel window_attn_choose(const AttnParams& p);
// second generation (attn_tc2.cu): key-chunked, one-pass softmax, windows of up to 1152 tokens
bool window_attn_tc2_supported(const AttnParams& p);
int window_attn_tc2_dispatch(const AttnParams& p, cudaStream_t st);
// third generation (attn_tc3.cu): 7 x 7 windows, row-parallel warpgroups, run-padded key layout with vector bias loads
bool window_attn_tc3_supported(const AttnParams& p);
int window_attn_tc3_dispatch(const AttnParams& p, cudaStream_t st);

// ---- backward pass (training step) ----
struct AttnBwdParams {
  const __nv_bfloat16* qkv;    // [rows, 3C] saved by the forward (q pre-scaled by hd^-0.5 * log2 e)
  const __nv_bfloat16* out;    // [rows, C]  forward output O
  const __nv_bfloat16* dout;   // [rows, C]  gradient of O
  const float* table_t;        // [nH, L]
  __nv_bfloat16* dqkv;         // [rows, 3C] gradient of the UNSCALED qkv projection output
  float* dtable_t;             // [nH, L] accumulated (+=), or nullptr
  const float* lse;            // [rows, nH] row statistics saved by the forward kernel, or nullptr (recomputed in a first pass)
  int C, nH, L;
  float qscale;                // hd^-0.5
  WinGeom win;
};
// workspace: fp32 scratch of window_attn_bwd_workspace_floats(p) floats (only attn_bwd_tc2.cu uses one)
int window_attn_bwd_dispatch(const AttnBwdParams& p, float* workspace, long long workspace_floats, cudaStream_t st);
// set < 0: query only; returns the previous value (0 = auto, 1 = mma.sync only, 2 = attn_bwd_tc.cu where it applies (= auto),
// 3 = attn_bwd_tc2.cu wherever it applies)
int attn_bwd_impl_setting(int set);
// The kernel window_attn_bwd_dispatch runs for p (host arithmetic only, no device call): attn_bwd_tc.cu (full 7 x 7 windows with an even
// frame count), the mma.sync kernel of attn_bwd.cu (windows whose Q / K / V / dO and table fit its shared memory: <= 496 tokens at w12),
// attn_bwd_tc2.cu (every other window of 16 ... 1152 tokens with saved lse), or NONE (no kernel: the dispatcher raises)
enum class AttnBwdKernel { NONE = 0, MMA = 1, TC = 2, TC2 = 3 };
AttnBwdKernel window_attn_bwd_choose(const AttnBwdParams& p);
long long window_attn_bwd_workspace_floats(const AttnBwdParams& p);
// tcgen05 / TMEM variant (attn_bwd_tc.cu): 7 x 7 windows with an even number of frames and the forward's saved row statistics
bool window_attn_bwd_tc_supported(const AttnBwdParams& p);
int window_attn_bwd_tc_dispatch(const AttnBwdParams& p, cudaStream_t st);
// tcgen05 / TMEM variant for any window of 16 ... 1152 tokens (attn_bwd_tc2.cu): key tiles outer, dQ partials through an fp32 scratch
bool window_attn_bwd_tc2_supported(const AttnBwdParams& p);
long long window_attn_bwd_tc2_workspace_floats(const AttnBwdParams& p);
int window_attn_bwd_tc2_dispatch(const AttnBwdParams& p, float* workspace, long long workspace_floats, cudaStream_t st);

struct LnBwdParams {
  const float* x;              // LN input rows (fp32, pitch ldx), gathered like the forward
  long long ldx;
  const __nv_bfloat16* dy;     // [M, Cn] gradient of the LN output, in OUTPUT-row order (row pitch lddy)
  long long lddy;
  const float* gamma;          // [Cn]
  const float* dres;           // [tokens, C] gradient already flowing on the residual stream (added), or nullptr
  float* dx;                   // [tokens, C] result (may alias dres)
  float* dgamma;               // [Cn] accumulated (+=)
  float* dbeta;                // [Cn] accumulated (+=)
  long long M;                 // output rows
  int C;
  float eps;
  WinGeom win;                 // MODE_WINDOW
  int mB, mD, mH, mW;          // MODE_MERGE
};
int ln_bwd_dispatch(int mode, const LnBwdParams& p, cudaStream_t st);
int transpose_bf16_dispatch(const __nv_bfloat16* in, long long ldi, __nv_bfloat16* out, long long ldo, long long M, int N,
                            cudaStream_t st);
int colsum_dispatch(const void* x, int is_bf16, long long ldx, long long M, int N, float* dst, cudaStream_t st);
int cast_rows_dispatch(const float* x, long long ldx, __nv_bfloat16* out, long long M, int C, const WinGeom* win, const float* rscale,
                       int rs_rows, cudaStream_t st);
int cast_rows_colsum_dispatch(const float* x, long long ldx, __nv_bfloat16* out, long long M, int C, const WinGeom* win, const float* rscale,
                              int rs_rows, float* colsum, cudaStream_t st);
int lang_project_bwd_dispatch(const float* l, const float* mask, const float* w0, const float* b0, const float* w2, const float* ds, float* dw0,
                              float* db0, float* dw2, float* db2, float* dl, float* workspace, int B, int Nl, int Lin, int C, cudaStream_t st);
int gelu_fwd_dispatch(const __nv_bfloat16* x, __nv_bfloat16* y, long long count, cudaStream_t st);
int gelu_bwd_dispatch(const __nv_bfloat16* dy, const __nv_bfloat16* x, __nv_bfloat16* dx, long long count, cudaStream_t st);

int bn_relu_apply_dispatch(const float* z, const float* stats, const float* gamma, const float* beta, __nv_bfloat16* t, long long npix,
                           int C, cudaStream_t st);
int bn_relu_bwd_dispatch(const __nv_bfloat16* dt, const __nv_bfloat16* t, const float* z, const float* stats, const float* gamma,
                         float* sums, __nv_bfloat16* dz, long long npix, long long n_stat, int C, int phase, cudaStream_t st);
int nhwc_pad_transpose_dispatch(const __nv_bfloat16* in, long long ldi, __nv_bfloat16* out, long long ldo, int n_img, int H, int W, int C,
                                int Wp, int dshift, int D, cudaStream_t st);
int upsample_concat_bwd_dispatch(const __nv_bfloat16* dcat, int Ct, __nv_bfloat16* dprev, int ph, int pw, int C1, int n_img, int H, int W,
                                 cudaStream_t st);
int conv1x1_logits_bwd_dispatch(const float* dlog, const __nv_bfloat16* y, const float* w, __nv_bfloat16* dy, float* dw, float* db,
                                long long npix, int C, cudaStream_t st);
int upsample_logits_bwd_dispatch(const float* dout, float* din, int n_img, int h, int w, int H, int W, cudaStream_t st);
int ce_loss_dispatch(const float* logits, const long long* target, float w0, float w1, float* acc, float* dlogits, float gscale, int n_img,
                     int H, int W, int phase, cudaStream_t st);
int normalize_u8_dispatch(const uint8_t* in, float* out, int n_img, int H, int W, const float* mean, const float* stdv, cudaStream_t st);
int logits_to_mask_dispatch(const float* logits, uint8_t* mask, int n_img, int H, int W, int oh, int ow, cudaStream_t st);
int pwam_attend_bwd_dispatch(const float* qpre, const float* stats, const float* k, const float* v, const float* mask,
                             const __nv_bfloat16* dO, float* dqhat, __nv_bfloat16* qs_out, __nv_bfloat16* P_bd, __nv_bfloat16* dS_bd,
                             float* sums, int B, long long n, int C, int Nl, int NlPad, int heads, cudaStream_t st);
int pwam_mul_bwd_dispatch(const __nv_bfloat16* da2, const __nv_bfloat16* vis, const __nv_bfloat16* vispre, const float* langpre,
                          const float* stats, __nv_bfloat16* dvispre, float* sums, int B, long long n, int C, cudaStream_t st);
int instnorm_bwd_dispatch(const float* g32, const __nv_bfloat16* ga, const __nv_bfloat16* gb, const float* xpre, const float* stats,
                          const float* sums, __nv_bfloat16* out, int B, long long n, int C, cudaStream_t st);
int instnorm_bwd_reduce_dispatch(const float* g, const float* xpre, const float* stats, float* sums, int B, long long n, int C,
                                 cudaStream_t st);
int pwam_kv_bwd_dispatch(const float* dkbuf, const float* dvbuf, const float* mask, const float* l, const float* wk, const float* wv,
                         float* dwk, float* dbk, float* dwv, float* dbv, float* dl, int B, int Nl, int NlPad, int Lin, int C, int heads,
                         cudaStream_t st);
int gate_elem_dispatch(int mode, const __nv_bfloat16* a, const __nv_bfloat16* b, const float* f, const float* f2, __nv_bfloat16* out_bf16,
                       float* out_f32, long long count, cudaStream_t st);

int pwam_kv_dispatch(const float* l, const float* mask, const float* wk, const float* bk, const float* wv, const float* bv,
                     float* k, float* v, int B, int Nl, int Lin, int C, cudaStream_t st);
int lang_project_dispatch(const float* l, const float* mask, const float* w0, const float* b0, const float* w2, const float* b2,
                          float* stats, int B, int Nl, int Lin, int C, cudaStream_t st);
int pwam_core_dispatch(const float* qpre, const float* stats, const float* k, const float* v, const float* mask,
                       __nv_bfloat16* o, int B, long long n, int C, int Nl, int heads, cudaStream_t st);

int bert_embed_dispatch(const long long* ids, const float* word, const float* pos, const float* type0, float* out, int B, int Nl,
                        int H, int vocab, cudaStream_t st);
int bert_attention_dispatch(const __nv_bfloat16* qkv, const float* mask, __nv_bfloat16* out, int B, int Nl, int H, int heads,
                            cudaStream_t st);
int split3_bf16_dispatch(const float* x, long long ldx, __nv_bfloat16* out, long long M, int Kd, cudaStream_t st);
int bert_attention_f32_dispatch(const float* qkv, const float* mask, float* out, int B, int Nl, int H, int heads, cudaStream_t st);
int rows_to_cf_dispatch(const float* in, float* out, int B, int Nl, int C, cudaStream_t st);

int upsample_concat_dispatch(const __nv_bfloat16* prev, int ph, int pw, int C1, const __nv_bfloat16* skip, int C2,
                             __nv_bfloat16* out, int n_img, int H, int W, cudaStream_t st);
int upconv_blend_dispatch(const __nv_bfloat16* Z, int h, int w, int hid, const float* P, const float* s, const float* b,
                          __nv_bfloat16* out, int n_img, int H, int W, cudaStream_t st);
int conv1x1_logits_dispatch(const __nv_bfloat16* y, const float* w, const float* b, float* out, long long npix, int C,
                            cudaStream_t st);
int upsample_logits_dispatch(const float* in, float* out, int n_img, int h, int w, int H, int W, cudaStream_t st);
int nhwc_to_nchw_dispatch(const float* in, float* out, int n_img, int P, int C, cudaStream_t st);
int nchw_to_nhwc_bf16_dispatch(const float* in, __nv_bfloat16* out, int n_img, int P, int C, cudaStream_t st);

}  // namespace lavt
