// extern "C" boundary (include/lavt_b200.h): argument validation + translation into kernel params.
#include "../../include/lavt_b200.h"
#include "common.cuh"
#include "gemm_tc.cuh"
#include "kernels.cuh"

#include <cstring>

namespace lavt {
const char* last_error();
int gemm_dispatch(const void* A, long long lda, const void* Bw, long long ldb, const GemmParams& p,
                  cudaStream_t stream);

static_assert(sizeof(lavt_win_geom_t) == sizeof(WinGeom), "public/private window geometry mismatch");

static int fill_epilogue(GemmParams& p, const lavt_epilogue_t* e) {
  LAVT_REQUIRE(e != nullptr, "epilogue pointer is NULL");
  p.cscale = e->cscale;
  p.bias = e->bias;
  p.act = e->act;
  p.mul = static_cast<const __nv_bfloat16*>(e->mul);
  p.ldm = e->ldm;
  p.mul_act = e->mul_act;
  p.out_pre = static_cast<__nv_bfloat16*>(e->out_pre);
  p.pre_mode = e->pre_mode;
  LAVT_REQUIRE(e->pre_mode == 0 || (e->pre_mode == 1 && e->out_pre && e->act == LAVT_ACT_GELU),
               "epilogue: pre_mode 1 (out_pre = GELU'(pre)) needs out_pre and act = LAVT_ACT_GELU");
  LAVT_REQUIRE(e->mul_act == 0 || (e->mul_act == LAVT_ACT_GELU && e->mul), "epilogue: mul_act must be 0 or LAVT_ACT_GELU with a mul operand");
  p.resid = e->resid;
  p.out_f32 = e->out_f32;
  p.out_bf16 = static_cast<__nv_bfloat16*>(e->out_bf16);
  p.ldo = e->ldo;
  p.rscale = e->rscale;
  p.rs_rows = e->rscale_rows;
  LAVT_REQUIRE(!e->rscale || e->rscale_rows > 0, "epilogue: rscale needs rscale_rows > 0");
  LAVT_REQUIRE(e->act >= 0 && e->act <= 4, "bad activation id %d", e->act);
  if (e->win) {
    p.rowmap = ROWMAP_WINDOW;
    std::memcpy(&p.win, e->win, sizeof(WinGeom));
  } else {
    p.rowmap = ROWMAP_IDENTITY;
  }
  return LAVT_OK;
}
}  // namespace lavt

using namespace lavt;

extern "C" {

const char* lavt_last_error(void) { return lavt::last_error(); }
int lavt_abi_version(void) { return LAVT_ABI_VERSION; }

int lavt_check_device(void) {
  int dev = 0;
  LAVT_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  LAVT_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) {
    set_last_error("device %d is sm_%d%d; this library is built for sm_100a only", dev, prop.major, prop.minor);
    return LAVT_ERR_ARCH;
  }
  return LAVT_OK;
}

int lavt_gemm_bf16(const void* A, int64_t lda, const void* Wt, int64_t ldw, int32_t M, int32_t N, int32_t K,
                   const lavt_epilogue_t* epi, void* stream) {
  GemmParams p;
  std::memset(&p, 0, sizeof(p));
  p.M = M; p.N = N; p.K = K;
  int rc = fill_epilogue(p, epi);
  if (rc) return rc;
  if (p.rowmap == ROWMAP_WINDOW) {
    const WinGeom& g = p.win;
    long long rows = 1LL * g.B * g.nwd * g.nwh * g.nww * g.N;
    LAVT_REQUIRE(rows == M, "gemm: window geometry rows %lld != M %d", rows, M);
  }
  return gemm_dispatch(A, lda, Wt, ldw, p, static_cast<cudaStream_t>(stream));
}

static void conv_pick_tile(GemmParams& p, int H, int W) {
  // 128-pixel tile: widest power-of-two strip that wastes the least padded area
  int best_tw = 8; long long best_area = -1;
  for (int tw = 8; tw <= 128; tw *= 2) {
    int th = 128 / tw;
    long long area = 1LL * ((H + th - 1) / th) * th * ((W + tw - 1) / tw) * tw;
    if (best_area < 0 || area < best_area || (area == best_area && tw > best_tw)) { best_area = area; best_tw = tw; }
  }
  p.cTW = best_tw; p.cTH = 128 / best_tw;
  p.cTilesW = (W + p.cTW - 1) / p.cTW;
  p.cTilesH = (H + p.cTH - 1) / p.cTH;
}

int lavt_conv3x3_bf16(const void* x_nhwc, int64_t ldx, int32_t n_img, int32_t H, int32_t W, int32_t Cin,
                      const void* Wt, int32_t Cout, const lavt_epilogue_t* epi, void* stream) {
  GemmParams p;
  std::memset(&p, 0, sizeof(p));
  LAVT_REQUIRE(n_img > 0 && H > 0 && W > 0, "conv: empty input");
  p.M = n_img * H * W; p.N = Cout; p.K = 9 * Cin;
  int rc = fill_epilogue(p, epi);
  if (rc) return rc;
  LAVT_REQUIRE(p.rowmap == ROWMAP_IDENTITY, "conv: window row map not applicable");
  p.rowmap = ROWMAP_CONV;
  p.cH = H; p.cW = W; p.cCin = Cin; p.taps = 9;
  conv_pick_tile(p, H, W);
  return gemm_dispatch(x_nhwc, ldx, Wt, 9LL * Cin, p, static_cast<cudaStream_t>(stream));
}

int lavt_conv3d_bf16(const void* x_ndhwc, int64_t ldx, int32_t n_clip, int32_t D, int32_t H, int32_t W, int32_t Cin,
                     const void* Wt, int32_t Cout, const lavt_epilogue_t* epi, void* stream) {
  GemmParams p;
  std::memset(&p, 0, sizeof(p));
  LAVT_REQUIRE(n_clip > 0 && D > 0 && H > 0 && W > 0, "conv3d: empty input");
  LAVT_REQUIRE(1LL * n_clip * D * H * W < (1LL << 31), "conv3d: too many output positions");
  p.M = n_clip * D * H * W; p.N = Cout; p.K = 27 * Cin;
  int rc = fill_epilogue(p, epi);
  if (rc) return rc;
  LAVT_REQUIRE(p.rowmap == ROWMAP_IDENTITY, "conv3d: window row map not applicable");
  p.rowmap = ROWMAP_CONV;
  p.cH = H; p.cW = W; p.cCin = Cin; p.taps = 27; p.cD = D;
  conv_pick_tile(p, H, W);
  return gemm_dispatch(x_ndhwc, ldx, Wt, 27LL * Cin, p, static_cast<cudaStream_t>(stream));
}

static inline cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }
static inline const __nv_bfloat16* CB(const void* p) { return static_cast<const __nv_bfloat16*>(p); }
static inline __nv_bfloat16* MB(void* p) { return static_cast<__nv_bfloat16*>(p); }

int lavt_layernorm_rows(const float* x, int64_t ldx, int64_t M, int32_t C, const float* gamma, const float* beta,
                        float eps, void* out_bf16, float* out_f32, void* stream) {
  LnParams p;
  std::memset(&p, 0, sizeof(p));
  p.x = x; p.ldx = ldx; p.gamma = gamma; p.beta = beta; p.out_bf16 = MB(out_bf16); p.out_f32 = out_f32;
  p.M = M; p.C = C; p.eps = eps;
  return ln_rows_dispatch(MODE_IDENTITY, p, S(stream));
}

int lavt_layernorm_window_gather(const float* x, int32_t C, const lavt_win_geom_t* geom, const float* gamma,
                                 const float* beta, float eps, void* out_bf16, void* stream) {
  LAVT_REQUIRE(geom != nullptr, "window gather: geometry is NULL");
  LnParams p;
  std::memset(&p, 0, sizeof(p));
  std::memcpy(&p.win, geom, sizeof(WinGeom));
  p.x = x; p.ldx = C; p.gamma = gamma; p.beta = beta; p.out_bf16 = MB(out_bf16);
  p.M = 1LL * geom->B * geom->nwd * geom->nwh * geom->nww * geom->N; p.C = C; p.eps = eps;
  return ln_rows_dispatch(MODE_WINDOW, p, S(stream));
}

int lavt_patch_merge_layernorm(const float* x, int32_t B, int32_t D, int32_t H, int32_t W, int32_t C,
                               const float* gamma, const float* beta, float eps, void* out_bf16, void* stream) {
  LnParams p;
  std::memset(&p, 0, sizeof(p));
  p.x = x; p.ldx = C; p.gamma = gamma; p.beta = beta; p.out_bf16 = MB(out_bf16);
  p.M = 1LL * B * D * ((H + 1) / 2) * ((W + 1) / 2); p.C = C; p.eps = eps;
  p.mB = B; p.mD = D; p.mH = H; p.mW = W;
  return ln_rows_dispatch(MODE_MERGE, p, S(stream));
}

int lavt_patch_embed_im2col(const float* x, int64_t stride_b, int64_t stride_c, int64_t stride_t, int32_t B, int32_t T,
                            int32_t H, int32_t W, void* out_bf16, void* stream) {
  return im2col_patch4_dispatch(x, stride_b, stride_c, stride_t, MB(out_bf16), B, T, H, W, S(stream));
}

int lavt_window_attention(const void* qkv, const float* table_t, int32_t L, int32_t nH, const lavt_win_geom_t* geom,
                          void* out_bf16, void* stream) {
  LAVT_REQUIRE(geom != nullptr, "attention: geometry is NULL");
  AttnParams p;
  std::memset(&p, 0, sizeof(p));
  std::memcpy(&p.win, geom, sizeof(WinGeom));
  p.qkv = CB(qkv); p.table_t = table_t; p.out = MB(out_bf16); p.nH = nH; p.C = nH * 32; p.L = L;
  return window_attn_dispatch(p, S(stream));
}

int lavt_window_attention_lse(const void* qkv, const float* table_t, int32_t L, int32_t nH, const lavt_win_geom_t* geom, void* out_bf16,
                              float* lse, void* stream) {
  LAVT_REQUIRE(geom != nullptr, "attention: geometry is NULL");
  AttnParams p;
  std::memset(&p, 0, sizeof(p));
  std::memcpy(&p.win, geom, sizeof(WinGeom));
  p.qkv = CB(qkv); p.table_t = table_t; p.out = MB(out_bf16); p.nH = nH; p.C = nH * 32; p.L = L; p.lse = lse;
  return window_attn_dispatch(p, S(stream));
}

int lavt_window_attention_has_lse(const lavt_win_geom_t* geom, int32_t L, int32_t nH) {
  if (geom == nullptr) return 0;
  AttnParams p;
  std::memset(&p, 0, sizeof(p));
  std::memcpy(&p.win, geom, sizeof(WinGeom));
  p.nH = nH; p.C = nH * 32; p.L = L;
  return window_attn_choose(p) != AttnKernel::MMA ? 1 : 0;
}

int lavt_set_attention_bwd_impl(int32_t impl) { return attn_bwd_impl_setting(impl >= 0 && impl <= 3 ? impl : 0); }
int lavt_set_attention_impl(int32_t impl) { return attn_impl_setting(impl == 3 || impl == 4 ? impl : 0); }

int64_t lavt_instnorm_workspace_floats(int32_t B, int64_t n, int32_t C) { return colstats_workspace_floats(B, n, C); }

int lavt_instnorm_stats(const float* x, int32_t B, int64_t n, int32_t C, float eps, float* stats, float* workspace,
                        void* stream) {
  return colstats_dispatch(x, stats, workspace, B, n, C, eps, S(stream));
}

int lavt_pwam_kv(const float* l, const float* mask, const float* wk, const float* bk, const float* wv, const float* bv,
                 float* k, float* v, int32_t B, int32_t Nl, int32_t Lin, int32_t C, void* stream) {
  return pwam_kv_dispatch(l, mask, wk, bk, wv, bv, k, v, B, Nl, Lin, C, S(stream));
}

int lavt_lang_project(const float* l, const float* mask, const float* w0, const float* b0, const float* w2, const float* b2, float* stats,
                      int32_t B, int32_t Nl, int32_t Lin, int32_t C, void* stream) {
  return lang_project_dispatch(l, mask, w0, b0, w2, b2, stats, B, Nl, Lin, C, S(stream));
}

int lavt_pwam_attend(const float* qpre, const float* stats, const float* k, const float* v, const float* mask,
                     void* o_bf16, int32_t B, int64_t n, int32_t C, int32_t Nl, int32_t heads, void* stream) {
  return pwam_core_dispatch(qpre, stats, k, v, mask, MB(o_bf16), B, n, C, Nl, heads, S(stream));
}

int lavt_pwam_mul_norm(const void* vis_bf16, const float* lang, const float* stats, void* out_bf16, int32_t B,
                       int64_t n, int32_t C, void* stream) {
  return pwam_mul_dispatch(CB(vis_bf16), lang, stats, MB(out_bf16), B, n, C, S(stream));
}

int lavt_instnorm_sum2(const float* a, const float* stats_a, const float* b, const float* stats_b, float* out, int32_t B,
                       int64_t n, int32_t C, void* stream) {
  return instnorm_sum2_dispatch(a, stats_a, b, stats_b, out, B, n, C, S(stream));
}

int lavt_bert_embed(const int64_t* ids, const float* word, const float* pos, const float* type0, float* out, int32_t B, int32_t Nl,
                    int32_t H, int32_t vocab, void* stream) {
  return bert_embed_dispatch(reinterpret_cast<const long long*>(ids), word, pos, type0, out, B, Nl, H, vocab, S(stream));
}

int lavt_bert_attention(const void* qkv_bf16, const float* mask, void* out_bf16, int32_t B, int32_t Nl, int32_t H, int32_t heads,
                        void* stream) {
  return bert_attention_dispatch(CB(qkv_bf16), mask, MB(out_bf16), B, Nl, H, heads, S(stream));
}

int lavt_split3_bf16(const float* x, int64_t ldx, void* out_bf16, int64_t M, int32_t K, void* stream) {
  return split3_bf16_dispatch(x, ldx, MB(out_bf16), M, K, S(stream));
}
int lavt_bert_attention_f32(const float* qkv, const float* mask, float* out, int32_t B, int32_t Nl, int32_t H, int32_t heads, void* stream) {
  return bert_attention_f32_dispatch(qkv, mask, out, B, Nl, H, heads, S(stream));
}
int lavt_rows_to_channels_first(const float* in, float* out, int32_t B, int32_t Nl, int32_t C, void* stream) {
  return rows_to_cf_dispatch(in, out, B, Nl, C, S(stream));
}

int lavt_upsample_concat(const void* prev_bf16, int32_t ph, int32_t pw, int32_t C1, const void* skip_bf16, int32_t C2,
                         void* out_bf16, int32_t n_img, int32_t H, int32_t W, void* stream) {
  return upsample_concat_dispatch(CB(prev_bf16), ph, pw, C1, CB(skip_bf16), C2, MB(out_bf16), n_img, H, W, S(stream));
}

int lavt_upconv_blend(const void* z_bf16, int32_t h, int32_t w, int32_t hid, const float* P, const float* s, const float* b, void* out_bf16,
                      int32_t n_img, int32_t H, int32_t W, void* stream) {
  return upconv_blend_dispatch(CB(z_bf16), h, w, hid, P, s, b, MB(out_bf16), n_img, H, W, S(stream));
}

int lavt_conv1x1_logits(const void* y_bf16, const float* w, const float* b, float* out, int64_t npix, int32_t C, void* stream) {
  return conv1x1_logits_dispatch(CB(y_bf16), w, b, out, npix, C, S(stream));
}

int lavt_upsample_logits(const float* in, float* out, int32_t n_img, int32_t h, int32_t w, int32_t H, int32_t W, void* stream) {
  return upsample_logits_dispatch(in, out, n_img, h, w, H, W, S(stream));
}

int lavt_nhwc_to_nchw(const float* in, float* out, int32_t n_img, int32_t P, int32_t C, void* stream) {
  return nhwc_to_nchw_dispatch(in, out, n_img, P, C, S(stream));
}

int lavt_nchw_to_nhwc_bf16(const float* in, void* out_bf16, int32_t n_img, int32_t P, int32_t C, void* stream) {
  return nchw_to_nhwc_bf16_dispatch(in, MB(out_bf16), n_img, P, C, S(stream));
}

/* ------------------------------------------------------------------------------------------------
 * backward pass (training step)
 * ------------------------------------------------------------------------------------------------ */
static void splitk_plan(int M, int N, int K, int* ksplit, int* kbs) {
  // (tile, split) work items over the CTA slots of the variant gemm_variant() will pick.  The first planner filled at most ONE wave
  // (tiles x 5 = 320 items on 296 slots had run as two waves, the second one 8 % full: ncu showed the tensor pipe at 30 %), which
  // left 92 tiles of the Cin = 640 conv weight gradient on 148 SMs unsplit (62 % of the machine) and capped single-tile problems at
  // 64 items.  Now: the split count with the lowest modelled time, in units of one k-block of one tile --
  //   waves(s) * (k-blocks per item + per-item overhead) + s * (write + read of one fp32 partial of the whole output)
  // so that several FULL waves (92 x 8 = 736 items = 4.97 waves) are as good as one.
  const int num_kb = (K + 63) / 64;
  const bool wide = (N % 256) == 0;                       // 128 x 256 tiles, one CTA per SM
  const long long tiles = 1LL * ((M + 127) / 128) * (wide ? N / 256 : (N + 127) / 128);
  const long long slots = wide ? 148 : (K >= 1024 ? 296 : 148);
  const double part = 1.0 * M * N * (wide ? 1.6e-6 : 3.2e-6);          // partial traffic of one split / time of one k-block
  const double ovh = 6.0;                                 // pipeline fill + the part of the drain the next item cannot hide
  long long smax = num_kb < 512 ? num_kb : 512;
  const long long ws_cap = (64LL << 20) / (1LL * M * N);  // <= 256 MB of fp32 partials
  if (smax > ws_cap) smax = ws_cap < 1 ? 1 : ws_cap;
  double best = 0.0;
  int best_kbs = num_kb;
  for (long long s = 1; s <= smax; ++s) {
    const long long kb = (num_kb + s - 1) / s;
    const long long sp = (num_kb + kb - 1) / kb;          // splits that actually own k-blocks
    const long long waves = (tiles * sp + slots - 1) / slots;
    const double cost = waves * (kb + ovh) + (sp > 1 ? sp * part : 0.0);
    if (s == 1 || cost < best * 0.98) {                   // a finer split has to win by 2 % to be taken
      best = cost;
      best_kbs = static_cast<int>(kb);
    }
  }
  *kbs = best_kbs;
  *ksplit = (num_kb + *kbs - 1) / *kbs;
}

int64_t lavt_gemm_splitk_workspace_floats(int32_t M, int32_t N, int32_t K) {
  int ks, kbs;
  splitk_plan(M, N, K, &ks, &kbs);
  return 1LL * ks * M * N;
}

int lavt_gemm_bf16_splitk(const void* A, int64_t lda, const void* Bt, int64_t ldb, int32_t M, int32_t N, int32_t K, int32_t b_koff,
                          float* workspace, int64_t workspace_floats, float* dst, int64_t ldd, int32_t accumulate, void* stream) {
  GemmParams p;
  std::memset(&p, 0, sizeof(p));
  p.M = M; p.N = N; p.K = K;
  int ks, kbs;
  splitk_plan(M, N, K, &ks, &kbs);
  LAVT_REQUIRE(workspace && workspace_floats >= 1LL * ks * M * N, "split-K gemm: workspace too small (%lld < %lld floats)",
               static_cast<long long>(workspace_floats), 1LL * ks * M * N);
  LAVT_REQUIRE(dst != nullptr && ldd >= N, "split-K gemm: bad destination");
  LAVT_REQUIRE(b_koff % 8 == 0, "split-K gemm: b_koff=%d must be a multiple of 8 elements (TMA needs a 16-byte aligned inner coordinate)", b_koff);
  p.out_f32 = workspace;
  p.ldo = N;
  p.rowmap = ROWMAP_IDENTITY;
  p.ksplit = ks;
  p.kbs = kbs;
  p.split_stride = 1LL * M * N;
  p.b_koff = b_koff;
  int rc = gemm_dispatch(A, lda, Bt, ldb, p, S(stream));
  if (rc) return rc;
  return splitk_reduce_dispatch(workspace, ks, 1LL * M * N, N, dst, ldd, accumulate, S(stream));
}

int lavt_gemm_bf16_smallm(const void* A, int64_t lda, const void* Wt, int64_t ldw, int32_t M, int32_t N, int32_t K,
                          const lavt_epilogue_t* epi, float* workspace, int64_t workspace_floats, void* stream) {
  GemmParams e;
  std::memset(&e, 0, sizeof(e));
  int rc = fill_epilogue(e, epi);
  if (rc) return rc;
  LAVT_REQUIRE(e.rowmap == ROWMAP_IDENTITY && !e.mul && !e.out_pre && !e.pre_mode && !e.rscale && (e.act == 0 || e.act == 1), "small-M gemm: epilogue not supported");
  GemmParams p;
  std::memset(&p, 0, sizeof(p));
  p.M = M; p.N = N; p.K = K;
  int ks, kbs;
  splitk_plan(M, N, K, &ks, &kbs);
  LAVT_REQUIRE(workspace && workspace_floats >= 1LL * ks * M * N, "small-M gemm: workspace too small (%lld < %lld floats)",
               static_cast<long long>(workspace_floats), 1LL * ks * M * N);
  p.out_f32 = workspace;
  p.ldo = N;
  p.rowmap = ROWMAP_IDENTITY;
  p.ksplit = ks;
  p.kbs = kbs;
  p.split_stride = 1LL * M * N;
  rc = gemm_dispatch(A, lda, Wt, ldw, p, S(stream));
  if (rc) return rc;
  return splitk_epilogue_dispatch(workspace, ks, M, N, e.cscale, e.bias, e.act, e.resid, e.out_f32, e.out_bf16, e.ldo, S(stream));
}

int lavt_gemm_bf16_wgrad(const void* dy, int64_t lddy, const void* x, int64_t ldx, int64_t tokens, int32_t n_out, int32_t n_in,
                         float* workspace, int64_t workspace_floats, float* dst, int64_t ldd, int32_t accumulate, void* stream) {
  LAVT_REQUIRE(tokens > 0 && tokens < (1LL << 31), "wgrad gemm: token count out of range");
  GemmParams p;
  std::memset(&p, 0, sizeof(p));
  p.M = n_out; p.N = n_in; p.K = static_cast<int>(tokens);
  int ks, kbs;
  splitk_plan(p.M, p.N, p.K, &ks, &kbs);
  LAVT_REQUIRE(workspace && workspace_floats >= 1LL * ks * p.M * p.N, "wgrad gemm: workspace too small (%lld < %lld floats)",
               static_cast<long long>(workspace_floats), 1LL * ks * p.M * p.N);
  LAVT_REQUIRE(dst != nullptr && ldd >= n_in, "wgrad gemm: bad destination");
  p.out_f32 = workspace;
  p.ldo = p.N;
  p.rowmap = ROWMAP_IDENTITY;
  p.ksplit = ks;
  p.kbs = kbs;
  p.split_stride = 1LL * p.M * p.N;
  p.mnmajor = 1;
  int rc = gemm_dispatch(dy, lddy, x, ldx, p, S(stream));
  if (rc) return rc;
  return splitk_reduce_dispatch(workspace, ks, 1LL * p.M * p.N, p.N, dst, ldd, accumulate, S(stream));
}

static void wgrad_tile(GemmParams& p, int H, int W) {
  int tw = 8; long long best = -1;
  for (int t = 1; t <= 64; t *= 2) {          // 64-pixel tile with the least padded area
    const int th = 64 / t;
    const long long area = 1LL * ((H + th - 1) / th) * th * ((W + t - 1) / t) * t;
    if (best < 0 || area < best || (area == best && t > tw)) { best = area; tw = t; }
  }
  p.cTW = tw; p.cTH = 64 / tw;
  p.cTilesW = (W + p.cTW - 1) / p.cTW;
  p.cTilesH = (H + p.cTH - 1) / p.cTH;
  p.cH = H; p.cW = W;
}

static int conv_wgrad_impl(const void* dz, const void* x, int n_frames, int D, int H, int W, int Cin, int Cout, int taps, float* workspace,
                           int64_t workspace_floats, float* dw_taps, int accumulate, void* stream, int64_t* need_only) {
  GemmParams p;
  std::memset(&p, 0, sizeof(p));
  wgrad_tile(p, H, W);
  p.cCin = Cin; p.taps = taps; p.cD = D;
  const long long K = 1LL * n_frames * p.cTilesH * p.cTilesW * 64;
  LAVT_REQUIRE(K < (1LL << 31), "conv wgrad: too many pixels");
  p.M = Cout; p.N = taps * Cin; p.K = static_cast<int>(K);
  int ks, kbs;
  splitk_plan(p.M, p.N, p.K, &ks, &kbs);
  if (need_only) { *need_only = 1LL * ks * p.M * p.N; return LAVT_OK; }
  LAVT_REQUIRE(n_frames > 0 && H > 0 && W > 0 && Cin % 64 == 0 && Cout % 8 == 0, "conv wgrad: need Cin %% 64 == 0 and Cout %% 8 == 0 (Cin=%d, Cout=%d)", Cin, Cout);
  LAVT_REQUIRE(workspace && workspace_floats >= 1LL * ks * p.M * p.N, "conv wgrad: workspace too small");
  p.out_f32 = workspace;
  p.ldo = p.N;
  p.rowmap = ROWMAP_WGCONV;
  p.mnmajor = 1;
  p.ksplit = ks; p.kbs = kbs; p.split_stride = 1LL * p.M * p.N;
  int rc = gemm_dispatch(dz, Cout, x, Cin, p, S(stream));
  if (rc) return rc;
  return splitk_reduce_dispatch(workspace, ks, 1LL * p.M * p.N, p.N, dw_taps, p.N, accumulate, S(stream));
}

int64_t lavt_conv3x3_wgrad_workspace_floats(int32_t n_img, int32_t H, int32_t W, int32_t Cin, int32_t Cout) {
  int64_t need = 0;
  conv_wgrad_impl(nullptr, nullptr, n_img, 0, H, W, Cin, Cout, 9, nullptr, 0, nullptr, 0, nullptr, &need);
  return need;
}
int lavt_conv3x3_wgrad(const void* dz_nhwc, const void* x_nhwc, int32_t n_img, int32_t H, int32_t W, int32_t Cin, int32_t Cout,
                       float* workspace, int64_t workspace_floats, float* dw_taps, int32_t accumulate, void* stream) {
  return conv_wgrad_impl(dz_nhwc, x_nhwc, n_img, 0, H, W, Cin, Cout, 9, workspace, workspace_floats, dw_taps, accumulate, stream, nullptr);
}
int64_t lavt_conv3d_wgrad_workspace_floats(int32_t n_clip, int32_t D, int32_t H, int32_t W, int32_t Cin, int32_t Cout) {
  int64_t need = 0;
  conv_wgrad_impl(nullptr, nullptr, n_clip * D, D, H, W, Cin, Cout, 27, nullptr, 0, nullptr, 0, nullptr, &need);
  return need;
}
int lavt_conv3d_wgrad(const void* dz_ndhwc, const void* x_ndhwc, int32_t n_clip, int32_t D, int32_t H, int32_t W, int32_t Cin, int32_t Cout,
                      float* workspace, int64_t workspace_floats, float* dw_taps, int32_t accumulate, void* stream) {
  LAVT_REQUIRE(D >= 1, "conv3d wgrad: D must be >= 1");
  return conv_wgrad_impl(dz_ndhwc, x_ndhwc, n_clip * D, D, H, W, Cin, Cout, 27, workspace, workspace_floats, dw_taps, accumulate, stream, nullptr);
}

int lavt_transpose_bf16(const void* in, int64_t ldi, void* out, int64_t ldo, int64_t M, int32_t N, void* stream) {
  return transpose_bf16_dispatch(CB(in), ldi, MB(out), ldo, M, N, S(stream));
}

int lavt_colsum_accumulate(const void* x, int32_t is_bf16, int64_t ldx, int64_t M, int32_t N, float* dst, void* stream) {
  return colsum_dispatch(x, is_bf16, ldx, M, N, dst, S(stream));
}

int lavt_cast_rows_scaled_bf16(const float* x, int64_t ldx, int64_t M, int32_t C, const lavt_win_geom_t* geom, const float* rscale,
                               int32_t rscale_rows, void* out_bf16, void* stream) {
  WinGeom g;
  if (geom) {
    std::memcpy(&g, geom, sizeof(g));
    LAVT_REQUIRE(M == 1LL * g.B * g.nwd * g.nwh * g.nww * g.N, "cast rows: M does not match the window geometry");
  }
  LAVT_REQUIRE(!rscale || rscale_rows > 0, "cast rows: rscale needs rscale_rows > 0");
  return cast_rows_dispatch(x, ldx, MB(out_bf16), M, C, geom ? &g : nullptr, rscale, rscale_rows, S(stream));
}
int lavt_cast_rows_colsum_bf16(const float* x, int64_t ldx, int64_t M, int32_t C, const lavt_win_geom_t* geom, const float* rscale,
                               int32_t rscale_rows, void* out_bf16, float* colsum, void* stream) {
  WinGeom g;
  if (geom) {
    std::memcpy(&g, geom, sizeof(g));
    LAVT_REQUIRE(M == 1LL * g.B * g.nwd * g.nwh * g.nww * g.N, "cast rows: M does not match the window geometry");
  }
  LAVT_REQUIRE(!rscale || rscale_rows > 0, "cast rows: rscale needs rscale_rows > 0");
  return cast_rows_colsum_dispatch(x, ldx, MB(out_bf16), M, C, geom ? &g : nullptr, rscale, rscale_rows, colsum, S(stream));
}
int lavt_cast_rows_bf16(const float* x, int64_t ldx, int64_t M, int32_t C, const lavt_win_geom_t* geom, void* out_bf16, void* stream) {
  return lavt_cast_rows_scaled_bf16(x, ldx, M, C, geom, nullptr, 0, out_bf16, stream);
}

int lavt_lang_project_bwd(const float* l, const float* mask, const float* w0, const float* b0, const float* w2, const float* ds, float* dw0,
                          float* db0, float* dw2, float* db2, float* dl, float* workspace, int32_t B, int32_t Nl, int32_t Lin, int32_t C, void* stream) {
  return lang_project_bwd_dispatch(l, mask, w0, b0, w2, ds, dw0, db0, dw2, db2, dl, workspace, B, Nl, Lin, C, S(stream));
}
int lavt_gelu_fwd(const void* x_bf16, void* y_bf16, int64_t count, void* stream) {
  return gelu_fwd_dispatch(CB(x_bf16), MB(y_bf16), count, S(stream));
}
int lavt_gelu_bwd(const void* dy_bf16, const void* x_bf16, void* dx_bf16, int64_t count, void* stream) {
  return gelu_bwd_dispatch(CB(dy_bf16), CB(x_bf16), MB(dx_bf16), count, S(stream));
}

int lavt_layernorm_rows_bwd(const float* x, int64_t ldx, int64_t M, int32_t C, const void* dy_bf16, int64_t lddy, const float* gamma, float eps,
                            const float* dres, float* dx, float* dgamma, float* dbeta, void* stream) {
  LnBwdParams p;
  std::memset(&p, 0, sizeof(p));
  p.x = x; p.ldx = ldx; p.dy = CB(dy_bf16); p.lddy = lddy; p.gamma = gamma; p.dres = dres; p.dx = dx; p.dgamma = dgamma; p.dbeta = dbeta;
  p.M = M; p.C = C; p.eps = eps;
  return ln_bwd_dispatch(MODE_IDENTITY, p, S(stream));
}

int lavt_layernorm_window_gather_bwd(const float* x, int32_t C, const lavt_win_geom_t* geom, const void* dy_bf16, const float* gamma,
                                     float eps, const float* dres, float* dx, float* dgamma, float* dbeta, void* stream) {
  LAVT_REQUIRE(geom != nullptr, "window gather backward: geometry is NULL");
  LnBwdParams p;
  std::memset(&p, 0, sizeof(p));
  std::memcpy(&p.win, geom, sizeof(WinGeom));
  p.x = x; p.ldx = C; p.dy = CB(dy_bf16); p.lddy = C; p.gamma = gamma; p.dres = dres; p.dx = dx; p.dgamma = dgamma; p.dbeta = dbeta;
  p.M = 1LL * p.win.B * p.win.nwd * p.win.nwh * p.win.nww * p.win.N; p.C = C; p.eps = eps;
  return ln_bwd_dispatch(MODE_WINDOW, p, S(stream));
}

int lavt_patch_merge_layernorm_bwd(const float* x, int32_t B, int32_t D, int32_t H, int32_t W, int32_t C, const void* dy_bf16,
                                   const float* gamma, float eps, float* dx, float* dgamma, float* dbeta, void* stream) {
  LnBwdParams p;
  std::memset(&p, 0, sizeof(p));
  p.x = x; p.ldx = C; p.dy = CB(dy_bf16); p.lddy = 4 * C; p.gamma = gamma; p.dres = nullptr; p.dx = dx; p.dgamma = dgamma; p.dbeta = dbeta;
  p.M = 1LL * B * D * ((H + 1) / 2) * ((W + 1) / 2); p.C = C; p.eps = eps;
  p.mB = B; p.mD = D; p.mH = H; p.mW = W;
  return ln_bwd_dispatch(MODE_MERGE, p, S(stream));
}

static AttnBwdParams attn_bwd_params(const lavt_win_geom_t* geom, int32_t L, int32_t nH) {
  AttnBwdParams p;
  std::memset(&p, 0, sizeof(p));
  std::memcpy(&p.win, geom, sizeof(WinGeom));
  p.C = nH * 32; p.nH = nH; p.L = L;
  p.qscale = 0.17677669529663687f;      // 32^-0.5
  return p;
}

int lavt_window_attention_bwd(const void* qkv, const void* out, const void* dout, const float* table_t, int32_t L, int32_t nH,
                              const lavt_win_geom_t* geom, const float* lse, void* dqkv, float* dtable_t, float* workspace,
                              int64_t workspace_floats, void* stream) {
  LAVT_REQUIRE(geom != nullptr, "attention backward: geometry is NULL");
  AttnBwdParams p = attn_bwd_params(geom, L, nH);
  p.qkv = CB(qkv); p.out = CB(out); p.dout = CB(dout); p.table_t = table_t; p.dqkv = MB(dqkv); p.dtable_t = dtable_t; p.lse = lse;
  LAVT_REQUIRE(L == (2 * p.win.Wd - 1) * (2 * p.win.Wh - 1) * (2 * p.win.Ww - 1), "attention backward: table length %d does not match the window", L);
  return window_attn_bwd_dispatch(p, workspace, workspace_floats, S(stream));
}

int lavt_window_attention_bwd_kernel(const lavt_win_geom_t* geom, int32_t L, int32_t nH, int32_t has_lse) {
  if (geom == nullptr) return 0;
  static const float lse_tag = 0.f;      // only compared against NULL: the choice is host arithmetic
  AttnBwdParams p = attn_bwd_params(geom, L, nH);
  if (has_lse) p.lse = &lse_tag;
  return static_cast<int>(window_attn_bwd_choose(p));
}

int64_t lavt_window_attention_bwd_workspace_floats(const lavt_win_geom_t* geom, int32_t L, int32_t nH) {
  if (geom == nullptr) return 0;
  static const float lse_tag = 0.f;
  AttnBwdParams p = attn_bwd_params(geom, L, nH);
  p.lse = &lse_tag;                      // the training path always saves lse; without it no kernel with a workspace applies
  return window_attn_bwd_workspace_floats(p);
}

int lavt_pwam_attend_bwd(const float* qpre, const float* stats, const float* k, const float* v, const float* mask, const void* do_bf16,
                         float* dqhat, void* qs_bf16, void* p_bd, void* ds_bd, float* sums, int32_t B, int64_t n, int32_t C, int32_t Nl,
                         int32_t NlPad, int32_t heads, void* stream) {
  return pwam_attend_bwd_dispatch(qpre, stats, k, v, mask, CB(do_bf16), dqhat, MB(qs_bf16), MB(p_bd), MB(ds_bd), sums, B, n, C, Nl, NlPad,
                                  heads, S(stream));
}
int lavt_pwam_mul_norm_bwd(const void* da2, const void* vis, const void* vispre, const float* langpre, const float* stats, void* dvispre,
                           float* sums, int32_t B, int64_t n, int32_t C, void* stream) {
  return pwam_mul_bwd_dispatch(CB(da2), CB(vis), CB(vispre), langpre, stats, MB(dvispre), sums, B, n, C, S(stream));
}
int lavt_instnorm_bwd(const float* g_f32, const void* ga_bf16, const void* gb_bf16, const float* xpre, const float* stats, const float* sums,
                      void* out_bf16, int32_t B, int64_t n, int32_t C, void* stream) {
  return instnorm_bwd_dispatch(g_f32, CB(ga_bf16), CB(gb_bf16), xpre, stats, sums, MB(out_bf16), B, n, C, S(stream));
}
int lavt_instnorm_bwd_reduce(const float* g, const float* xpre, const float* stats, float* sums, int32_t B, int64_t n, int32_t C,
                             void* stream) {
  return instnorm_bwd_reduce_dispatch(g, xpre, stats, sums, B, n, C, S(stream));
}
int lavt_pwam_kv_bwd(const float* dkbuf, const float* dvbuf, const float* mask, const float* l, const float* wk, const float* wv, float* dwk,
                     float* dbk, float* dwv, float* dbv, float* dl, int32_t B, int32_t Nl, int32_t NlPad, int32_t Lin, int32_t C,
                     int32_t heads, void* stream) {
  return pwam_kv_bwd_dispatch(dkbuf, dvbuf, mask, l, wk, wv, dwk, dbk, dwv, dbv, dl, B, Nl, NlPad, Lin, C, heads, S(stream));
}
int lavt_gate_elementwise(int32_t mode, const void* a_bf16, const void* b_bf16, const float* f, const float* f2, void* out_bf16,
                          float* out_f32, int64_t count, void* stream) {
  return gate_elem_dispatch(mode, CB(a_bf16), CB(b_bf16), f, f2, MB(out_bf16), out_f32, count, S(stream));
}

int lavt_bn_relu_apply(const float* z, const float* stats, const float* gamma, const float* beta, void* t_bf16, int64_t npix, int32_t C,
                       void* stream) {
  return bn_relu_apply_dispatch(z, stats, gamma, beta, MB(t_bf16), npix, C, S(stream));
}
int lavt_bn_relu_bwd_reduce(const void* dt_bf16, const void* t_bf16, const float* z, const float* stats, float* sums, int64_t npix, int32_t C,
                            void* stream) {
  return bn_relu_bwd_dispatch(CB(dt_bf16), CB(t_bf16), z, stats, nullptr, sums, nullptr, npix, npix, C, 0, S(stream));
}
int lavt_bn_relu_bwd_apply(const void* dt_bf16, const void* t_bf16, const float* z, const float* stats, const float* gamma, const float* sums,
                           void* dz_bf16, int64_t npix, int64_t n_stat, int32_t C, void* stream) {
  return bn_relu_bwd_dispatch(CB(dt_bf16), CB(t_bf16), z, stats, gamma, const_cast<float*>(sums), MB(dz_bf16), npix, n_stat, C, 1, S(stream));
}
int lavt_nhwc_pad_transpose(const void* in_bf16, int64_t ldi, void* out_bf16, int64_t ldo, int32_t n_img, int32_t H, int32_t W, int32_t C,
                            int32_t Wp, int32_t dshift, int32_t D, void* stream) {
  return nhwc_pad_transpose_dispatch(CB(in_bf16), ldi, MB(out_bf16), ldo, n_img, H, W, C, Wp, dshift, D, S(stream));
}
int lavt_upsample_concat_bwd(const void* dcat_bf16, int32_t Ct, void* dprev_bf16, int32_t ph, int32_t pw, int32_t C1, int32_t n_img, int32_t H,
                             int32_t W, void* stream) {
  return upsample_concat_bwd_dispatch(CB(dcat_bf16), Ct, MB(dprev_bf16), ph, pw, C1, n_img, H, W, S(stream));
}
int lavt_conv1x1_logits_bwd(const float* dlogits, const void* y_bf16, const float* w, void* dy_bf16, float* dw, float* db, int64_t npix,
                            int32_t C, void* stream) {
  return conv1x1_logits_bwd_dispatch(dlogits, CB(y_bf16), w, MB(dy_bf16), dw, db, npix, C, S(stream));
}
int lavt_upsample_logits_bwd(const float* dout, float* din, int32_t n_img, int32_t h, int32_t w, int32_t H, int32_t W, void* stream) {
  return upsample_logits_bwd_dispatch(dout, din, n_img, h, w, H, W, S(stream));
}
int lavt_cross_entropy(const float* logits, const int64_t* target, float w0, float w1, float* acc, float* dlogits, float gscale, int32_t n_img,
                       int32_t H, int32_t W, int32_t phase, void* stream) {
  return ce_loss_dispatch(logits, reinterpret_cast<const long long*>(target), w0, w1, acc, dlogits, gscale, n_img, H, W, phase, S(stream));
}

}  // extern "C"
