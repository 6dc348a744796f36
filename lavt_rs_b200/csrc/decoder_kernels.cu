// Bandwidth-bound pieces of SimpleDecoding (reference lib/mask_predictor.py:56-99) and the final logits
// upsample (lib/_utils.py:106).  The conv3x3+BN+ReLU stack itself runs on the tcgen05 implicit-GEMM kernel.
//
//   upsample_concat   cat[ bilinear(prev -> skip size, align_corners=True), skip ]  -> NHWC bf16 conv input
//   conv1x1_logits    512 -> 2 pointwise conv + bias (one warp per pixel)          -> (pix, 2) fp32
//   upsample_logits   (n,h,w,2) fp32 -> (n,2,H,W) fp32 NCHW, bilinear align_corners=True
//   nhwc_to_nchw      fp32 NHWC -> NCHW (API-compat output layout of backbone.forward) via smem transpose
//   nchw_to_nhwc_bf16 fp32 NCHW -> NHWC bf16 (API-compat input layout of classifier.forward)
#include "kernels.cuh"

namespace lavt {

__device__ __forceinline__ void bilinear_taps(int o, int in, int out, int& i0, int& i1, float& f) {
  // align_corners=True: src = o * (in-1)/(out-1)
  const float s = (out > 1) ? static_cast<float>(o) * (static_cast<float>(in - 1) / static_cast<float>(out - 1)) : 0.f;
  i0 = min(static_cast<int>(s), in - 1);
  i1 = min(i0 + 1, in - 1);
  f = s - static_cast<float>(i0);
}

// thread per (pixel, 8-channel group): consecutive threads touch consecutive 16-byte chunks, so every load / store
// instruction of a warp covers 512 contiguous bytes (the bilinear taps of neighbouring pixels share cache lines)
__global__ void __launch_bounds__(256) upsample_concat_kernel(const __nv_bfloat16* __restrict__ prev, int ph, int pw, int C1,
                                                              const __nv_bfloat16* __restrict__ skip, int C2,
                                                              __nv_bfloat16* __restrict__ out, int n_img, int H, int W) {
  // grid = (chunks of one output row, H, images): no 64-bit index arithmetic on the per-thread path
  const int Ct = C1 + C2, g8 = Ct / 8;
  const int xi = blockIdx.x * blockDim.x + threadIdx.x;
  if (xi >= W * g8) return;
  const int w = xi / g8;
  const int c = (xi - w * g8) * 8;
  const int h = blockIdx.y;
  const long long img = blockIdx.z;
  const long long pix = (img * H + h) * W + w;
  uint4 r;
  if (c >= C1) {
    r = __ldg(reinterpret_cast<const uint4*>(skip + pix * C2 + (c - C1)));
  } else if (ph == H && pw == W) {
    r = __ldg(reinterpret_cast<const uint4*>(prev + pix * C1 + c));
  } else {
    int y0, y1, x0, x1;
    float fy, fx;
    bilinear_taps(h, ph, H, y0, y1, fy);
    bilinear_taps(w, pw, W, x0, x1, fx);
    const float w00 = (1.f - fy) * (1.f - fx), w01 = (1.f - fy) * fx, w10 = fy * (1.f - fx), w11 = fy * fx;
    const __nv_bfloat16* pbase = prev + img * ph * pw * C1 + c;
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(pbase + (static_cast<long long>(y0) * pw + x0) * C1));
    const uint4 bq = __ldg(reinterpret_cast<const uint4*>(pbase + (static_cast<long long>(y0) * pw + x1) * C1));
    const uint4 cc = __ldg(reinterpret_cast<const uint4*>(pbase + (static_cast<long long>(y1) * pw + x0) * C1));
    const uint4 d = __ldg(reinterpret_cast<const uint4*>(pbase + (static_cast<long long>(y1) * pw + x1) * C1));
    const uint32_t ua[4] = {a.x, a.y, a.z, a.w}, ub[4] = {bq.x, bq.y, bq.z, bq.w}, uc[4] = {cc.x, cc.y, cc.z, cc.w},
                   ud[4] = {d.x, d.y, d.z, d.w};
    uint32_t uo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 fa = unpack_bf16x2(ua[j]), fb = unpack_bf16x2(ub[j]), fc = unpack_bf16x2(uc[j]), fd = unpack_bf16x2(ud[j]);
      uo[j] = pack_bf16x2(w00 * fa.x + w01 * fb.x + w10 * fc.x + w11 * fd.x, w00 * fa.y + w01 * fb.y + w10 * fc.y + w11 * fd.y);
    }
    r = make_uint4(uo[0], uo[1], uo[2], uo[3]);
  }
  *reinterpret_cast<uint4*>(out + pix * Ct + c) = r;
}

// Exact x2 upsampling (H == 2 ph, W == 2 pw: every level of SimpleDecoding): a thread produces a 2 x 2 block of output pixels for 8 channels.
// With align_corners the source coordinate of output 2j lies in (j - 1, j] and that of 2j + 1 in (j, j + 1/2), so the block reads the 3 x 3
// input neighbourhood (j - 1 .. j + 1, clamped) once -- 9 loads and 9 unpacks for 4 outputs instead of 16 -- and blends separably in
// packed fp32x2 (x first, then y).  Per output byte: 2.6x fewer instructions than the per-pixel kernel, which was issue-bound (437 us for
// the 96 x 96 level where a plain copy of the output tensor takes 230 us; tools/bench_upsample.py).
__device__ __forceinline__ uint64_t up_pk2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ uint64_t up_lerp2(uint64_t a, uint64_t b, uint64_t f) {      // a + f * (b - a)
  uint64_t d, r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(b), "l"(a));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(f), "l"(d), "l"(a));
  return r;
}
__global__ void __launch_bounds__(256) upsample2x_concat_kernel(const __nv_bfloat16* __restrict__ prev, int ph, int pw, int C1,
                                                                const __nv_bfloat16* __restrict__ skip, int C2,
                                                                __nv_bfloat16* __restrict__ out, int n_img) {
  const int H = 2 * ph, W = 2 * pw;
  const int Ct = C1 + C2, g8 = Ct / 8;
  const int xi = blockIdx.x * blockDim.x + threadIdx.x;
  if (xi >= pw * g8) return;
  const int j = xi / g8;                        // output columns 2j, 2j + 1
  const int c = (xi - j * g8) * 8;
  const int i = blockIdx.y;                     // output rows 2i, 2i + 1
  const long long img = blockIdx.z;
  __nv_bfloat16* o00 = out + ((img * H + 2 * i) * W + 2 * j) * Ct + c;
  const long long orow = static_cast<long long>(W) * Ct;
  if (c >= C1) {
    const __nv_bfloat16* s00 = skip + ((img * H + 2 * i) * W + 2 * j) * C2 + (c - C1);
    const long long srow = static_cast<long long>(W) * C2;
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(s00)), b = __ldg(reinterpret_cast<const uint4*>(s00 + C2));
    const uint4 cc = __ldg(reinterpret_cast<const uint4*>(s00 + srow)), d = __ldg(reinterpret_cast<const uint4*>(s00 + srow + C2));
    *reinterpret_cast<uint4*>(o00) = a;
    *reinterpret_cast<uint4*>(o00 + Ct) = b;
    *reinterpret_cast<uint4*>(o00 + orow) = cc;
    *reinterpret_cast<uint4*>(o00 + orow + Ct) = d;
    return;
  }
  // fractions relative to the fixed tap pairs (j - 1, j) / (j, j + 1): clamped, so a source coordinate that rounds across an integer
  // still gives the same value
  const float sx = static_cast<float>(pw - 1) / static_cast<float>(W - 1), sy = static_cast<float>(ph - 1) / static_cast<float>(H - 1);
  const float fxa = fminf(fmaxf(static_cast<float>(2 * j) * sx - static_cast<float>(j - 1), 0.f), 1.f);
  const float fxb = fminf(fmaxf(static_cast<float>(2 * j + 1) * sx - static_cast<float>(j), 0.f), 1.f);
  const float fya = fminf(fmaxf(static_cast<float>(2 * i) * sy - static_cast<float>(i - 1), 0.f), 1.f);
  const float fyb = fminf(fmaxf(static_cast<float>(2 * i + 1) * sy - static_cast<float>(i), 0.f), 1.f);
  const int xs[3] = {max(j - 1, 0), j, min(j + 1, pw - 1)};
  const int ys[3] = {max(i - 1, 0), i, min(i + 1, ph - 1)};
  const __nv_bfloat16* pbase = prev + img * ph * pw * C1 + c;
  uint4 t[3][3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int q = 0; q < 3; ++q) t[r][q] = __ldg(reinterpret_cast<const uint4*>(pbase + (static_cast<long long>(ys[r]) * pw + xs[q]) * C1));
  const uint64_t FXA = up_pk2(fxa, fxa), FXB = up_pk2(fxb, fxb), FYA = up_pk2(fya, fya), FYB = up_pk2(fyb, fyb);
  uint32_t oaa[4], oab[4], oba[4], obb[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {               // channel pair k of the 8
    uint64_t xa[3], xb[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const uint32_t w0 = reinterpret_cast<const uint32_t*>(&t[r][0])[k], w1 = reinterpret_cast<const uint32_t*>(&t[r][1])[k],
                     w2 = reinterpret_cast<const uint32_t*>(&t[r][2])[k];
      const uint64_t v0 = up_pk2(__uint_as_float(w0 << 16), __uint_as_float(w0 & 0xffff0000u));
      const uint64_t v1 = up_pk2(__uint_as_float(w1 << 16), __uint_as_float(w1 & 0xffff0000u));
      const uint64_t v2 = up_pk2(__uint_as_float(w2 << 16), __uint_as_float(w2 & 0xffff0000u));
      xa[r] = up_lerp2(v0, v1, FXA);
      xb[r] = up_lerp2(v1, v2, FXB);
    }
    const uint64_t raa = up_lerp2(xa[0], xa[1], FYA), rab = up_lerp2(xb[0], xb[1], FYA);
    const uint64_t rba = up_lerp2(xa[1], xa[2], FYB), rbb = up_lerp2(xb[1], xb[2], FYB);
    float lo, hi;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(raa)); oaa[k] = pack_bf16x2(lo, hi);
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(rab)); oab[k] = pack_bf16x2(lo, hi);
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(rba)); oba[k] = pack_bf16x2(lo, hi);
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(rbb)); obb[k] = pack_bf16x2(lo, hi);
  }
  *reinterpret_cast<uint4*>(o00) = make_uint4(oaa[0], oaa[1], oaa[2], oaa[3]);
  *reinterpret_cast<uint4*>(o00 + Ct) = make_uint4(oab[0], oab[1], oab[2], oab[3]);
  *reinterpret_cast<uint4*>(o00 + orow) = make_uint4(oba[0], oba[1], oba[2], oba[3]);
  *reinterpret_cast<uint4*>(o00 + orow + Ct) = make_uint4(obb[0], obb[1], obb[2], obb[3]);
}

int upsample_concat_dispatch(const __nv_bfloat16* prev, int ph, int pw, int C1, const __nv_bfloat16* skip, int C2,
                             __nv_bfloat16* out, int n_img, int H, int W, cudaStream_t st) {
  // C2 == 0 (skip may be NULL): plain bilinear upsample -- the nn.Upsample(x2) steps of ProgressiveDecoding (lib/vlt.py:437-452)
  LAVT_REQUIRE(C1 % 8 == 0 && C2 % 8 == 0 && C1 > 0 && C2 >= 0 && (C2 == 0 || skip != nullptr), "upsample_concat: channels must be multiples of 8");
  LAVT_REQUIRE(ph <= H && pw <= W && ph > 0 && pw > 0, "upsample_concat: prev (%dx%d) larger than skip (%dx%d)", ph, pw, H, W);
  LAVT_REQUIRE(n_img > 0 && n_img < 65536 && H > 0 && H < 65536 && W > 0, "upsample_concat: empty or too large input");
  if (H == 2 * ph && W == 2 * pw && ph >= 2 && pw >= 2) {
    const int per_row = pw * ((C1 + C2) / 8);
    upsample2x_concat_kernel<<<dim3((per_row + 255) / 256, ph, n_img), 256, 0, st>>>(prev, ph, pw, C1, skip, C2, out, n_img);
    LAVT_LAUNCH_CHECK("upsample2x_concat_kernel");
    return LAVT_OK;
  }
  const int per_row = W * ((C1 + C2) / 8);
  upsample_concat_kernel<<<dim3((per_row + 255) / 256, H, n_img), 256, 0, st>>>(prev, ph, pw, C1, skip, C2, out, n_img, H, W);
  LAVT_LAUNCH_CHECK("upsample_concat_kernel");
  return LAVT_OK;
}

// ---- conv3x3 of a bilinear upsample, evaluated on the coarse grid ----
// conv3x3(up(Y))[p] = sum_tap [p + tap inside H x W] sum_corner beta(p + tap, corner) * Z[corner, tap], Z = W_tap . Y (one GEMM on the
// coarse map).  The blend below finishes a decoder conv+BN+ReLU: out = ReLU(addend + s * that sum), addend = the skip half of the conv
// with the BN folded in (P, fp32) or, without a skip, the folded BN shift b.
__device__ __forceinline__ void blend_epilogue(const float* acc, const float* __restrict__ P, const float* __restrict__ s,
                                               const float* __restrict__ b, long long pix, int hid, int c, __nv_bfloat16* __restrict__ out) {
  const float4 s0 = __ldg(reinterpret_cast<const float4*>(s + c)), s1 = __ldg(reinterpret_cast<const float4*>(s + c + 4));
  const float* add = P ? P + pix * hid + c : b + c;
  const float4 a0 = __ldg(reinterpret_cast<const float4*>(add)), a1 = __ldg(reinterpret_cast<const float4*>(add + 4));
  const float sv[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w}, av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
  uint32_t o[4];
#pragma unroll
  for (int k = 0; k < 4; ++k)
    o[k] = pack_bf16x2(fmaxf(fmaf(sv[2 * k], acc[2 * k], av[2 * k]), 0.f), fmaxf(fmaf(sv[2 * k + 1], acc[2 * k + 1], av[2 * k + 1]), 0.f));
  *reinterpret_cast<uint4*>(out + pix * hid + c) = make_uint4(o[0], o[1], o[2], o[3]);
}

// any (h, w) -> (H, W): thread per (fine pixel, 8 channels), the 9 x 4 (tap, corner) terms read straight from Z
__global__ void __launch_bounds__(256) upconv_blend_kernel(const __nv_bfloat16* __restrict__ Z, int h, int w, int hid,
                                                           const float* __restrict__ P, const float* __restrict__ s,
                                                           const float* __restrict__ b, __nv_bfloat16* __restrict__ out, int H, int W) {
  const int g8 = hid / 8;
  const int xi = blockIdx.x * blockDim.x + threadIdx.x;
  if (xi >= W * g8) return;
  const int x = xi / g8;
  const int c = (xi - x * g8) * 8;
  const int y = blockIdx.y;
  const long long img = blockIdx.z;
  const long long ldz = 9LL * hid;
  const __nv_bfloat16* zimg = Z + img * h * w * ldz + c;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int ky = 0; ky < 3; ++ky) {
    const int qy = y + ky - 1;
    if (qy < 0 || qy >= H) continue;              // zero padding of the fine image
    int y0, y1;
    float fy;
    bilinear_taps(qy, h, H, y0, y1, fy);
    for (int kx = 0; kx < 3; ++kx) {
      const int qx = x + kx - 1;
      if (qx < 0 || qx >= W) continue;
      int x0, x1;
      float fx;
      bilinear_taps(qx, w, W, x0, x1, fx);
      const float w00 = (1.f - fy) * (1.f - fx), w01 = (1.f - fy) * fx, w10 = fy * (1.f - fx), w11 = fy * fx;
      const __nv_bfloat16* zt = zimg + (ky * 3 + kx) * hid;
      const uint4 a = __ldg(reinterpret_cast<const uint4*>(zt + (static_cast<long long>(y0) * w + x0) * ldz));
      const uint4 bq = __ldg(reinterpret_cast<const uint4*>(zt + (static_cast<long long>(y0) * w + x1) * ldz));
      const uint4 cc = __ldg(reinterpret_cast<const uint4*>(zt + (static_cast<long long>(y1) * w + x0) * ldz));
      const uint4 d = __ldg(reinterpret_cast<const uint4*>(zt + (static_cast<long long>(y1) * w + x1) * ldz));
      const uint32_t ua[4] = {a.x, a.y, a.z, a.w}, ub[4] = {bq.x, bq.y, bq.z, bq.w}, uc[4] = {cc.x, cc.y, cc.z, cc.w},
                     ud[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 fa = unpack_bf16x2(ua[j]), fb = unpack_bf16x2(ub[j]), fc = unpack_bf16x2(uc[j]), fd = unpack_bf16x2(ud[j]);
        acc[2 * j] += w00 * fa.x + w01 * fb.x + w10 * fc.x + w11 * fd.x;
        acc[2 * j + 1] += w00 * fa.y + w01 * fb.y + w10 * fc.y + w11 * fd.y;
      }
    }
  }
  blend_epilogue(acc, P, s, b, (img * H + y) * W + x, hid, c, out);
}

// Exact x2 (H == 2h, W == 2w: every SimpleDecoding level).  A block stages the Z rows of a UB_TI x UB_TJ coarse tile plus a one-pixel
// border (all 9 taps, UB_CC channels) in shared memory; a thread owns the 2 x 2 fine pixels above coarse pixel (i, j) for 8 channels.
// Their 9 taps x 4 corners touch 7 x 7 of the 9 x 9 (window pixel, tap) entries of the 3 x 3 window (i-1 .. i+1, j-1 .. j+1): 49 shared
// loads for 4 outputs instead of 144.  Fine row q = 2i - 1 + u (u = 0..3) interpolates window rows (0, 1) for u < 2 and (1, 2) otherwise;
// its fraction is taken against that fixed pair and clamped, as in upsample2x_concat_kernel, so the clamped window at the map border
// (weight 0 or an identical row) gives the same value.  Accumulation in packed fp32x2.
constexpr int UB_TI = 4, UB_TJ = 8, UB_CC = 32;
constexpr int UB_THREADS = UB_TI * UB_TJ * (UB_CC / 8);
constexpr int UB_G = UB_CC / 8;
static_assert(UB_G == 4, "the addend prefetch gives each of a coarse pixel's 4 channel groups one of its 4 fine pixels");
__global__ void __launch_bounds__(UB_THREADS) upconv2x_blend_kernel(const __nv_bfloat16* __restrict__ Z, int h, int w, int hid,
                                                                    const float* __restrict__ P, const float* __restrict__ s,
                                                                    const float* __restrict__ b, __nv_bfloat16* __restrict__ out) {
  __shared__ uint4 zs[(UB_TI + 2) * (UB_TJ + 2) * 9 * UB_G];        // [window row][window col][tap][8-channel group]
  const int H = 2 * h, W = 2 * w;
  const int cgroups = hid / UB_CC;
  const int jt = blockIdx.x / cgroups;
  const int c0 = (blockIdx.x - jt * cgroups) * UB_CC;
  const int i0 = blockIdx.y * UB_TI, j0 = jt * UB_TJ;
  const long long img = blockIdx.z;
  const long long ldz = 9LL * hid;
  const __nv_bfloat16* zimg = Z + img * h * w * ldz + c0;
  const int g = threadIdx.x % UB_G, tj = (threadIdx.x / UB_G) % UB_TJ, ti = threadIdx.x / (UB_G * UB_TJ);
  const int i = i0 + ti, j = j0 + tj;
  // the UB_G threads of a coarse pixel read its 4 fine pixels' addend rows (UB_CC fp32 = one 128-byte line each) in the epilogue:
  // start pulling them into L2 now, so that those loads do not wait on HBM after the blend
  if (P != nullptr && i < h && j < w)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(P + ((img * H + 2 * i + (g >> 1)) * W + 2 * j + (g & 1)) * hid + c0));
  // asynchronous copies: every thread has all of its staging loads in flight at once
  for (int e = threadIdx.x; e < (UB_TI + 2) * (UB_TJ + 2) * 9 * UB_G; e += UB_THREADS) {
    const int ge = e % UB_G;
    int r = e / UB_G;
    const int tap = r % 9;
    r /= 9;
    const int wc = r % (UB_TJ + 2), wr = r / (UB_TJ + 2);
    const int ci = min(max(i0 - 1 + wr, 0), h - 1), cj = min(max(j0 - 1 + wc, 0), w - 1);
    cp_async_16(&zs[e], zimg + (static_cast<long long>(ci) * w + cj) * ldz + tap * hid + ge * 8, true);
  }
  cp_async_commit();
  cp_async_wait<0>();
  __syncthreads();
  if (i >= h || j >= w) return;
  const float sy = (H > 1) ? static_cast<float>(h - 1) / static_cast<float>(H - 1) : 0.f;
  const float sx = (W > 1) ? static_cast<float>(w - 1) / static_cast<float>(W - 1) : 0.f;
  float ylo[4], yhi[4], xlo[4], xhi[4];         // weights of the lower / upper row (column) of the pair; 0 outside the fine image
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int qy = 2 * i - 1 + u, qx = 2 * j - 1 + u;
    const float fy = fminf(fmaxf(static_cast<float>(qy) * sy - static_cast<float>(u < 2 ? i - 1 : i), 0.f), 1.f);
    const float fx = fminf(fmaxf(static_cast<float>(qx) * sx - static_cast<float>(u < 2 ? j - 1 : j), 0.f), 1.f);
    const bool vy = qy >= 0 && qy < H, vx = qx >= 0 && qx < W;
    ylo[u] = vy ? 1.f - fy : 0.f;
    yhi[u] = vy ? fy : 0.f;
    xlo[u] = vx ? 1.f - fx : 0.f;
    xhi[u] = vx ? fx : 0.f;
  }
  uint64_t acc[4][4];                           // [fine pixel a * 2 + b][channel pair]
#pragma unroll
  for (int o = 0; o < 4; ++o)
#pragma unroll
    for (int k = 0; k < 4; ++k) acc[o][k] = 0;
  const uint4* zb = zs + (ti * (UB_TJ + 2) + tj) * 9 * UB_G + g;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
      for (int wr = 0; wr < 3; ++wr)
#pragma unroll
        for (int wc = 0; wc < 3; ++wc) {
          // window rows used by this tap: ky + a for a in {0, 1}, pair base (ky + a >= 2)
          if (wr < (ky >= 2 ? 1 : 0) || wr > (ky >= 1 ? 2 : 1) || wc < (kx >= 2 ? 1 : 0) || wc > (kx >= 1 ? 2 : 1)) continue;
          const uint4 v = zb[((wr * (UB_TJ + 2) + wc) * 9 + ky * 3 + kx) * UB_G];
          const uint32_t uv[4] = {v.x, v.y, v.z, v.w};
          uint64_t f[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) f[k] = up_pk2(__uint_as_float(uv[k] << 16), __uint_as_float(uv[k] & 0xffff0000u));
#pragma unroll
          for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int bb = 0; bb < 2; ++bb) {
              const int u = ky + a, x = kx + bb, rb = u >= 2 ? 1 : 0, cb = x >= 2 ? 1 : 0;
              if (wr != rb && wr != rb + 1) continue;
              if (wc != cb && wc != cb + 1) continue;
              const float wt = (wr == rb ? ylo[u] : yhi[u]) * (wc == cb ? xlo[x] : xhi[x]);
              const uint64_t W2 = up_pk2(wt, wt);
#pragma unroll
              for (int k = 0; k < 4; ++k) asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc[a * 2 + bb][k]) : "l"(W2), "l"(f[k]));
            }
        }
  const int c = c0 + g * 8;
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int bb = 0; bb < 2; ++bb) {
      float av[8];
#pragma unroll
      for (int k = 0; k < 4; ++k) asm("mov.b64 {%0, %1}, %2;" : "=f"(av[2 * k]), "=f"(av[2 * k + 1]) : "l"(acc[a * 2 + bb][k]));
      blend_epilogue(av, P, s, b, (img * H + 2 * i + a) * W + 2 * j + bb, hid, c, out);
    }
}

int upconv_blend_dispatch(const __nv_bfloat16* Z, int h, int w, int hid, const float* P, const float* s, const float* b,
                          __nv_bfloat16* out, int n_img, int H, int W, cudaStream_t st) {
  LAVT_REQUIRE(hid % 8 == 0 && hid > 0 && s != nullptr && (P != nullptr || b != nullptr), "upconv_blend: hid must be a multiple of 8; s and P or b required");
  LAVT_REQUIRE(h <= H && w <= W && h > 0 && w > 0, "upconv_blend: coarse map (%dx%d) larger than the output (%dx%d)", h, w, H, W);
  LAVT_REQUIRE(n_img > 0 && n_img < 65536 && H > 0 && H < 65536 && W > 0, "upconv_blend: empty or too large input");
  if (H == 2 * h && W == 2 * w && hid % UB_CC == 0) {
    const long long gx = static_cast<long long>((w + UB_TJ - 1) / UB_TJ) * (hid / UB_CC);
    LAVT_REQUIRE(gx < (1LL << 31), "upconv_blend: map too wide");
    upconv2x_blend_kernel<<<dim3(static_cast<unsigned>(gx), (h + UB_TI - 1) / UB_TI, n_img), UB_THREADS, 0, st>>>(Z, h, w, hid, P, s, b, out);
    LAVT_LAUNCH_CHECK("upconv2x_blend_kernel");
    return LAVT_OK;
  }
  const int per_row = W * (hid / 8);
  upconv_blend_kernel<<<dim3((per_row + 255) / 256, H, n_img), 256, 0, st>>>(Z, h, w, hid, P, s, b, out, H, W);
  LAVT_LAUNCH_CHECK("upconv_blend_kernel");
  return LAVT_OK;
}

// 8 lanes per pixel (4 pixels per warp): logits[pix, o] = sum_c y[pix, c] * w[o, c] + b[o], o in {0, 1}; w staged in smem
__global__ void __launch_bounds__(256) conv1x1_logits_kernel(const __nv_bfloat16* __restrict__ y, const float* __restrict__ w,
                                                             const float* __restrict__ b, float* __restrict__ out, long long npix,
                                                             int C) {
  extern __shared__ float sw[];   // [2][C]
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) sw[i] = w[i];
  __syncthreads();
  const int sub = threadIdx.x & 7;
  const long long pix = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 3;
  const bool live = pix < npix;
  float a0 = 0.f, a1 = 0.f;
  if (live) {
    const __nv_bfloat16* row = y + pix * C;
    for (int c = sub * 8; c < C; c += 64) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(row + c));
      const uint32_t uu[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack_bf16x2(uu[j]);
        a0 = fmaf(f.x, sw[c + 2 * j], fmaf(f.y, sw[c + 2 * j + 1], a0));
        a1 = fmaf(f.x, sw[C + c + 2 * j], fmaf(f.y, sw[C + c + 2 * j + 1], a1));
      }
    }
  }
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) {
    a0 += __shfl_xor_sync(0xffffffffu, a0, o);
    a1 += __shfl_xor_sync(0xffffffffu, a1, o);
  }
  if (live && sub == 0) *reinterpret_cast<float2*>(out + pix * 2) = make_float2(a0 + b[0], a1 + b[1]);
}

int conv1x1_logits_dispatch(const __nv_bfloat16* y, const float* w, const float* b, float* out, long long npix, int C,
                            cudaStream_t st) {
  LAVT_REQUIRE(npix > 0 && C % 8 == 0 && C <= 4096, "conv1x1: bad shape");
  const long long threads = npix * 8;
  conv1x1_logits_kernel<<<static_cast<unsigned>((threads + 255) / 256), 256, 2 * C * sizeof(float), st>>>(y, w, b, out, npix, C);
  LAVT_LAUNCH_CHECK("conv1x1_logits_kernel");
  return LAVT_OK;
}

// thread per output pixel (both classes); writes NCHW
__global__ void __launch_bounds__(256) upsample_logits_kernel(const float* __restrict__ in, float* __restrict__ out, int n_img,
                                                              int h, int w, int H, int W) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(n_img) * H * W;
  if (idx >= total) return;
  const int x = static_cast<int>(idx % W), y = static_cast<int>((idx / W) % H);
  const long long img = idx / (static_cast<long long>(W) * H);
  int y0, y1, x0, x1; float fy, fx;
  bilinear_taps(y, h, H, y0, y1, fy);
  bilinear_taps(x, w, W, x0, x1, fx);
  const float2* base = reinterpret_cast<const float2*>(in) + img * h * w;
  const float2 a = __ldg(base + y0 * w + x0), b = __ldg(base + y0 * w + x1), c = __ldg(base + y1 * w + x0),
               d = __ldg(base + y1 * w + x1);
  const float w00 = (1.f - fy) * (1.f - fx), w01 = (1.f - fy) * fx, w10 = fy * (1.f - fx), w11 = fy * fx;
  const long long plane = static_cast<long long>(H) * W;
  float* o = out + img * 2 * plane + static_cast<long long>(y) * W + x;
  o[0] = w00 * a.x + w01 * b.x + w10 * c.x + w11 * d.x;
  o[plane] = w00 * a.y + w01 * b.y + w10 * c.y + w11 * d.y;
}

// four consecutive output pixels of a row per thread (W % 4 == 0): the row taps are shared and each class is written with one 16-byte store
// (one 4-byte store per pixel and class ran at 1.1 TB/s: 74 us for the 75 MB of full-resolution logits of 8 clips)
__global__ void __launch_bounds__(256) upsample_logits4_kernel(const float* __restrict__ in, float* __restrict__ out, int n_img,
                                                               int h, int w, int H, int W) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int W4 = W >> 2;
  const long long total = static_cast<long long>(n_img) * H * W4;
  if (idx >= total) return;
  const int x4 = static_cast<int>(idx % W4) * 4, y = static_cast<int>((idx / W4) % H);
  const long long img = idx / (static_cast<long long>(W4) * H);
  int y0, y1; float fy;
  bilinear_taps(y, h, H, y0, y1, fy);
  const float2* r0 = reinterpret_cast<const float2*>(in) + (img * h + y0) * w;
  const float2* r1 = reinterpret_cast<const float2*>(in) + (img * h + y1) * w;
  float o0[4], o1[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    int x0, x1; float fx;
    bilinear_taps(x4 + k, w, W, x0, x1, fx);
    const float2 a = __ldg(r0 + x0), b = __ldg(r0 + x1), c = __ldg(r1 + x0), d = __ldg(r1 + x1);
    const float w00 = (1.f - fy) * (1.f - fx), w01 = (1.f - fy) * fx, w10 = fy * (1.f - fx), w11 = fy * fx;
    o0[k] = w00 * a.x + w01 * b.x + w10 * c.x + w11 * d.x;
    o1[k] = w00 * a.y + w01 * b.y + w10 * c.y + w11 * d.y;
  }
  const long long plane = static_cast<long long>(H) * W;
  float* o = out + img * 2 * plane + static_cast<long long>(y) * W + x4;
  *reinterpret_cast<float4*>(o) = make_float4(o0[0], o0[1], o0[2], o0[3]);
  *reinterpret_cast<float4*>(o + plane) = make_float4(o1[0], o1[1], o1[2], o1[3]);
}

int upsample_logits_dispatch(const float* in, float* out, int n_img, int h, int w, int H, int W, cudaStream_t st) {
  const long long total = static_cast<long long>(n_img) * H * W;
  LAVT_REQUIRE(total > 0 && h > 0 && w > 0, "upsample_logits: empty input");
  if (W % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    upsample_logits4_kernel<<<static_cast<unsigned>((total / 4 + 255) / 256), 256, 0, st>>>(in, out, n_img, h, w, H, W);
    LAVT_LAUNCH_CHECK("upsample_logits4_kernel");
    return LAVT_OK;
  }
  upsample_logits_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(in, out, n_img, h, w, H, W);
  LAVT_LAUNCH_CHECK("upsample_logits_kernel");
  return LAVT_OK;
}

// (n, P, C) fp32 -> (n, C, P) fp32, 32x32 smem tiles.  grid (ceil(P/32), ceil(C/32), n), block (32, 8)
__global__ void nhwc_to_nchw_kernel(const float* __restrict__ in, float* __restrict__ out, int P, int C) {
  __shared__ float tile[32][33];
  const long long img = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int p = p0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (p < P && c < C) ? in[(img * P + p) * C + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i, p = p0 + threadIdx.x;
    if (p < P && c < C) out[(img * C + c) * P + p] = tile[threadIdx.x][i];
  }
}

int nhwc_to_nchw_dispatch(const float* in, float* out, int n_img, int P, int C, cudaStream_t st) {
  LAVT_REQUIRE(n_img > 0 && P > 0 && C > 0 && n_img < 65536, "nhwc_to_nchw: bad shape");
  nhwc_to_nchw_kernel<<<dim3((P + 31) / 32, (C + 31) / 32, n_img), dim3(32, 8), 0, st>>>(in, out, P, C);
  LAVT_LAUNCH_CHECK("nhwc_to_nchw_kernel");
  return LAVT_OK;
}

// (n, C, P) fp32 -> (n, P, C) bf16
__global__ void nchw_to_nhwc_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, int P, int C) {
  __shared__ float tile[32][33];
  const long long img = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i, p = p0 + threadIdx.x;
    tile[i][threadIdx.x] = (p < P && c < C) ? in[(img * C + c) * P + p] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int p = p0 + i, c = c0 + threadIdx.x;
    if (p < P && c < C) out[(img * P + p) * C + c] = __float2bfloat16(tile[threadIdx.x][i]);
  }
}

int nchw_to_nhwc_bf16_dispatch(const float* in, __nv_bfloat16* out, int n_img, int P, int C, cudaStream_t st) {
  LAVT_REQUIRE(n_img > 0 && P > 0 && C > 0 && n_img < 65536, "nchw_to_nhwc: bad shape");
  nchw_to_nhwc_bf16_kernel<<<dim3((P + 31) / 32, (C + 31) / 32, n_img), dim3(32, 8), 0, st>>>(in, out, P, C);
  LAVT_LAUNCH_CHECK("nchw_to_nhwc_bf16_kernel");
  return LAVT_OK;
}

}  // namespace lavt
