// Shifted-window attention forward: the one dispatch decision (window_attn_choose) and the mma.sync fallback for the
// windows that neither tcgen05 kernel takes.  window_attn_dispatch sends every window of 16+ tokens to attn_tc3.cu (full
// 7 x 7 / 12 x 12 windows) or attn_tc2.cu (every other window of up to 1152 tokens); what is left are clamped windows of
// fewer than 16 tokens (e.g. stage 3 of a 32 px clip), too small for a 128-row tcgen05 tile to be worth it.
//
// Fallback (reference WindowAttention3D.forward, lib/video_swin_transformer.py:147-165; 2-D twin lib/backbone.py:127-138):
// per (window, head)
//     S = q k^T  (+ relative-position bias, + shifted-window mask)  ->  softmax  ->  O = P v
// computed flash-style: the N x N score matrix never leaves registers.  q arrives pre-scaled by
// head_dim^-0.5 * log2(e) (folded into the qkv GEMM epilogue) so the softmax runs in base 2 with one FADD + one
// MUFU.EX2 per score.  The bias is gathered from the per-head table column held in shared memory (pre-multiplied by
// log2 e) through the closed form  idx(i,j) = code(i) - code(j) + const ; the -100 mask comes from per-token region
// ids (geom.cuh) and is skipped entirely for windows that do not straddle the cyclic-shift seam -- neither the (N,N)
// index buffer nor the (nW,N,N) mask tensor exists on the device.
// mma.sync.m16n8k16 (bf16 -> fp32), window_attn_resident_kernel: one CTA per (window, head) keeps the whole K and V of
// the head in shared memory (loaded once with cp.async); a single warp walks the one 16-row query strip against one
// key tile of 48.  It writes no row statistics (lse), so a training forward of such a window recomputes them in the backward.
#include "kernels.cuh"

#include <cstdlib>
#include <cstring>

namespace lavt {

constexpr int AT_HD = 32;        // head dim
constexpr float AT_LOG2E = 1.4426950408889634f;
constexpr float AT_MASKV = -100.0f * AT_LOG2E;

// 16-byte chunk swizzle inside a 64-byte row so that ldmatrix (8 rows x 16 B) is bank-conflict free
__device__ __forceinline__ int kv_off(int row, int chunk) { return row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4); }

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct RowState {
  float o[4][4];
  float m0, m1, l0, l1;
};

// One K/V tile (KVT keys at smem kt / vt, first key index kv0) against this warp's 16 query rows.
template <int KVT>
__device__ __forceinline__ void attn_tile(const uint8_t* kt, const uint8_t* vt, int kv0, int N, int Npad, const uint16_t* codes,
                                          const uint8_t* rids, const float* tq0, const float* tq1, int rq0, int rq1,
                                          bool need_mask, const uint32_t (&qf)[2][4], RowState& st, int lane) {
  constexpr int NT = KVT / 8;       // n8 tiles
  constexpr int KS = KVT / 16;      // k16 steps
  const int t = lane & 3;
  // accumulators start from the relative-position bias: S = bias + q k^T
  float s[NT][4];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    const int key = kv0 + nt * 8 + 2 * t;          // even; codes[] is zero-padded to a multiple of 8 past N
    const int kc = min(key, Npad - 2);
    const uint32_t cc = *reinterpret_cast<const uint32_t*>(codes + kc);
    const int c0 = cc & 0xffff, c1 = cc >> 16;
    s[nt][0] = tq0[-c0];
    s[nt][1] = tq0[-c1];
    s[nt][2] = tq1[-c0];
    s[nt][3] = tq1[-c1];
  }
  if (need_mask) {
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int key = kv0 + nt * 8 + 2 * t;
      const int kc = min(key, Npad - 2);
      const uint32_t rr = *reinterpret_cast<const uint16_t*>(rids + kc);
      const int r0 = rr & 0xff, r1 = rr >> 8;
      if (r0 != rq0) s[nt][0] += AT_MASKV;
      if (r1 != rq0) s[nt][1] += AT_MASKV;
      if (r0 != rq1) s[nt][2] += AT_MASKV;
      if (r1 != rq1) s[nt][3] += AT_MASKV;
    }
  }
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    uint32_t kf[4];
    ldmatrix_x4(kf, kt + kv_off(nt * 8 + (lane & 7), lane >> 3));
    mma_bf16_16816(s[nt], qf[0], kf[0], kf[1]);
    mma_bf16_16816(s[nt], qf[1], kf[2], kf[3]);
  }
  if (kv0 + KVT > N) {          // only the last tile can contain padded keys
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        if (kv0 + nt * 8 + 2 * t + e >= N) {
          s[nt][e] = -INFINITY;
          s[nt][2 + e] = -INFINITY;
        }
      }
    }
  }
  float mx0 = s[0][0], mx1 = s[0][2];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
    mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
  }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  const float nm0 = fmaxf(st.m0, mx0), nm1 = fmaxf(st.m1, mx1);
  const float c0 = ex2f(st.m0 - nm0), c1 = ex2f(st.m1 - nm1);
  st.m0 = nm0;
  st.m1 = nm1;
  float rs0 = 0.f, rs1 = 0.f;
  uint32_t pf[KS][4];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    const float p0 = ex2f(s[nt][0] - nm0), p1 = ex2f(s[nt][1] - nm0);
    const float p2 = ex2f(s[nt][2] - nm1), p3 = ex2f(s[nt][3] - nm1);
    rs0 += p0 + p1;
    rs1 += p2 + p3;
    pf[nt >> 1][(nt & 1) * 2 + 0] = pack_bf16x2(p0, p1);
    pf[nt >> 1][(nt & 1) * 2 + 1] = pack_bf16x2(p2, p3);
  }
  st.l0 = st.l0 * c0 + rs0;
  st.l1 = st.l1 * c1 + rs1;
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
    st.o[dt][0] *= c0; st.o[dt][1] *= c0; st.o[dt][2] *= c1; st.o[dt][3] *= c1;
  }
#pragma unroll
  for (int kk = 0; kk < KS; ++kk) {       // 16 keys per step
#pragma unroll
    for (int dp = 0; dp < 2; ++dp) {      // two d-chunks (8 each) per ldmatrix.x4
      uint32_t vf[4];
      ldmatrix_x4_trans(vf, vt + kv_off(kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, dp * 2 + (lane >> 4)));
      mma_bf16_16816(st.o[dp * 2 + 0], pf[kk], vf[0], vf[1]);
      mma_bf16_16816(st.o[dp * 2 + 1], pf[kk], vf[2], vf[3]);
    }
  }
}

__device__ __forceinline__ void load_q_frags(uint32_t (&qf)[2][4], const __nv_bfloat16* qbase, int ld, int qc0, int qc1, int t) {
  const __nv_bfloat16* r0p = qbase + static_cast<long long>(qc0) * ld;
  const __nv_bfloat16* r1p = qbase + static_cast<long long>(qc1) * ld;
#pragma unroll
  for (int ksb = 0; ksb < 2; ++ksb) {
    qf[ksb][0] = __ldg(reinterpret_cast<const uint32_t*>(r0p + ksb * 16 + 2 * t));
    qf[ksb][1] = __ldg(reinterpret_cast<const uint32_t*>(r1p + ksb * 16 + 2 * t));
    qf[ksb][2] = __ldg(reinterpret_cast<const uint32_t*>(r0p + ksb * 16 + 8 + 2 * t));
    qf[ksb][3] = __ldg(reinterpret_cast<const uint32_t*>(r1p + ksb * 16 + 8 + 2 * t));
  }
}

__device__ __forceinline__ void store_rows(const RowState& st, __nv_bfloat16* ob, int C, int qr0, int qr1, int N, int t) {
  float l0 = st.l0, l1 = st.l1;
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.0f / l0, i1 = 1.0f / l1;
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
    if (qr0 < N)
      *reinterpret_cast<uint32_t*>(ob + static_cast<long long>(qr0) * C + dt * 8 + 2 * t) = pack_bf16x2(st.o[dt][0] * i0, st.o[dt][1] * i0);
    if (qr1 < N)
      *reinterpret_cast<uint32_t*>(ob + static_cast<long long>(qr1) * C + dt * 8 + 2 * t) = pack_bf16x2(st.o[dt][2] * i1, st.o[dt][3] * i1);
  }
}

// Fills codes / rids / tab for one (window, head); returns (through *need_mask_smem) whether the window straddles the seam.
__device__ __forceinline__ void setup_window(const AttnParams& p, long long row0, int head, int N, int Npad, uint16_t* codes,
                                             uint8_t* rids, float* tab, int* need_mask_smem, bool shifted) {
  int differs = 0;
  int rid0 = 0;
  if (shifted) rid0 = win_token(p.win, row0).rid;
  for (int i = threadIdx.x; i < Npad; i += blockDim.x) {
    if (i < N) {
      const WinTok tk = win_token(p.win, row0 + i);
      codes[i] = static_cast<uint16_t>(tk.code);
      rids[i] = static_cast<uint8_t>(tk.rid);
      differs |= (tk.rid != rid0);
    } else {
      codes[i] = 0;
      rids[i] = 0;
    }
  }
  if (shifted && differs) *need_mask_smem = 1;     // benign race: every writer stores 1
  // table_t is [nH, L] (transposed on the host) so this read is coalesced
  const float* src = p.table_t + static_cast<long long>(head) * p.L;
  for (int i = threadIdx.x; i < p.L; i += blockDim.x) tab[i] = __ldg(src + i) * AT_LOG2E;
}

// ------------------------------------------------------------------------------------------------------------------
// resident K/V: grid (nH, windows), blockDim = 32 * warps
// ------------------------------------------------------------------------------------------------------------------
template <int KVT>
__global__ void __launch_bounds__(256, 2) window_attn_resident_kernel(const AttnParams p) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int N = p.win.N;
  const int Npad = (N + 7) & ~7;
  const int ntiles = (N + KVT - 1) / KVT;
  const int rows = ntiles * KVT;                                  // K/V rows in smem (zero beyond N)
  uint8_t* ks = smem;                                             // [rows][64 B]
  uint8_t* vs = ks + rows * 64;
  uint16_t* codes = reinterpret_cast<uint16_t*>(vs + rows * 64);
  uint8_t* rids = reinterpret_cast<uint8_t*>(codes + Npad);
  float* tab = reinterpret_cast<float*>(rids + Npad);
  __shared__ int s_need_mask;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int head = blockIdx.x;
  const long long row0 = static_cast<long long>(blockIdx.y) * N;
  const int ld = 3 * p.C;
  const __nv_bfloat16* qbase = p.qkv + row0 * ld + head * AT_HD;
  const __nv_bfloat16* kbase = qbase + p.C;
  const __nv_bfloat16* vbase = qbase + 2 * p.C;
  const bool shifted = (p.win.sd | p.win.sh | p.win.sw) != 0;

  if (threadIdx.x == 0) s_need_mask = 0;
  for (int i = threadIdx.x; i < 2 * rows * 4; i += blockDim.x) {
    const int isv = i >= rows * 4;
    const int j = isv ? i - rows * 4 : i;
    const int r = j >> 2, c = j & 3;
    const bool ok = r < N;
    const __nv_bfloat16* src = (isv ? vbase : kbase) + static_cast<long long>(ok ? r : 0) * ld + c * 8;
    cp_async_16((isv ? vs : ks) + kv_off(r, c), src, ok);
  }
  cp_async_commit();
  __syncthreads();
  setup_window(p, row0, head, N, Npad, codes, rids, tab, &s_need_mask, shifted);
  cp_async_wait<0>();
  __syncthreads();
  const bool need_mask = s_need_mask != 0;
  const int rc = rel_const(p.win);
  __nv_bfloat16* ob = p.out + row0 * p.C + head * AT_HD;

  const int nstrips = (N + 15) >> 4;
  for (int strip = warp; strip < nstrips; strip += nwarps) {
    const int qr0 = strip * 16 + g, qr1 = qr0 + 8;
    const int qc0 = min(qr0, N - 1), qc1 = min(qr1, N - 1);
    uint32_t qf[2][4];
    load_q_frags(qf, qbase, ld, qc0, qc1, t);
    const float* tq0 = tab + (static_cast<int>(codes[qc0]) + rc);    // bias(i, j) = tq[-code(j)]
    const float* tq1 = tab + (static_cast<int>(codes[qc1]) + rc);
    const int rq0 = rids[qc0], rq1 = rids[qc1];
    RowState st;
#pragma unroll
    for (int i = 0; i < 4; ++i) st.o[i][0] = st.o[i][1] = st.o[i][2] = st.o[i][3] = 0.f;
    st.m0 = st.m1 = -INFINITY;
    st.l0 = st.l1 = 0.f;
    for (int tile = 0; tile < ntiles; ++tile)
      attn_tile<KVT>(ks + tile * KVT * 64, vs + tile * KVT * 64, tile * KVT, N, Npad, codes, rids, tq0, tq1, rq0, rq1, need_mask,
                     qf, st, lane);
    store_rows(st, ob, p.C, qr0, qr1, N, t);
  }
}


// ------------------------------------------------------------------------------------------------------------------
// N < 16: one 16-row query strip, one warp, one key tile of 48
static int launch_resident(const AttnParams& p, long long nwin, cudaStream_t st) {
  constexpr int KVT = 48;
  const int N = p.win.N;
  const int Npad = (N + 7) & ~7;
  const int rows = ((N + KVT - 1) / KVT) * KVT;
  const size_t smem = 2 * static_cast<size_t>(rows) * 64 + static_cast<size_t>(Npad) * 3 + static_cast<size_t>(p.L) * 4 + 16;
  auto kfn = window_attn_resident_kernel<KVT>;
  static size_t configured = 0;
  if (smem > configured) {
    LAVT_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    configured = smem;
  }
  dim3 grid(p.nH, static_cast<unsigned>(nwin));
  kfn<<<grid, 32, smem, st>>>(p);
  LAVT_LAUNCH_CHECK("window_attn_resident_kernel");
  return LAVT_OK;
}

int attn_impl_setting(int set) {
  static int impl = -1;
  if (impl < 0) {
    const char* e = getenv("LAVT_ATTN_IMPL");      // A/B runs: "tc2" / "tc3"; anything else is auto
    impl = e && !strcmp(e, "tc2") ? 3 : e && !strcmp(e, "tc3") ? 4 : 0;
  }
  const int prev = impl;
  if (set >= 0) impl = set;
  return prev;
}

AttnKernel window_attn_choose(const AttnParams& p) {
  // tc3 is the faster kernel wherever it applies (stage 2 of the bench at N = 392: 203 vs 331 us, DESIGN 4.1); forcing tc2 is for A/B runs
  if (attn_impl_setting(-1) == 3 && window_attn_tc2_supported(p)) return AttnKernel::TC2;
  if (window_attn_tc3_supported(p)) return AttnKernel::TC3;
  if (window_attn_tc2_supported(p)) return AttnKernel::TC2;
  return AttnKernel::MMA;
}

int window_attn_dispatch(const AttnParams& p, cudaStream_t st) {
  const WinGeom& g = p.win;
  LAVT_REQUIRE(p.C == p.nH * AT_HD, "attention: head_dim must be 32 (C=%d, heads=%d)", p.C, p.nH);
  LAVT_REQUIRE(g.N == g.wd * g.wh * g.ww && g.N > 0, "attention: inconsistent window geometry");
  LAVT_REQUIRE(p.L == (2 * g.Wd - 1) * (2 * g.Wh - 1) * (2 * g.Ww - 1), "attention: bias table rows %d do not match window", p.L);
  LAVT_REQUIRE(p.L < 65536, "attention: bias table too large");
  LAVT_REQUIRE(g.N <= g.Wd * g.Wh * g.Ww, "attention: effective window larger than configured window");
  const long long nwin = 1LL * g.B * g.nwd * g.nwh * g.nww;
  LAVT_REQUIRE(nwin > 0 && nwin < 65536, "attention: window count %lld out of range", nwin);
  switch (window_attn_choose(p)) {
    case AttnKernel::TC3: return window_attn_tc3_dispatch(p, st);
    case AttnKernel::TC2: return window_attn_tc2_dispatch(p, st);
    case AttnKernel::MMA: break;
  }
  LAVT_REQUIRE(g.N < 16, "attention: no kernel takes a window of %d tokens (tcgen05: 16 ... 1152, mma.sync fallback: < 16)", g.N);
  LAVT_REQUIRE(p.lse == nullptr, "attention: row statistics (lse) are produced by the tcgen05 kernels only (N=%d)", g.N);
  return launch_resident(p, nwin, st);
}

}  // namespace lavt
