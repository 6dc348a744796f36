// tcgen05 / TMEM shifted-window attention core, second generation: every window size (N = 49 ... 1152 tokens), one pass over the scores.
// (reference WindowAttention3D.forward, lib/video_swin_transformer.py:147-165; 2-D twin lib/backbone.py:127-138)
//     S = q k^T + relative-position bias (+ shifted-window mask)  ->  softmax  ->  O = P v       per (window, head)
//
// What changed against the first generation (DESIGN.md 4.1: it kept the whole score row of <= 400 keys in TMEM and walked it twice):
//   * the KEY axis is cut into chunks of <= 112 columns that alternate between TWO softmax warpgroups; every warpgroup owns two
//     S buffers in TMEM, so the Q K^T of its next chunk is issued while it is still exponentiating the current one, and windows of
//     any size (8 x 12 x 12 = 1152 keys) fit: 2 groups x 2 buffers x 112 columns + 2 x 32 accumulator columns = 512
//   * ONE pass over S: a thread (= query row) takes the running maximum from the first piece it sees and keeps it while every later
//     piece satisfies  sum_j 2^(s_j - m) <= 2^20  (which bounds every p_j; bf16 / fp32 have the exponent range to spare).  Only when
//     a piece breaks that bound does the warp take the slow path: new maximum, rescale l, the P columns already written for the chunk
//     and -- after waiting for the previous P.V -- the O accumulator in TMEM.  No second TMEM read, no write-back of s + bias.
//   * per group the chunks of a tile accumulate into one O accumulator (online softmax); the two groups' partial (m, l, O) are merged
//     in the epilogue like flash-decoding splits
//   * K / V of a unit stay resident in shared memory (double-buffered across units when they fit), Q arrives per 128-row tile through
//     a 3-slot ring
// Warp roles: warps 0-7 softmax (group g = warp / 4, TMEM lane quadrant warp % 4; group 1 also runs the epilogue of the previous tile),
// warp 8 TMA producer, warps 9-10 tcgen05.mma issuers of group 0 / 1.
// q arrives pre-scaled by head_dim^-0.5 * log2(e) (qkv GEMM epilogue); the table is multiplied by log2(e) when it is staged.
#include "kernels.cuh"
#include "attn_tc_ptx.cuh"

#include <cstdio>
#include <cstdlib>

namespace lavt {

constexpr int T2_HD = 32;
constexpr int T2_G = 2;
constexpr int T2_SM_WARPS = 4 * T2_G;
constexpr int T2_SM_THREADS = 32 * T2_SM_WARPS;
constexpr int T2_TMA_WARP = T2_SM_WARPS;
constexpr int T2_MMA_WARP0 = T2_SM_WARPS + 1;
constexpr int T2_THREADS = 32 * (T2_MMA_WARP0 + T2_G);
constexpr int T2_EPI = T2_G - 1;            // the group that runs the epilogue
constexpr int T2_CW = 112;                  // S columns per buffer
constexpr int T2_O_COL = 2 * T2_G * T2_CW;  // 448: the two O accumulators live at columns 448..511
constexpr int T2_MAXCH = 16;
constexpr int T2_NQ = 3;                    // Q-tile ring slots
constexpr int T2_MAX_TAIL = 32;             // replicated tail tile: up to one lane quadrant of rows
constexpr float T2_LOG2E = 1.4426950408889634f;
constexpr float T2_MASKV = -100.0f * T2_LOG2E;
constexpr float T2_PSUM_LIMIT = 1048576.0f;  // 2^20

__host__ __device__ constexpr int t2_stride(int lo, int r) { return lo + ((r - lo) % 32 + 32) % 32; }

struct AttnTc2Args {
  int N, NP, ntiles;        // tokens per window, padded to 16, 128-row query tiles
  int nwin, units;
  int BR, nb;               // K / V TMA box rows, boxes per operand
  int nchunks, ngact;       // key chunks per tile; groups that own at least one chunk
  int cstart[T2_MAXCH], clen[T2_MAXCH];
  int SH, SD, L2, rc;       // bias-table strides in shared memory, size (floats), rel_const in that layout
  int nkv, kv_bytes;        // K|V stages and bytes per stage
  int off_q, off_tab, off_cf, off_negoff, off_pm, off_ps, off_xq, off_bar;
  int shifted;
  int r4, tail_rows;
  int mode;                 // 0 generic pieces, 1 runs of 7 keys (56-column pieces), 2 runs of 12 keys (48-column pieces)
};

// W consecutive columns as the fewest power-of-two transfers (any even W)
template <int W>
__device__ __forceinline__ void tmem_ld_n(uint32_t taddr, uint32_t* r) {
  if constexpr (W >= 32) { tmem_ld_x32(taddr, r); if constexpr (W > 32) tmem_ld_n<W - 32>(taddr + 32, r + 32); }
  else if constexpr (W >= 16) { tmem_ld_x16(taddr, r); if constexpr (W > 16) tmem_ld_n<W - 16>(taddr + 16, r + 16); }
  else if constexpr (W >= 8) { tmem_ld_x8(taddr, r); if constexpr (W > 8) tmem_ld_n<W - 8>(taddr + 8, r + 8); }
  else if constexpr (W >= 4) { tmem_ld_x4(taddr, r); if constexpr (W > 4) tmem_ld_n<W - 4>(taddr + 4, r + 4); }
  else { static_assert(W == 2, "unsupported TMEM transfer width"); tmem_ld_x2(taddr, r); }
}
template <int W>
__device__ __forceinline__ void tmem_st_n(uint32_t taddr, const uint32_t* r) {
  if constexpr (W >= 32) { tmem_st_x32(taddr, r); if constexpr (W > 32) tmem_st_n<W - 32>(taddr + 32, r + 32); }
  else if constexpr (W >= 16) { tmem_st_x16(taddr, r); if constexpr (W > 16) tmem_st_n<W - 16>(taddr + 16, r + 16); }
  else if constexpr (W >= 8) { tmem_st_x8(taddr, r); if constexpr (W > 8) tmem_st_n<W - 8>(taddr + 8, r + 8); }
  else if constexpr (W >= 4) { tmem_st_x4(taddr, r); if constexpr (W > 4) tmem_st_n<W - 4>(taddr + 4, r + 4); }
  else { static_assert(W == 2, "unsupported TMEM transfer width"); tmem_st_x2(taddr, r); }
}

// per-row state of the one-pass softmax
struct T2Row {
  const float* tabq;     // table + code(i) + rc : bias(i, j) = tabq[-code(j)]
  const int* negoff;     // generic pieces: -code(j) per key
  const int* runcode;    // run pieces: code(first key of the run) per run of Ww consecutive keys
  const float* cf;       // per-key region class of this window (floats), or nullptr when the window needs no mask
  float cif;             // region class of this row
  int N;
  float m, l;
  bool first;
};

// Softmax of one piece whose W scores s[] already hold q.k + bias: mask, padding, running maximum, exp2, row sum, bf16 P -> TMEM.
//   chunk column c (TMEM address ts_buf + c), global key index gc
//   o_acc / pv_done / pv_parity / tmem_o: the group's O accumulator already holds earlier chunks of this tile (slow path rescales it)
template <int W>
__device__ __forceinline__ void t2_mask_pad(float (&s)[W], int gc, const T2Row& r) {
  if (r.cf != nullptr) {
    float cfv[W];
#pragma unroll
    for (int j = 0; j < W; j += 4) *reinterpret_cast<float4*>(&cfv[j]) = *reinterpret_cast<const float4*>(r.cf + gc + j);
#pragma unroll
    for (int j = 0; j < W; ++j)
      if (cfv[j] != r.cif) s[j] += T2_MASKV;
  }
  if (gc + W > r.N) {
#pragma unroll
    for (int j = 0; j < W; ++j)
      if (gc + j >= r.N) s[j] = -INFINITY;
  }
}

template <int W>
__device__ __forceinline__ void t2_exp_store(float (&s)[W], uint32_t ts_buf, int c, T2Row& r, bool o_acc, uint64_t* pv_done,
                                             uint32_t pv_parity, uint32_t tmem_o) {
  if (r.first) {
    float m0 = -1e30f, m1 = -1e30f;
#pragma unroll
    for (int j = 0; j < W; j += 4) {
      m0 = max3(m0, s[j], s[j + 1]);
      m1 = max3(m1, s[j + 2], s[j + 3]);
    }
    r.m = fmaxf(m0, m1);
    r.first = false;
  }
  float p[W];
  float l0, l1;
  {
    // three phases with no consumer next to its producer (a warp issues in order): arguments, W back-to-back MUFU.EX2 (the XU pipe
    // takes one warp instruction per 8 cycles: the other warp of the SM sub-partition issues in the gaps), then a sum TREE and the packs
    const float nm = -r.m;
#pragma unroll
    for (int j = 0; j < W; j += 2) {
      p[j] = s[j];
      p[j + 1] = s[j + 1];
      add2(p[j], p[j + 1], nm, nm);
    }
#pragma unroll
    for (int j = 0; j < W; ++j) p[j] = ex2_ftz(p[j]);
    float t0[W / 4 * 2];
#pragma unroll
    for (int j = 0; j < W / 4; ++j) {
      t0[2 * j] = p[4 * j];
      t0[2 * j + 1] = p[4 * j + 1];
      add2(t0[2 * j], t0[2 * j + 1], p[4 * j + 2], p[4 * j + 3]);
    }
#pragma unroll
    for (int n = W / 4; n > 1; n = (n + 1) / 2) {
#pragma unroll
      for (int j = 0; j < n / 2; ++j) add2(t0[2 * j], t0[2 * j + 1], t0[2 * (n - 1 - j)], t0[2 * (n - 1 - j) + 1]);
    }
    l0 = t0[0];
    l1 = t0[1];
  }
  float ps = l0 + l1;
  if (__any_sync(0xffffffffu, !(ps <= T2_PSUM_LIMIT))) {
    // ---- slow path (rare): some score of this piece exceeds the running maximum by more than ~2^14 ----
    float m0 = r.m, m1 = r.m;
#pragma unroll
    for (int j = 0; j < W; j += 4) {
      m0 = max3(m0, s[j], s[j + 1]);
      m1 = max3(m1, s[j + 2], s[j + 3]);
    }
    const float m2 = fmaxf(m0, m1);
    const float f = ex2_ftz(r.m - m2);          // 1 for the lanes whose maximum did not move
    r.l *= f;
    for (int pc = 0; pc < (c >> 1); pc += 2) {   // P columns of this chunk that were already written (bf16 pairs)
      uint32_t w2[2];
      tmem_ld_x2(ts_buf + pc, w2);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const float2 t = unpack_bf16x2(w2[j]);
        w2[j] = pack_bf16x2(t.x * f, t.y * f);
      }
      tmem_st_x2(ts_buf + pc, w2);
    }
    if (o_acc) {
      mbar_wait(pv_done, pv_parity);             // every P.V issued so far into this accumulator has retired
      tc_fence_after();
      uint32_t o[32];
      tmem_ld_x32(tmem_o, o);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) o[j] = __float_as_uint(__uint_as_float(o[j]) * f);
      tmem_st_x32(tmem_o, o);
    }
    tmem_st_wait();
    r.m = m2;
    l0 = 0.f;
    l1 = 0.f;
    const float nm = -m2;
#pragma unroll
    for (int j = 0; j < W; j += 2) {
      float a0 = s[j], a1 = s[j + 1];
      add2(a0, a1, nm, nm);
      p[j] = ex2_ftz(a0);
      p[j + 1] = ex2_ftz(a1);
      add2(l0, l1, p[j], p[j + 1]);
    }
    ps = l0 + l1;
  }
  r.l += ps;
  uint32_t pk[W / 2];
#pragma unroll
  for (int j = 0; j < W; j += 2) pk[j >> 1] = pack_bf16x2(p[j], p[j + 1]);
  tmem_st_n<W / 2>(ts_buf + (c >> 1), pk);
}

// generic piece: any window geometry, one shared-memory index + one gather per score
template <int W>
__device__ __forceinline__ void t2_softmax_piece(float (&s)[W], uint32_t ts_buf, int c, int gc, T2Row& r, bool o_acc, uint64_t* pv_done,
                                                 uint32_t pv_parity, uint32_t tmem_o) {
  t2_mask_pad<W>(s, gc, r);
  t2_exp_store<W>(s, ts_buf, c, r, o_acc, pv_done, pv_parity, tmem_o);
}

template <int W>
__device__ __forceinline__ void t2_piece(uint32_t ts_buf, int c, int gc, T2Row& r, bool o_acc, uint64_t* pv_done, uint32_t pv_parity,
                                         uint32_t tmem_o) {
  uint32_t v[W];
  tmem_ld_n<W>(ts_buf + c, v);
  int no[W];
#pragma unroll
  for (int j = 0; j < W; j += 4) *reinterpret_cast<int4*>(&no[j]) = *reinterpret_cast<const int4*>(r.negoff + gc + j);
  float s[W];
#pragma unroll
  for (int j = 0; j < W; ++j) s[j] = r.tabq[no[j]];
  tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < W; j += 2) add2(s[j], s[j + 1], __uint_as_float(v[j]), __uint_as_float(v[j + 1]));
  t2_softmax_piece<W>(s, ts_buf, c, gc, r, o_acc, pv_done, pv_parity, tmem_o);
}

// run piece: NR runs of RW consecutive keys (RW = configured window width, so a run shares (d_j, h_j) and its bias entries are RW
// consecutive table words): one address per run, the RW loads use immediate offsets -- no per-score index or address arithmetic.
//   issue : tcgen05.ld of the scores + shared-memory loads of the bias        finish: wait::ld, s + bias, mask, padding
// (a 28-column software-pipelined stream -- loads of piece k+1 in flight under the exponentials of piece k -- was measured slower than
// these wider pieces: 302 vs 265 us at the stage-2 shape; per-piece bookkeeping and instruction-cache misses outweigh the overlap)
template <int RW, int NR>
__device__ __forceinline__ void t2_run_issue(uint32_t ts_buf, int c, int gc, const T2Row& r, uint32_t (&v)[RW * NR], float (&b)[RW * NR]) {
  constexpr int W = RW * NR;
  tmem_ld_n<W>(ts_buf + c, v);
  int rcd[NR];
  const int run0 = gc / RW;                      // gc is a multiple of W, so run0 is a multiple of NR
  if constexpr (NR % 4 == 0) {
#pragma unroll
    for (int k = 0; k < NR; k += 4) *reinterpret_cast<int4*>(&rcd[k]) = *reinterpret_cast<const int4*>(r.runcode + run0 + k);
  } else {
    static_assert(NR % 2 == 0, "runs per piece must be even");
#pragma unroll
    for (int k = 0; k < NR; k += 2) *reinterpret_cast<int2*>(&rcd[k]) = *reinterpret_cast<const int2*>(r.runcode + run0 + k);
  }
#pragma unroll
  for (int k = 0; k < NR; ++k) {
    const float* ar = r.tabq - rcd[k];
#pragma unroll
    for (int w = 0; w < RW; ++w) b[k * RW + w] = *(ar - w);
  }
}
template <int W>
__device__ __forceinline__ void t2_run_finish(const uint32_t (&v)[W], const float (&b)[W], float (&x)[W], int gc, const T2Row& r) {
  tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < W; j += 2) {
    float a0 = b[j], a1 = b[j + 1];
    add2(a0, a1, __uint_as_float(v[j]), __uint_as_float(v[j + 1]));
    x[j] = a0;
    x[j + 1] = a1;
  }
  t2_mask_pad<W>(x, gc, r);
}
template <int RW, int NR>
__device__ __forceinline__ void t2_piece_runs(uint32_t ts_buf, int c, int gc, T2Row& r, bool o_acc, uint64_t* pv_done, uint32_t pv_parity,
                                              uint32_t tmem_o) {
  constexpr int W = RW * NR;
  uint32_t v[W];
  float b[W], x[W];
  t2_run_issue<RW, NR>(ts_buf, c, gc, r, v, b);
  t2_run_finish<W>(v, b, x, gc, r);
  t2_exp_store<W>(x, ts_buf, c, r, o_acc, pv_done, pv_parity, tmem_o);
}

template <int W>
__device__ __forceinline__ void t2_zero_piece(uint32_t ts_buf, int c) {
  uint32_t z[W / 2];
#pragma unroll
  for (int j = 0; j < W / 2; ++j) z[j] = 0u;
  tmem_st_n<W / 2>(ts_buf + (c >> 1), z);
}

// columns [cc, cl) of a chunk exist only to round the MMA N up to 16: P = 0 there
__device__ __forceinline__ void t2_zero_tail(uint32_t ts_buf, int cc, int cl) {
  const uint32_t z[2] = {0u, 0u};
  for (int pc = cc >> 1; pc < (cl >> 1); pc += 2) tmem_st_x2(ts_buf + pc, z);
}

// all pieces of one chunk (cl columns starting at key cs) for this warp's 32 rows.  MODE 0: generic 32 / 16-column pieces;
// MODE 1: 56-column pieces of 8 runs of 7 keys; MODE 2: 48-column pieces of 4 runs of 12 keys.  ``piece`` = running piece index of the
// group within the tile (replicated tail tile: quadrant q owns every fourth piece, the others get P = 0).
template <int MODE>
__device__ __forceinline__ void t2_chunk(uint32_t ts_buf, int cs, int cl, T2Row& row, bool rep, int q, int& piece, bool o_acc,
                                         uint64_t* pv_done, uint32_t pvp, uint32_t tmem_o) {
  if constexpr (MODE == 0) {
    int cc = 0;
    for (; cc + 32 <= cl; cc += 32, ++piece) {
      if (!rep || (piece & 3) == q) t2_piece<32>(ts_buf, cc, cs + cc, row, o_acc, pv_done, pvp, tmem_o);
      else t2_zero_piece<32>(ts_buf, cc);
    }
    if (cc < cl) {
      if (!rep || (piece & 3) == q) t2_piece<16>(ts_buf, cc, cs + cc, row, o_acc, pv_done, pvp, tmem_o);
      else t2_zero_piece<16>(ts_buf, cc);
      ++piece;
    }
  } else {
    constexpr int RW = MODE == 1 ? 7 : 12, NR = MODE == 1 ? 8 : 4, W = RW * NR;
    int cc = 0;
#pragma unroll 1
    for (; cc + W <= cl; cc += W, ++piece) {
      if (!rep || (piece & 3) == q) t2_piece_runs<RW, NR>(ts_buf, cc, cs + cc, row, o_acc, pv_done, pvp, tmem_o);
      else t2_zero_piece<W>(ts_buf, cc);
    }
    t2_zero_tail(ts_buf, cc, cl);
  }
}

template <int MODE>
__global__ void __launch_bounds__(T2_THREADS, 1)
window_attn_tc2_kernel(const __grid_constant__ CUtensorMap tmKV, const __grid_constant__ CUtensorMap tmQ,
                       const __grid_constant__ CUtensorMap tmQT, const AttnParams p, const AttnTc2Args a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* qring = smem + a.off_q;
  float* tab = reinterpret_cast<float*>(smem + a.off_tab);
  float* cfall = reinterpret_cast<float*>(smem + a.off_cf);       // [T2_G][NP]
  int* negoff = reinterpret_cast<int*>(smem + a.off_negoff);      // MODE 0: -code(j) per key; run modes: code(first key) per run
  float* pm = reinterpret_cast<float*>(smem + a.off_pm);          // [4][T2_G][128] group row max (tile index mod 4: with one chunk per
                                                                  // group and tile, group 0 runs up to three tiles ahead of the epilogue)
  float* ps = reinterpret_cast<float*>(smem + a.off_ps);          // [4][T2_G][128] group row sum
  float* xq = reinterpret_cast<float*>(smem + a.off_xq);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + a.off_bar);
  uint64_t* kv_full = bars;                // [2]
  uint64_t* kv_free = bars + 2;            // [2]
  uint64_t* q_full = bars + 4;             // [T2_NQ]
  uint64_t* q_free = bars + 4 + T2_NQ;     // [T2_NQ]
  uint64_t* s_full = bars + 4 + 2 * T2_NQ;             // [T2_G][2]
  uint64_t* p_ready = s_full + 2 * T2_G;               // [T2_G][2]
  uint64_t* pv_done = p_ready + 2 * T2_G;              // [T2_G]
  uint64_t* o_full = pv_done + T2_G;
  uint64_t* o_free = o_full + 1;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(o_free + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int N = a.N, NP = a.NP, ntiles = a.ntiles;
  const int SH = a.SH, SD = a.SD;
  const WinGeom& wg = p.win;

  // contiguous unit range of this CTA; unit u = head * nwin + window (head-major: the bias table is reloaded rarely)
  const int u_begin = static_cast<int>(1LL * a.units * blockIdx.x / gridDim.x);
  const int u_end = static_cast<int>(1LL * a.units * (blockIdx.x + 1) / gridDim.x);
  const int nunits = u_end - u_begin;
  const int T = nunits * ntiles;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmQ);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_free[i], a.ngact);
    }
    for (int i = 0; i < T2_NQ; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_free[i], a.ngact);
    }
    for (int i = 0; i < 2 * T2_G; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], 4);
    }
    for (int g = 0; g < T2_G; ++g) mbar_init(&pv_done[g], 1);
    mbar_init(o_full, a.ngact);
    mbar_init(o_free, 4);
    fence_mbar_init();
  }
  if (warp == T2_TMA_WARP) tmem_alloc(tmem_ptr_smem, 512);
  // per-launch table: -code(j) of the key tokens; zero the K / V pad rows of every stage
  if constexpr (MODE == 0) {
    for (int j = threadIdx.x; j < NP; j += blockDim.x) {
      int code = 0;
      if (j < N) code = (j / (wg.Wh * wg.Ww)) * SD + ((j / wg.Ww) % wg.Wh) * SH + j % wg.Ww;
      negoff[j] = -code;
    }
  } else {
    constexpr int RW = MODE == 1 ? 7 : 12;
    for (int rr = threadIdx.x; rr * RW < NP + RW; rr += blockDim.x) {
      const int j = rr * RW;                       // first key of the run: w_j = 0 (RW == configured window width)
      negoff[rr] = j < N ? (j / (wg.Wh * wg.Ww)) * SD + ((j / wg.Ww) % wg.Wh) * SH : 0;
    }
  }
  {
    const int npad = NP - N;
    for (int i = threadIdx.x; i < a.nkv * 2 * npad * 16; i += blockDim.x) {
      const int w = i & 15, rest = i >> 4;
      const int row = N + rest % npad, which = rest / npad;               // which: stage * 2 + {K, V}
      uint32_t* dst = reinterpret_cast<uint32_t*>(smem + (which >> 1) * a.kv_bytes + (which & 1) * NP * 64 + row * 64);
      dst[w] = 0;
    }
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == T2_TMA_WARP) {
    // =============================== TMA producer (one thread) ===============================
    if (lane == 0) {
      for (int lu = 0; lu < nunits; ++lu) {
        const int u = u_begin + lu, s = lu % a.nkv;
        const int head = u / a.nwin, win = u - head * a.nwin;
        if (lu >= a.nkv) mbar_wait(&kv_free[s], ((lu / a.nkv) - 1) & 1);      // every P.V of the unit that used this stage retired
        uint8_t* st = smem + s * a.kv_bytes;
        mbar_expect_tx(&kv_full[s], 2u * N * 64u);
        for (int op = 0; op < 2; ++op)
          for (int b = 0; b < a.nb; ++b)
            tma_load_2d(st + op * NP * 64 + b * a.BR * 64, &tmKV, &kv_full[s], (1 + op) * p.C + head * T2_HD, win * N + b * a.BR);
        for (int qt = 0; qt < ntiles; ++qt) {
          const int tq = lu * ntiles + qt, slot = tq % T2_NQ;
          if (tq >= T2_NQ) mbar_wait(&q_free[slot], ((tq / T2_NQ) - 1) & 1);
          uint8_t* qs = qring + slot * (128 * 64);
          mbar_expect_tx(&q_full[slot], 128u * 64u);
          if (a.r4 && qt == ntiles - 1) {
            // tail query rows, one copy per TMEM lane quadrant (rows past the tensor end are zero-filled by TMA)
            for (int qd = 0; qd < 4; ++qd)
              tma_load_2d(qs + qd * 32 * 64, &tmQT, &q_full[slot], head * T2_HD, win * N + qt * 128);
          } else {
            tma_load_2d(qs, &tmQ, &q_full[slot], head * T2_HD, win * N + qt * 128);
          }
        }
      }
    }
  } else if (warp >= T2_MMA_WARP0) {
    // =============================== MMA issuer of one group (warp-uniform loop, one elected lane issues) ===============================
    const int g = __shfl_sync(0xffffffffu, warp - T2_MMA_WARP0, 0);
    const int cg = (a.nchunks - g + T2_G - 1) / T2_G;            // chunks of a tile owned by this group
    const int per_unit = ntiles * cg;
    const int total = nunits * per_unit;
    const uint32_t idesc_pv = make_idesc_bf16_f32(128, T2_HD) | (1u << 16);     // B (= V) is MN-major
    const uint32_t tmem_o = tmem_base + T2_O_COL + g * T2_HD;
    int nq = 0, np = 0;
    while (np < total) {
      // Q K^T one item ahead of the P.V being waited for (never into a K/V stage that an un-issued P.V still has to release)
      while (nq < total && nq <= np + 1 && (nq / per_unit) < (np / per_unit) + a.nkv) {
        const int lu = nq / per_unit, rem = nq - lu * per_unit;
        const int qt = rem / cg, j = rem - qt * cg;
        const int s = lu % a.nkv, tq = lu * ntiles + qt, slot = tq % T2_NQ;
        const int c = g + j * T2_G;
        if (rem == 0) mbar_wait(&kv_full[s], (lu / a.nkv) & 1);
        if (j == 0) mbar_wait(&q_full[slot], (tq / T2_NQ) & 1);
        tc_fence_after();
        const uint64_t dq = make_sw64_desc(smem_u32(qring + slot * (128 * 64)));
        const uint64_t dk = make_sw64_desc(smem_u32(smem + s * a.kv_bytes) + a.cstart[c] * 64);
        const uint32_t idesc_qk = make_idesc_bf16_f32(128, a.clen[c]);
        const uint32_t tmem_s = tmem_base + (g * 2 + (nq & 1)) * T2_CW;
        if (elect_one_sync()) {
          umma_bf16_ss(tmem_s, dq, dk, idesc_qk, 0);
          umma_bf16_ss(tmem_s, dq + 2, dk + 2, idesc_qk, 1);
          umma_commit(&s_full[g * 2 + (nq & 1)]);
          if (j == cg - 1) umma_commit(&q_free[slot]);
        }
        __syncwarp();
        ++nq;
      }
      {
        const int lu = np / per_unit, rem = np - lu * per_unit;
        const int qt = rem / cg, j = rem - qt * cg;
        const int s = lu % a.nkv, tq = lu * ntiles + qt;
        const int c = g + j * T2_G;
        mbar_wait(&p_ready[g * 2 + (np & 1)], (np >> 1) & 1);
        if (j == 0 && tq >= 1) mbar_wait(o_free, (tq - 1) & 1);      // the epilogue of the previous tile no longer reads O_g
        tc_fence_after();
        const uint32_t tmem_s = tmem_base + (g * 2 + (np & 1)) * T2_CW;
        const uint64_t dv = make_sw64_desc(smem_u32(smem + s * a.kv_bytes) + NP * 64 + a.cstart[c] * 64);
        const int nks = a.clen[c] >> 4;
        if (elect_one_sync()) {
#pragma unroll 1
          for (int ks = 0; ks < nks; ++ks)               // 16 keys per step: 8 packed P columns, 16 V rows (1 KB)
            umma_bf16_ts(tmem_o, tmem_s + 8 * ks, dv + 64 * ks, idesc_pv, (j > 0 || ks > 0) ? 1u : 0u);
          umma_commit(&pv_done[g]);
          if (j == cg - 1) umma_commit(o_full);
          if (rem == per_unit - 1) umma_commit(&kv_free[s]);
        }
        __syncwarp();
        ++np;
      }
    }
  } else {
    // =============================== softmax warps (group 1: + epilogue of the previous tile) ===============================
    const int g = warp >> 2, q = warp & 3, r = q * 32 + lane;
    const int cg = (a.nchunks - g + T2_G - 1) / T2_G;
    const uint32_t tlane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t tmem_o = tlane + T2_O_COL + g * T2_HD;
    float* cf = cfall + g * NP;
    const int nW = wg.nwd * wg.nwh * wg.nww;
    const int Dp = wg.nwd * wg.wd, Hp = wg.nwh * wg.wh, Wp = wg.nww * wg.ww;

    // epilogue of tile te (group T2_EPI only): O = sum_g 2^(m_g - m) O_g / sum_g 2^(m_g - m) l_g
    auto epilogue = [&](int te) {
      const int lu = te / ntiles, qt = te - lu * ntiles;
      const int u = u_begin + lu;
      const int head = u / a.nwin, win = u - head * a.nwin;
      const bool rep = a.r4 && qt == ntiles - 1;            // replicated tail tile: every quadrant holds the same rows
      const int i = rep ? qt * 128 + lane : qt * 128 + r;
      const bool wvalid = rep || (qt * 128 + q * 32) < N;
      mbar_wait(o_full, te & 1);
      tc_fence_after();
      if (wvalid) {
        const float* pmb = pm + (te & 3) * T2_G * 128 + r;
        const float* psb = ps + (te & 3) * T2_G * 128 + r;
        float mg[T2_G], lg[T2_G];
        float m = -1e30f;
#pragma unroll
        for (int gg = 0; gg < T2_G; ++gg) {
          mg[gg] = gg < a.ngact ? pmb[gg * 128] : -1e30f;
          lg[gg] = gg < a.ngact ? psb[gg * 128] : 0.f;
          m = fmaxf(m, mg[gg]);
        }
        float wgt[T2_G];
        float l = 0.f;
#pragma unroll
        for (int gg = 0; gg < T2_G; ++gg) {
          wgt[gg] = ex2_ftz(mg[gg] - m);
          l = fmaf(wgt[gg], lg[gg], l);
        }
        const float inv = rep ? 1.0f : 1.0f / l;
        float lse_val = 0.f;                                // row statistic for the backward pass (base 2, like the scores)
        if (p.lse) lse_val = m + __log2f(l);
        float acc[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] = 0.f;
#pragma unroll
        for (int gg = 0; gg < T2_G; ++gg) {
          if (gg < a.ngact) {
            uint32_t o[32];
            tmem_ld_x32(tlane + T2_O_COL + gg * T2_HD, o);
            tmem_ld_wait();
            const float w = wgt[gg] * inv;
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[j] = fmaf(w, __uint_as_float(o[j]), acc[j]);
          }
        }
        if (rep) {
          // this quadrant only saw a quarter of the pieces: merge the four partials through shared memory
          if (lane < a.tail_rows) {
            float* dstq = xq + (q * T2_MAX_TAIL + lane) * 34;
            dstq[0] = m;
            dstq[1] = l;
#pragma unroll
            for (int j = 0; j < 32; ++j) dstq[2 + j] = acc[j];
          }
          named_bar(1 + T2_EPI, 128);
          if (q == 0 && lane < a.tail_rows) {
            const float* x0 = xq + lane * 34;
            const int QS = T2_MAX_TAIL * 34;
            const float mm = fmaxf(fmaxf(x0[0], x0[QS]), fmaxf(x0[2 * QS], x0[3 * QS]));
            float wq[4], ll = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              wq[k] = ex2_ftz(x0[k * QS] - mm);
              ll = fmaf(wq[k], x0[k * QS + 1], ll);
            }
            const float iv = 1.0f / ll;
            if (p.lse) lse_val = mm + __log2f(ll);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              float v = 0.f;
#pragma unroll
              for (int k = 0; k < 4; ++k) v = fmaf(wq[k], x0[k * QS + 2 + j], v);
              acc[j] = v * iv;
            }
          }
          named_bar(1 + T2_EPI, 128);
        }
        if (i < N && (!rep || q == 0)) {
          if (p.lse) p.lse[(static_cast<long long>(win) * N + i) * p.nH + head] = lse_val;
          __nv_bfloat16* dst = p.out + (static_cast<long long>(win) * N + i) * p.C + head * T2_HD;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            uint32_t w8[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) w8[j] = pack_bf16x2(acc[h * 16 + 2 * j], acc[h * 16 + 2 * j + 1]);
            asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + h * 16), "r"(w8[0]),
                         "r"(w8[1]), "r"(w8[2]), "r"(w8[3]), "r"(w8[4]), "r"(w8[5]), "r"(w8[6]), "r"(w8[7])
                         : "memory");
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_free);
    };

    int cur_head = -1;
    int t = 0, n = 0;
    for (int lu = 0; lu < nunits; ++lu) {
      const int u = u_begin + lu;
      const int head = u / a.nwin, win = u - head * a.nwin;
      if (head != cur_head) {
        // all softmax warps are past the previous head's tiles -> restage the table in its shared-memory layout
        named_bar(5, T2_SM_THREADS);
        const float* src = p.table_t + static_cast<long long>(head) * p.L;
        const int e2 = 2 * wg.Ww - 1, e1 = 2 * wg.Wh - 1;
        for (int i = threadIdx.x; i < p.L; i += T2_SM_THREADS) {
          const int cc = i % e2, bb = (i / e2) % e1, aa = i / (e2 * e1);
          tab[aa * SD + bb * SH + cc] = __ldg(src + i) * T2_LOG2E;
        }
        cur_head = head;
        named_bar(5, T2_SM_THREADS);
      }
      bool need_mask = false;
      int wa = 0, wb = 0, wc = 0, rd0 = 0, rh0 = 0, rw0 = 0;
      if (a.shifted) {
        const int wi = win % nW;
        wc = wi % wg.nww; wb = (wi / wg.nww) % wg.nwh; wa = wi / (wg.nww * wg.nwh);
        need_mask = (wg.sd && wa == wg.nwd - 1) || (wg.sh && wb == wg.nwh - 1) || (wg.sw && wc == wg.nww - 1);
        if (need_mask) {
          // region class of a token = per-axis (region - region of the window's first token): at most two regions per axis
          rd0 = shift_region(wa * wg.wd, Dp, wg.wd, wg.sd);
          rh0 = shift_region(wb * wg.wh, Hp, wg.wh, wg.sh);
          rw0 = shift_region(wc * wg.ww, Wp, wg.ww, wg.sw);
          named_bar(1 + g, 128);                      // the group is done with the previous window's classes
          for (int j = threadIdx.x & 127; j < NP; j += 128) {
            int cj = 0;
            if (j < N) {
              const int tw = j % wg.ww, th = (j / wg.ww) % wg.wh, td = j / (wg.ww * wg.wh);
              cj = 4 * (shift_region(wa * wg.wd + td, Dp, wg.wd, wg.sd) - rd0) +
                   2 * (shift_region(wb * wg.wh + th, Hp, wg.wh, wg.sh) - rh0) +
                   (shift_region(wc * wg.ww + tw, Wp, wg.ww, wg.sw) - rw0);
            }
            cf[j] = static_cast<float>(cj);
          }
          named_bar(1 + g, 128);
        }
      }

      for (int qt = 0; qt < ntiles; ++qt, ++t) {
        // Tail tile with <= 32 live rows: the rows are replicated into all four lane quadrants (see the TMA producer) and quadrant q
        // processes every fourth piece, so the tile costs a quarter of a full one instead of idling three SM sub-partitions.
        const bool rep = a.r4 && qt == ntiles - 1;
        const int i = rep ? qt * 128 + lane : qt * 128 + r;
        const bool wvalid = rep || (qt * 128 + q * 32) < N;   // warp-uniform: any live query row in this warp?
        T2Row row;
        {
          const int ic = i < N ? i : N - 1;
          const int code_i = (ic / (wg.Wh * wg.Ww)) * SD + ((ic / wg.Ww) % wg.Wh) * SH + ic % wg.Ww;
          row.tabq = tab + code_i + a.rc;
          row.negoff = negoff;
          row.runcode = negoff;
          row.cf = nullptr;
          row.cif = 0.f;
          if (need_mask) {
            const int tw = ic % wg.ww, th = (ic / wg.ww) % wg.wh, td = ic / (wg.ww * wg.wh);
            const int ci = 4 * (shift_region(wa * wg.wd + td, Dp, wg.wd, wg.sd) - rd0) +
                           2 * (shift_region(wb * wg.wh + th, Hp, wg.wh, wg.sh) - rh0) +
                           (shift_region(wc * wg.ww + tw, Wp, wg.ww, wg.sw) - rw0);
            row.cf = cf;
            row.cif = static_cast<float>(ci);
          }
          row.N = N;
          row.m = -1e30f;
          row.l = 0.f;
          row.first = true;
        }
        if (g == T2_EPI && cg == 0 && t >= 1) epilogue(t - 1);
        {
          int piece = 0;                                         // running piece index of this group within the tile
          for (int j = 0; j < cg; ++j, ++n) {
            const int c = g + j * T2_G;
            const int cs = a.cstart[c], cl = a.clen[c];
            const uint32_t ts_buf = tlane + (g * 2 + (n & 1)) * T2_CW;
            mbar_wait(&s_full[g * 2 + (n & 1)], (n >> 1) & 1);
            tc_fence_after();
            if (wvalid) {
              const uint32_t pvp = static_cast<uint32_t>((n - 1) & 1);
              t2_chunk<MODE>(ts_buf, cs, cl, row, rep, q, piece, j > 0, &pv_done[g], pvp, tmem_o);
              tmem_st_wait();
              if (j == cg - 1) {
                pm[((t & 3) * T2_G + g) * 128 + r] = row.m;
                ps[((t & 3) * T2_G + g) * 128 + r] = row.l;
              }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&p_ready[g * 2 + (n & 1)]);
            // group 1 drains the PREVIOUS tile's accumulators after its first chunk of this tile: by then both groups' last P.V of
            // that tile retired long ago, and the first P.V of this tile (which overwrites O) waits for o_free
            if (g == T2_EPI && j == 0 && t >= 1) epilogue(t - 1);
          }
        }
      }
    }
    if (g == T2_EPI && T > 0) epilogue(T - 1);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == T2_TMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
static bool t2_plan(const AttnParams& p, AttnTc2Args& a, int& smem_out) {
  const WinGeom& g = p.win;
  if (g.N < 16 || g.N > 1152) return false;
  a.N = g.N;
  a.NP = (g.N + 15) & ~15;
  a.ntiles = (g.N + 127) / 128;
  // K / V TMA boxes: the fewest boxes of <= 256 rows that tile N exactly
  a.nb = 0;
  for (int nb = (g.N + 255) / 256; nb <= 16; ++nb)
    if (g.N % nb == 0) { a.nb = nb; break; }
  if (a.nb == 0) return false;
  a.BR = g.N / a.nb;
  static int env_mode = -2;
  if (env_mode == -2) {
    const char* e = getenv("LAVT_ATTN_MODE");       // debugging / A-B runs: 0 forces the generic pieces
    env_mode = e ? atoi(e) : -1;
  }
  a.mode = g.Ww == 7 ? 1 : g.Ww == 12 ? 2 : 0;
  if (env_mode == 0) a.mode = 0;
  if (a.mode == 0) {
    // key chunks: an even number of <= 112 columns each (multiples of 16), balanced
    const int n16 = a.NP / 16;
    int nch = (n16 + 6) / 7;
    if (nch < 2 && n16 >= 2) nch = 2;          // both softmax groups get work even for one small window
    if (nch > 1 && (nch & 1)) ++nch;
    if (nch > n16) nch = n16;
    if (nch > T2_MAXCH) return false;
    a.nchunks = nch;
    int pos = 0;
    for (int c = 0; c < nch; ++c) {
      const int blocks = n16 / nch + (c < n16 % nch ? 1 : 0);
      a.cstart[c] = pos;
      a.clen[c] = blocks * 16;
      pos += blocks * 16;
    }
  } else {
    // run pieces of 56 / 48 columns, two per chunk (112 / 96 columns); the last chunk may hold one, rounded up to the MMA's N granule
    const int PW = a.mode == 1 ? 56 : 48;
    const int npieces = (g.N + PW - 1) / PW;
    const int nch = (npieces + 1) / 2;
    if (nch > T2_MAXCH) return false;
    a.nchunks = nch;
    for (int c = 0; c < nch; ++c) {
      const int pcs = c == nch - 1 ? npieces - 2 * (nch - 1) : 2;
      a.cstart[c] = c * 2 * PW;
      a.clen[c] = (pcs * PW + 15) & ~15;
    }
    a.NP = a.cstart[nch - 1] + a.clen[nch - 1];
  }
  a.ngact = a.nchunks >= 2 ? 2 : 1;
  for (int c = a.nchunks; c < T2_MAXCH; ++c) a.cstart[c] = a.clen[c] = 0;
  a.tail_rows = g.N - (a.ntiles - 1) * 128;
  a.r4 = (a.ntiles >= 2 && a.tail_rows <= T2_MAX_TAIL) ? 1 : 0;
  a.shifted = (g.sd | g.sh | g.sw) != 0;
  const int kv_bytes = 2 * a.NP * 64;
  a.kv_bytes = kv_bytes;
  // shared-memory plan: prefer two K/V stages and the bank-conflict-free table layout, fall back to one stage / the compact table
  for (int attempt = 0; attempt < 4; ++attempt) {
    const int nkv = (attempt & 1) ? 1 : 2;
    const bool expanded = attempt < 2;
    a.SH = expanded ? t2_stride(2 * g.Ww - 1, g.Ww % 32) : 2 * g.Ww - 1;
    a.SD = expanded ? t2_stride((2 * g.Wh - 1) * a.SH, (g.Wh * g.Ww) % 32) : (2 * g.Wh - 1) * a.SH;
    a.L2 = (2 * g.Wd - 1) * a.SD;
    a.rc = (g.Wd - 1) * a.SD + (g.Wh - 1) * a.SH + (g.Ww - 1);
    a.nkv = nkv;
    int off = nkv * kv_bytes;
    a.off_q = off;          off += T2_NQ * 128 * 64;
    a.off_tab = off;        off += ((a.L2 * 4 + 127) / 128) * 128;
    a.off_cf = off;         off += ((T2_G * a.NP * 4 + 127) / 128) * 128;
    a.off_negoff = off;     off += ((a.NP * 4 + 127) / 128) * 128;
    a.off_pm = off;         off += 4 * T2_G * 128 * 4;
    a.off_ps = off;         off += 4 * T2_G * 128 * 4;
    a.off_xq = off;         off += a.r4 ? 4 * T2_MAX_TAIL * 34 * 4 : 0;
    a.off_bar = off;        off += 256;
    const int smem = off + 1024;
    if (smem <= 227 * 1024) {
      smem_out = smem;
      return true;
    }
  }
  return false;
}

bool window_attn_tc2_supported(const AttnParams& p) {
  AttnTc2Args a;
  int smem = 0;
  return t2_plan(p, a, smem);
}

int window_attn_tc2_dispatch(const AttnParams& p, cudaStream_t st) {
  const WinGeom& g = p.win;
  AttnTc2Args a;
  int smem = 0;
  LAVT_REQUIRE(t2_plan(p, a, smem), "attention(tc2): unsupported window (N=%d, L=%d)", g.N, p.L);
  const long long nwin = 1LL * g.B * g.nwd * g.nwh * g.nww;
  LAVT_REQUIRE(nwin * p.nH < (1LL << 30), "attention(tc2): too many units");
  a.nwin = static_cast<int>(nwin);
  a.units = static_cast<int>(nwin * p.nH);

  CUtensorMap tm_kv, tm_q, tm_tail;
  {
    uint64_t dims[2] = {static_cast<uint64_t>(3 * p.C), static_cast<uint64_t>(nwin * g.N)};
    uint64_t strides[1] = {static_cast<uint64_t>(3 * p.C) * 2};
    uint32_t box[2] = {T2_HD, static_cast<uint32_t>(a.BR)};
    int rc = make_tmap_bf16_l2_64b(&tm_kv, p.qkv, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
    uint32_t box_q[2] = {T2_HD, 128};
    rc = make_tmap_bf16_l2_64b(&tm_q, p.qkv, 2, dims, strides, box_q, CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
    uint32_t box_t[2] = {T2_HD, 32};
    rc = make_tmap_bf16_l2_64b(&tm_tail, p.qkv, 2, dims, strides, box_t, CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
  }
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
      sms = 148;
  }
  const int grid = a.units < sms ? a.units : sms;
  static int configured[3] = {0, 0, 0};
  auto kfn = a.mode == 1 ? window_attn_tc2_kernel<1> : a.mode == 2 ? window_attn_tc2_kernel<2> : window_attn_tc2_kernel<0>;
  if (smem > configured[a.mode]) {
    LAVT_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured[a.mode] = smem;
  }
  kfn<<<grid, T2_THREADS, smem, st>>>(tm_kv, tm_q, tm_tail, p, a);
  LAVT_LAUNCH_CHECK("window_attn_tc2_kernel");
  return LAVT_OK;
}

}  // namespace lavt
