// tcgen05 / TMEM backward of the shifted-window attention core for every window of 16 ... 1152 tokens (any clamped extent, shifted or
// not; the 8 x 12 x 12 windows of the --window12 video model are the reason it exists).  Same mathematics and ABI as attn_bwd.cu and
// attn_bwd_tc.cu (reference WindowAttention3D.forward, lib/video_swin_transformer.py:147-165, differentiated by autograd in train.py:330-360):
//     Z = q' k^T + table[idx(i,j)] log2 e + mask(i,j)    P = 2^(Z - lse_i)    (lse saved by the forward kernel)
//     dV = P^T dO     dP = dO V^T     dZ = P o (dP - delta_i)     dQ = dZ K     dK = dZ^T Q     dtable[idx(i,j)] += dZ[i,j]
//
// Structure of attn_bwd_tc.cu (transposed orientation: TMEM lane = key row, column = query; pointwise warpgroups that never merge;
// dV / dK as TS MMAs with P^T / dZ^T read straight from TMEM; dQ from an MN-major dZ tile in shared memory; fixed-point table gradient),
// with the FlashAttention-2 split that lets the window grow past what one CTA can hold:
//   * 128-key tiles are the outer loop; their dK | dV accumulate in TMEM (double-buffered, drained one tile late);
//   * Q / dO stream in 64-query chunks (plain row order, no padding) through a 4-slot TMA ring, K / V tiles through a 2-stage ring;
//   * dQ of a 128-query tile and one key tile (dZ K, K = 128 keys) lands in one of two 32-column TMEM buffers; the pointwise warps drain it
//     one pair late and add it, in fp32, into a scratch region of the caller's workspace that this CTA owns for its current unit (no
//     atomics).  The first key tile stores, the last one adds, scales and writes bf16 dqkv; a single key tile needs no scratch at all.
//   * bias / gradient addressing works for any extent: a per-query table offset code(i) + rc (shared memory, warp-uniform int4 loads) and
//     a per-key base table - code(j) (one gather per score); shifted windows compare per-token region ids.
// TMEM (448 of 512 columns): S^T 2 x 64 | dP^T 2 x 64 | (dK | dV) 2 x 64 | dQ 2 x 32.
// Warps 0-15: pointwise groups (g = warp / 4: 16 query columns of a chunk, lane quadrant q = warp % 4); warp 16: MMA issue (one thread);
// warp 17: TMA producer + TMEM allocation.
#include "kernels.cuh"
#include "attn_tc_ptx.cuh"

namespace lavt {

constexpr int B2_HD = 32;
constexpr int B2_NG = 4;
constexpr int B2_SM_THREADS = 128 * B2_NG;
constexpr int B2_MMA_WARP = 4 * B2_NG;
constexpr int B2_TMA_WARP = 4 * B2_NG + 1;
constexpr int B2_THREADS = B2_SM_THREADS + 128;
constexpr int B2_NQ = 4;                    // Q / dO ring slots (one 64-query chunk each)
constexpr int B2_MAXN = 1152;
constexpr float B2_LOG2E = 1.4426950408889634f;
constexpr float B2_MASKV = -100.0f * B2_LOG2E;
constexpr int B2_COL_ST = 0, B2_COL_DP = 128, B2_COL_DKV = 256, B2_COL_DQ = 384;

struct AttnBwdTc2Args {
  int N, NP, nch, ntk;      // tokens per window, padded to whole 128-query tiles, 64-query chunks (even), 128-key tiles
  int nwin, units;
  int shifted;
  int off_kv, off_q, off_dz, off_tab, off_itab, off_qc, off_qr, off_lse, off_del, off_bar;
  float* scratch;           // [grid][NP][32] fp32 dQ partials, one region per CTA (ntk >= 2 only)
};

__device__ __forceinline__ void b2_mul2(float& a0, float& a1, float b0, float b1) {
  uint64_t a, b, r;
  asm("mov.b64 %0, {%1,%2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1,%2};" : "=l"(b) : "f"(b0), "f"(b1));
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  asm("mov.b64 {%0,%1}, %2;" : "=f"(a0), "=f"(a1) : "l"(r));
}

// One chunk (64 queries) for this thread's key row: the 16 query columns i0 .. i0 + 15 of group g.
//   ts / td : TMEM address of this group's 16 fp32 columns of S^T / dP^T (P^T / dZ^T go back to the first 8 of them as bf16 pairs)
//   nl / nd / qc / qr : -lse, -delta, code(i) + rc and region id of the 16 queries (shared memory, warp-uniform addresses)
//   kb / ib : table - code(j) and the same base in the fixed-point gradient table;  krid: region id of the key
//   dzrow   : this key's 128-byte row in the MN-major dZ tile of the chunk;  r7 = row & 7 (swizzle phase)
template <bool MASKED, bool TAIL>
__device__ __forceinline__ void b2_chunk(uint32_t ts, uint32_t td, int g, const float* kb, int* ib, int krid, float kpen, const float* nl,
                                         const float* nd, const int* qc, const int* qr, uint8_t* dzrow, int r7, float fix, bool do_tab) {
  uint32_t sv[16], dv[16];
  tmem_ld_x16(ts, sv);
  tmem_ld_x16(td, dv);
  uint32_t pw[8], zw[8];
#pragma unroll
  for (int kk = 0; kk < 2; ++kk) {
    float t[8], d[8];
    int o[8];
    {
      const float4 l0 = *reinterpret_cast<const float4*>(nl + 8 * kk), l1 = *reinterpret_cast<const float4*>(nl + 8 * kk + 4);
      const float4 d0 = *reinterpret_cast<const float4*>(nd + 8 * kk), d1 = *reinterpret_cast<const float4*>(nd + 8 * kk + 4);
      const int4 c0 = *reinterpret_cast<const int4*>(qc + 8 * kk), c1 = *reinterpret_cast<const int4*>(qc + 8 * kk + 4);
      t[0] = l0.x; t[1] = l0.y; t[2] = l0.z; t[3] = l0.w; t[4] = l1.x; t[5] = l1.y; t[6] = l1.z; t[7] = l1.w;
      d[0] = d0.x; d[1] = d0.y; d[2] = d0.z; d[3] = d0.w; d[4] = d1.x; d[5] = d1.y; d[6] = d1.z; d[7] = d1.w;
      o[0] = c0.x; o[1] = c0.y; o[2] = c0.z; o[3] = c0.w; o[4] = c1.x; o[5] = c1.y; o[6] = c1.z; o[7] = c1.w;
    }
    float b[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) b[e] = kb[o[e]];
#pragma unroll
    for (int e = 0; e < 8; e += 2) add2(t[e], t[e + 1], b[e], b[e + 1]);
    if constexpr (MASKED) {
      const int4 r0 = *reinterpret_cast<const int4*>(qr + 8 * kk), r1 = *reinterpret_cast<const int4*>(qr + 8 * kk + 4);
      const int rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
      for (int e = 0; e < 8; ++e) t[e] += rr[e] != krid ? B2_MASKV : 0.f;
    }
    if constexpr (TAIL) {
#pragma unroll
      for (int e = 0; e < 8; e += 2) add2(t[e], t[e + 1], kpen, kpen);
    }
    if (kk == 0) tmem_ld_wait();
    float pr[8], dz[8];
#pragma unroll
    for (int e = 0; e < 8; e += 2) {
      pr[e] = __uint_as_float(sv[8 * kk + e]);
      pr[e + 1] = __uint_as_float(sv[8 * kk + e + 1]);
      add2(pr[e], pr[e + 1], t[e], t[e + 1]);
      dz[e] = __uint_as_float(dv[8 * kk + e]);
      dz[e + 1] = __uint_as_float(dv[8 * kk + e + 1]);
      add2(dz[e], dz[e + 1], d[e], d[e + 1]);
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) pr[e] = ex2_ftz(pr[e]);
#pragma unroll
    for (int e = 0; e < 8; e += 2) b2_mul2(dz[e], dz[e + 1], pr[e], pr[e + 1]);
#pragma unroll
    for (int e = 0; e < 8; e += 2) {
      pw[4 * kk + (e >> 1)] = pack_bf16x2(pr[e], pr[e + 1]);
      zw[4 * kk + (e >> 1)] = pack_bf16x2(dz[e], dz[e + 1]);
    }
    if (do_tab) {
#pragma unroll
      for (int e = 0; e < 8; ++e) atomicAdd(ib + o[e], __float2int_rn(dz[e] * fix));
    }
  }
  tmem_st_x8(ts, pw);
  tmem_st_x8(td, zw);
  *reinterpret_cast<uint4*>(dzrow + (((2 * g) ^ r7) << 4)) = make_uint4(zw[0], zw[1], zw[2], zw[3]);
  *reinterpret_cast<uint4*>(dzrow + (((2 * g + 1) ^ r7) << 4)) = make_uint4(zw[4], zw[5], zw[6], zw[7]);
}

__device__ __forceinline__ void b2_st_bf16x8(__nv_bfloat16* dst, const float* v, float sc) {
  uint32_t w[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) w[e] = pack_bf16x2(v[2 * e] * sc, v[2 * e + 1] * sc);
  *reinterpret_cast<uint4*>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
}

__global__ void __launch_bounds__(B2_THREADS, 1)
window_attn_bwd_tc2_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO,
                           const __grid_constant__ CUtensorMap tmKV, const AttnBwdParams p, const AttnBwdTc2Args a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  float* tab = reinterpret_cast<float*>(smem + a.off_tab);
  int* itab = reinterpret_cast<int*>(smem + a.off_itab);
  int* qcode = reinterpret_cast<int*>(smem + a.off_qc);          // [NP] code(i) + rc (rc for padding queries)
  int* qrid = reinterpret_cast<int*>(smem + a.off_qr);           // [NP] region id of the current (masked) window
  float* nlse_s = reinterpret_cast<float*>(smem + a.off_lse);    // [NP] -lse (-1e30 for padding queries: P = 0)
  float* ndel_s = reinterpret_cast<float*>(smem + a.off_del);    // [NP] -delta
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + a.off_bar);
  uint64_t* kv_full = bars;            // [2] K / V of a key tile landed
  uint64_t* kv_free = bars + 2;        // [2] every MMA that reads them retired
  uint64_t* q_full = bars + 4;         // [B2_NQ] Q / dO of a chunk landed
  uint64_t* q_free = bars + 8;         // [B2_NQ]
  uint64_t* s_full = bars + 12;        // [2] S^T and dP^T of an item are in TMEM
  uint64_t* p_ready = bars + 14;       // [2] the 16 pointwise warps wrote P^T / dZ^T (TMEM) and dZ (shared memory) of an item
  uint64_t* dz_free = bars + 16;       // [2] the dQ MMA that read this dZ tile retired
  uint64_t* dkv_full = bars + 18;      // [2] dK | dV of a key tile are complete
  uint64_t* dkv_free = bars + 20;      // [2] ... and have been read out
  uint64_t* dq_full = bars + 22;       // [2] dQ partial of a (key tile, query tile) pair is complete
  uint64_t* dq_free = bars + 24;       // [2] ... and has been read out
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 26);
  int* umax = reinterpret_cast<int*>(bars + 27);                 // [2][2] bit patterns of max ||dO_i||^2, max ||V_j||^2 per unit parity

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int N = a.N, NP = a.NP, nch = a.nch, ntk = a.ntk;
  const int NT = ntk * nch;                                // (key tile, chunk) items per unit
  const WinGeom& wg = p.win;
  const int u_begin = static_cast<int>(1LL * a.units * blockIdx.x / gridDim.x);
  const int u_end = static_cast<int>(1LL * a.units * (blockIdx.x + 1) / gridDim.x);
  const int nunits = u_end - u_begin;
  const int total = nunits * NT;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQKV);
    tma_prefetch_desc(&tmDO);
    tma_prefetch_desc(&tmKV);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_free[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], 4 * B2_NG);
      mbar_init(&dz_free[i], 1);
      mbar_init(&dkv_full[i], 1);
      mbar_init(&dkv_free[i], 4 * B2_NG);
      mbar_init(&dq_full[i], 1);
      mbar_init(&dq_free[i], 4 * B2_NG);
    }
    for (int i = 0; i < B2_NQ; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_free[i], 1);
    }
    umax[0] = umax[1] = umax[2] = umax[3] = 0;
    fence_mbar_init();
  }
  if (warp == B2_TMA_WARP) tmem_alloc(tmem_ptr_smem, 512);
  for (int i = threadIdx.x; i < p.L + 32; i += blockDim.x) itab[i] = 0;
  {
    const int rc = rel_const(wg);
    for (int i = threadIdx.x; i < NP; i += blockDim.x) {
      int code = 0;
      if (i < N) {
        const int cw = i % wg.Ww, chh = (i / wg.Ww) % wg.Wh, cd = i / (wg.Ww * wg.Wh);
        code = (cd * (2 * wg.Wh - 1) + chh) * (2 * wg.Ww - 1) + cw;
      }
      qcode[i] = code + rc;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp >= 4 * B2_NG) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
  if (warp == B2_TMA_WARP) {
    // =============================== TMA producer (one thread), in item order ===============================
    if (lane == 0) {
      for (int n = 0; n < total; ++n) {
        const int lu = n / NT, rem = n - lu * NT, j = rem / nch, c = rem - j * nch;
        const int u = u_begin + lu;
        const int head = u / a.nwin, win = u - head * a.nwin;
        if (c == 0) {
          const int kt = lu * ntk + j, s = kt & 1;
          if (kt >= 2) mbar_wait(&kv_free[s], ((kt >> 1) - 1) & 1);
          mbar_expect_tx(&kv_full[s], 16384u);
          tma_load_2d(smem + a.off_kv + s * 16384, &tmKV, &kv_full[s], p.C + head * B2_HD, win * N + j * 128);
          tma_load_2d(smem + a.off_kv + s * 16384 + 8192, &tmKV, &kv_full[s], 2 * p.C + head * B2_HD, win * N + j * 128);
        }
        const int slot = n % B2_NQ;
        if (n >= B2_NQ) mbar_wait(&q_free[slot], ((n / B2_NQ) - 1) & 1);
        mbar_expect_tx(&q_full[slot], 8192u);
        tma_load_2d(smem + a.off_q + slot * 8192, &tmQKV, &q_full[slot], head * B2_HD, win * N + c * 64);
        tma_load_2d(smem + a.off_q + slot * 8192 + 4096, &tmDO, &q_full[slot], head * B2_HD, win * N + c * 64);
      }
    }
  } else if (warp == B2_MMA_WARP) {
    // =============================== MMA issue (one thread; its tcgen05.mma execute in issue order) ===============================
    if (lane == 0) {
      const uint32_t idesc_s = make_idesc_bf16_f32(128, 64);
      const uint32_t idesc_kv = make_idesc_bf16_f32(128, B2_HD) | (1u << 16);                 // B (dO / Q rows) MN-major
      const uint32_t idesc_dq = make_idesc_bf16_f32(128, B2_HD) | (1u << 15) | (1u << 16);    // A (dZ tile) and B (K rows) MN-major
      const uint32_t sbase = smem_u32(smem);
      const uint32_t kv_base = sbase + a.off_kv, q_base = sbase + a.off_q, dz_base = sbase + a.off_dz;
      auto issue_sdp = [&](int n) {
        const int lu = n / NT, rem = n - lu * NT, j = rem / nch, c = rem - j * nch;
        const int kt = lu * ntk + j, s = kt & 1, slot = n % B2_NQ, buf = n & 1;
        if (c == 0) mbar_wait(&kv_full[s], (kt >> 1) & 1);
        mbar_wait(&q_full[slot], (n / B2_NQ) & 1);
        tc_fence_after();
        const uint64_t dk = make_sw64_desc(kv_base + s * 16384), dv = make_sw64_desc(kv_base + s * 16384 + 8192);
        const uint64_t dq = make_sw64_desc(q_base + slot * 8192), dd = make_sw64_desc(q_base + slot * 8192 + 4096);
        const uint32_t ts = tmem_base + B2_COL_ST + buf * 64, td = tmem_base + B2_COL_DP + buf * 64;
        umma_bf16_ss(ts, dk, dq, idesc_s, 0);
        umma_bf16_ss(ts, dk + 2, dq + 2, idesc_s, 1);
        umma_bf16_ss(td, dv, dd, idesc_s, 0);
        umma_bf16_ss(td, dv + 2, dd + 2, idesc_s, 1);
        umma_commit(&s_full[buf]);
      };
      if (total > 0) issue_sdp(0);
      if (total > 1) issue_sdp(1);
      for (int n = 0; n < total; ++n) {
        const int lu = n / NT, rem = n - lu * NT, j = rem / nch, c = rem - j * nch;
        const int kt = lu * ntk + j, s = kt & 1, slot = n % B2_NQ, buf = n & 1;
        mbar_wait(&p_ready[buf], (n >> 1) & 1);
        if (c == 0 && kt >= 2) mbar_wait(&dkv_free[kt & 1], ((kt >> 1) - 1) & 1);
        tc_fence_after();
        {
          const uint32_t tdk = tmem_base + B2_COL_DKV + (kt & 1) * 64, tdv = tdk + B2_HD;
          const uint32_t tp = tmem_base + B2_COL_ST + buf * 64, tz = tmem_base + B2_COL_DP + buf * 64;
          const uint64_t bq = make_sw64_desc(q_base + slot * 8192), bd = make_sw64_desc(q_base + slot * 8192 + 4096);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) umma_bf16_ts(tdv, tp + 16 * ks, bd + 64 * ks, idesc_kv, (c > 0 || ks > 0) ? 1u : 0u);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) umma_bf16_ts(tdk, tz + 16 * ks, bq + 64 * ks, idesc_kv, (c > 0 || ks > 0) ? 1u : 0u);
          umma_commit(&q_free[slot]);
        }
        if (c & 1) {
          const int m = n >> 1, dqb = m & 1;                       // (key tile, query tile) pair
          if (m >= 2) mbar_wait(&dq_free[dqb], ((m >> 1) - 1) & 1);
          tc_fence_after();
          const int nk = min(128, N - j * 128), nks = (nk + 15) >> 4;
          const uint64_t da = make_mnmajor_sw128_desc(dz_base + dqb * 32768, 16384);
          const uint64_t db = make_sw64_desc(kv_base + s * 16384);
          const uint32_t tq = tmem_base + B2_COL_DQ + dqb * B2_HD;
          for (int ks = 0; ks < nks; ++ks) umma_bf16_ss(tq, da + 128 * ks, db + 64 * ks, idesc_dq, ks > 0 ? 1u : 0u);
          umma_commit(&dz_free[dqb]);
          umma_commit(&dq_full[dqb]);
        }
        if (c == nch - 1) {
          umma_commit(&dkv_full[kt & 1]);
          umma_commit(&kv_free[s]);
        }
        if (n + 2 < total) issue_sdp(n + 2);
      }
    }
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    // =============================== pointwise warps ===============================
    const int g = warp >> 2, q = warp & 3, r = q * 32 + lane;
    const uint32_t tlane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const int nW = wg.nwd * wg.nwh * wg.nww;
    const bool do_tab = p.dtable_t != nullptr;
    const int tid = threadIdx.x;                        // 0 .. 511
    float* scratch = a.scratch + static_cast<long long>(blockIdx.x) * NP * B2_HD;
    int cur_head = -1;
    float prev_inv_fix = 0.f;
    int prev_head = 0;

    auto fold_table = [&]() {
      for (int pos = tid; pos < p.L; pos += B2_SM_THREADS) {
        const int v = itab[pos];
        if (v != 0) {
          atomicAdd(p.dtable_t + static_cast<long long>(prev_head) * p.L + pos, static_cast<float>(v) * prev_inv_fix);
          itab[pos] = 0;
        }
      }
    };
    // dK | dV of key tile (global index kt, tile j of the unit): group g < 2 holds 16 columns of dK, g >= 2 of dV
    auto drain_dkv = [&](int kt, int j, long long row0, int head) {
      mbar_wait(&dkv_full[kt & 1], (kt >> 1) & 1);
      tc_fence_after();
      if (j * 128 + q * 32 < N) {                        // warp-uniform: this warp holds live key rows
        uint32_t v[16];
        tmem_ld_x16(tlane + B2_COL_DKV + (kt & 1) * 64 + 16 * g, v);
        tmem_ld_wait();
        const int kr = j * 128 + r;
        if (kr < N) {
          // dy_k = dZ^T q' / log2 e  (q' = y_q hd^-0.5 log2 e),  dy_v = P^T dO
          const float sc = g < 2 ? (1.0f / B2_LOG2E) : 1.0f;
          __nv_bfloat16* dst = p.dqkv + (row0 + kr) * (3 * p.C) + (g < 2 ? p.C : 2 * p.C) + head * B2_HD + (g & 1) * 16;
          uint32_t w8[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) w8[e] = pack_bf16x2(__uint_as_float(v[2 * e]) * sc, __uint_as_float(v[2 * e + 1]) * sc);
          asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(w8[0]), "r"(w8[1]), "r"(w8[2]),
                       "r"(w8[3]), "r"(w8[4]), "r"(w8[5]), "r"(w8[6]), "r"(w8[7])
                       : "memory");
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&dkv_free[kt & 1]);
    };
    // dQ partial of pair m = (key tile j, query tile t): this thread owns query t * 128 + r, channels 8 g .. 8 g + 7
    auto drain_dq = [&](int m, int j, int t, long long row0, int head) {
      const int dqb = m & 1;
      mbar_wait(&dq_full[dqb], (m >> 1) & 1);
      tc_fence_after();
      const int i = t * 128 + r;
      if (t * 128 + q * 32 < N) {                        // warp-uniform
        uint32_t v[8];
        tmem_ld_x8(tlane + B2_COL_DQ + dqb * B2_HD + 8 * g, v);
        tmem_ld_wait();
        if (i < N) {
          float x[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(v[e]);
          float4* sp = reinterpret_cast<float4*>(scratch + i * B2_HD + 8 * g);
          if (j > 0) {
            const float4 s0 = sp[0], s1 = sp[1];
            x[0] += s0.x; x[1] += s0.y; x[2] += s0.z; x[3] += s0.w;
            x[4] += s1.x; x[5] += s1.y; x[6] += s1.z; x[7] += s1.w;
          }
          if (j == ntk - 1) {
            b2_st_bf16x8(p.dqkv + (row0 + i) * (3 * p.C) + head * B2_HD + 8 * g, x, p.qscale);
          } else {
            sp[0] = make_float4(x[0], x[1], x[2], x[3]);
            sp[1] = make_float4(x[4], x[5], x[6], x[7]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&dq_free[dqb]);
    };

    int n = 0;
    for (int lu = 0; lu < nunits; ++lu) {
      const int u = u_begin + lu;
      const int head = u / a.nwin, win = u - head * a.nwin;
      const long long row0 = static_cast<long long>(win) * N;
      // ---- unit prologue: fold the previous unit's table gradient, (re)stage the bias table, per-query -lse / -delta, scale ----
      if (lu >= 1 && do_tab) fold_table();
      if (head != cur_head) {
        const float* src = p.table_t + static_cast<long long>(head) * p.L;
        for (int pos = tid; pos < p.L; pos += B2_SM_THREADS) tab[pos] = __ldg(src + pos) * B2_LOG2E;
        cur_head = head;
      }
      bool need_mask = false;
      if (a.shifted) {
        const int wi_ = win % nW;
        const int wc = wi_ % wg.nww, wb = (wi_ / wg.nww) % wg.nwh, wa = wi_ / (wg.nww * wg.nwh);
        need_mask = (wg.sd && wa == wg.nwd - 1) || (wg.sh && wb == wg.nwh - 1) || (wg.sw && wc == wg.nww - 1);
      }
      {
        float ndo = 0.f, nv = 0.f;
        for (int i = tid; i < NP; i += B2_SM_THREADS) {
          float nl = -1e30f, ndl = 0.f;
          int rid = -1;
          if (i < N) {
            const long long row = row0 + i;
            const uint4* o4 = reinterpret_cast<const uint4*>(p.out + row * p.C + head * B2_HD);
            const uint4* d4 = reinterpret_cast<const uint4*>(p.dout + row * p.C + head * B2_HD);
            const uint4* v4 = reinterpret_cast<const uint4*>(p.qkv + row * (3 * p.C) + 2 * p.C + head * B2_HD);
            float acc = 0.f, sd = 0.f, sv = 0.f;
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {
              const uint4 x = __ldg(o4 + ch), y = __ldg(d4 + ch), z = __ldg(v4 + ch);
              const uint32_t xx[4] = {x.x, x.y, x.z, x.w}, yy[4] = {y.x, y.y, y.z, y.w}, zz[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float2 xo = unpack_bf16x2(xx[e]), yd = unpack_bf16x2(yy[e]), zv = unpack_bf16x2(zz[e]);
                acc += xo.x * yd.x + xo.y * yd.y;
                sd += yd.x * yd.x + yd.y * yd.y;
                sv += zv.x * zv.x + zv.y * zv.y;
              }
            }
            ndo = fmaxf(ndo, sd);
            nv = fmaxf(nv, sv);
            nl = -__ldg(p.lse + row * p.nH + head);
            ndl = -acc;
            if (need_mask) rid = win_token(wg, row).rid;
          }
          nlse_s[i] = nl;
          ndel_s[i] = ndl;
          if (need_mask) qrid[i] = rid;
        }
        ndo = warp_max(ndo);
        nv = warp_max(nv);
        if (lane == 0) {                       // non-negative floats order like their bit patterns
          atomicMax(&umax[(lu & 1) * 2], __float_as_int(ndo));
          atomicMax(&umax[(lu & 1) * 2 + 1], __float_as_int(nv));
        }
        if (tid == 0) umax[((lu + 1) & 1) * 2] = umax[((lu + 1) & 1) * 2 + 1] = 0;
      }
      named_bar(2, B2_SM_THREADS);
      // |dZ| <= |dP| + |delta| <= 2 max||dO_i|| max||V_j|| (Cauchy-Schwarz; O is a convex combination of V rows), <= N terms per entry:
      // scale = 2^30 / (2.5 N bound) cannot overflow int32
      const float bound = 2.5f * static_cast<float>(N) * sqrtf(__int_as_float(umax[(lu & 1) * 2]) * __int_as_float(umax[(lu & 1) * 2 + 1]));
      const float fix = (bound > 0.f && isfinite(bound)) ? 1073741824.0f / bound : 1.0f;

      for (int j = 0; j < ntk; ++j) {
        const int kt = lu * ntk + j;
        const int kr = j * 128 + r;
        const bool wvalid = j * 128 + q * 32 < N;           // warp-uniform
        const bool tail = (j + 1) * 128 > N;
        const int krc = kr < N ? kr : N - 1;
        const int kcode = qcode[krc] - rel_const(wg);
        const float* kb = tab - kcode;
        int* ib = itab - kcode;
        const float kpen = kr < N ? 0.f : -1e30f;
        const int krid = need_mask ? win_token(wg, row0 + krc).rid : 0;
        for (int c = 0; c < nch; ++c, ++n) {
          const int buf = n & 1;
          mbar_wait(&s_full[buf], (n >> 1) & 1);
          if ((n & 1) == 0 && (n >> 1) >= 2) mbar_wait(&dz_free[(n >> 1) & 1], (((n >> 1) >> 1) - 1) & 1);
          tc_fence_after();
          if (wvalid) {
            const uint32_t ts = tlane + B2_COL_ST + buf * 64 + 16 * g, td = tlane + B2_COL_DP + buf * 64 + 16 * g;
            uint8_t* dzrow = smem + a.off_dz + ((n >> 1) & 1) * 32768 + (c & 1) * 16384 + r * 128;
            const int i0 = c * 64 + 16 * g;
            if (need_mask) {
              if (tail) b2_chunk<true, true>(ts, td, g, kb, ib, krid, kpen, nlse_s + i0, ndel_s + i0, qcode + i0, qrid + i0, dzrow, r & 7, fix, do_tab);
              else b2_chunk<true, false>(ts, td, g, kb, ib, krid, kpen, nlse_s + i0, ndel_s + i0, qcode + i0, qrid + i0, dzrow, r & 7, fix, do_tab);
            } else {
              if (tail) b2_chunk<false, true>(ts, td, g, kb, ib, krid, kpen, nlse_s + i0, ndel_s + i0, qcode + i0, qrid + i0, dzrow, r & 7, fix, do_tab);
              else b2_chunk<false, false>(ts, td, g, kb, ib, krid, kpen, nlse_s + i0, ndel_s + i0, qcode + i0, qrid + i0, dzrow, r & 7, fix, do_tab);
            }
          }
          tmem_st_wait();
          tc_fence_before();
          fence_proxy_async_smem();                          // the dZ rows are read by the tensor core (async proxy)
          __syncwarp();
          if (lane == 0) mbar_arrive(&p_ready[buf]);
          if (c == 0 && j > 0) drain_dkv(kt - 1, j - 1, row0, head);    // previous key tile: its last MMAs retired long ago
          if (c & 1) {                                       // the dQ pair before the one this chunk completes (same unit only)
            if (c >= 3) drain_dq((n >> 1) - 1, j, (c >> 1) - 1, row0, head);
            else if (j > 0) drain_dq((n >> 1) - 1, j - 1, nch / 2 - 1, row0, head);
          }
        }
      }
      // ---- unit epilogue: last key tile, last dQ pair, and everybody's atomics before the table is folded ----
      drain_dkv(lu * ntk + ntk - 1, ntk - 1, row0, head);
      drain_dq((n >> 1) - 1, ntk - 1, nch / 2 - 1, row0, head);
      prev_inv_fix = 1.0f / fix;
      prev_head = head;
      named_bar(1, B2_SM_THREADS);
    }
    if (nunits > 0 && do_tab) fold_table();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == B2_TMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
static bool b2_plan(const AttnBwdParams& p, AttnBwdTc2Args& a, int& smem_out) {
  const WinGeom& g = p.win;
  if (g.N < 16 || g.N > B2_MAXN || g.N != g.wd * g.wh * g.ww) return false;
  if (p.C != p.nH * B2_HD || p.lse == nullptr) return false;
  if (p.L != (2 * g.Wd - 1) * (2 * g.Wh - 1) * (2 * g.Ww - 1)) return false;
  a.N = g.N;
  a.ntk = (g.N + 127) / 128;
  a.nch = 2 * a.ntk;
  a.NP = 128 * a.ntk;
  a.shifted = (g.sd | g.sh | g.sw) != 0;
  int off = 0;
  a.off_kv = off;    off += 2 * 16384;
  a.off_q = off;     off += B2_NQ * 8192;
  a.off_dz = off;    off += 2 * 32768;
  const int tab_bytes = ((p.L + 32) * 4 + 127) / 128 * 128;
  a.off_tab = off;   off += tab_bytes;
  a.off_itab = off;  off += tab_bytes;
  a.off_qc = off;    off += a.NP * 4;
  a.off_qr = off;    off += a.NP * 4;
  a.off_lse = off;   off += a.NP * 4;
  a.off_del = off;   off += a.NP * 4;
  a.off_bar = off;   off += 256;
  smem_out = off + 1024;
  return smem_out <= 227 * 1024;
}

bool window_attn_bwd_tc2_supported(const AttnBwdParams& p) {
  AttnBwdTc2Args a;
  int smem = 0;
  return b2_plan(p, a, smem);
}

static int b2_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) {
      cudaGetLastError();
      sms = 148;
    }
  }
  return sms;
}

// fp32 dQ scratch: one [NP][32] region per CTA of the persistent grid, needed only when a window spans more than one key tile
long long window_attn_bwd_tc2_workspace_floats(const AttnBwdParams& p) {
  AttnBwdTc2Args a;
  int smem = 0;
  if (!b2_plan(p, a, smem) || a.ntk < 2) return 0;
  const WinGeom& g = p.win;
  const long long units = 1LL * g.B * g.nwd * g.nwh * g.nww * p.nH;
  const long long grid = units < b2_sms() ? units : b2_sms();
  return grid * a.NP * B2_HD;
}

int window_attn_bwd_tc2_dispatch(const AttnBwdParams& p, float* workspace, long long workspace_floats, cudaStream_t st) {
  const WinGeom& g = p.win;
  AttnBwdTc2Args a;
  int smem = 0;
  LAVT_REQUIRE(b2_plan(p, a, smem), "attention backward (tcgen05, tc2): unsupported window (N=%d, L=%d)", g.N, p.L);
  const long long nwin = 1LL * g.B * g.nwd * g.nwh * g.nww;
  LAVT_REQUIRE(nwin * p.nH < (1LL << 30), "attention backward (tcgen05, tc2): too many units");
  a.nwin = static_cast<int>(nwin);
  a.units = static_cast<int>(nwin * p.nH);
  int grid = a.units < b2_sms() ? a.units : b2_sms();
  a.scratch = nullptr;
  if (a.ntk >= 2) {
    const long long per_cta = 1LL * a.NP * B2_HD;
    LAVT_REQUIRE(workspace != nullptr && workspace_floats >= per_cta,
                 "attention backward (tcgen05, tc2): window of %d tokens needs a workspace of lavt_window_attention_bwd_workspace_floats "
                 "floats (got %lld)", g.N, workspace_floats);
    if (workspace_floats / per_cta < grid) grid = static_cast<int>(workspace_floats / per_cta);
    a.scratch = workspace;
  }

  CUtensorMap tm_qkv, tm_do, tm_kv;
  {
    const uint64_t rowb = static_cast<uint64_t>(3 * p.C) * 2;
    uint64_t dims[2] = {static_cast<uint64_t>(3 * p.C), static_cast<uint64_t>(nwin * g.N)};
    uint64_t strides[1] = {rowb};
    uint32_t box_q[2] = {B2_HD, 64};
    int rc = make_tmap_bf16_l2_64b(&tm_qkv, p.qkv, 2, dims, strides, box_q, CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
    uint64_t dd[2] = {static_cast<uint64_t>(p.C), static_cast<uint64_t>(nwin * g.N)};
    uint64_t sd[1] = {static_cast<uint64_t>(p.C) * 2};
    rc = make_tmap_bf16_l2_64b(&tm_do, p.dout, 2, dd, sd, box_q, CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
    uint32_t box_kv[2] = {B2_HD, 128};
    rc = make_tmap_bf16_l2_64b(&tm_kv, p.qkv, 2, dims, strides, box_kv, CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
  }
  static int configured = 0;
  if (smem > configured) {
    LAVT_CUDA(cudaFuncSetAttribute(window_attn_bwd_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = smem;
  }
  window_attn_bwd_tc2_kernel<<<grid, B2_THREADS, smem, st>>>(tm_qkv, tm_do, tm_kv, p, a);
  LAVT_LAUNCH_CHECK("window_attn_bwd_tc2_kernel");
  return LAVT_OK;
}

}  // namespace lavt
