// Backward of the shifted-window attention core (reference WindowAttention3D.forward, lib/video_swin_transformer.py:147-165,
// differentiated by autograd in the reference's training loop, train.py:330-360).  Per (window, head), with the natural-log
// logits  Z = hd^-0.5 (y_q . y_k) + table[idx(i,j)] + mask(i,j),  P = softmax_j Z,  O = P V:
//     dV = P^T dO          dP = dO V^T          dZ = P o (dP - delta),  delta_i = sum_c dO[i,c] O[i,c]
//     dy_q = hd^-0.5 dZ K  dy_k = hd^-0.5 dZ^T y_q                      dtable[idx(i,j), head] += dZ[i,j]
// Inputs are what the forward saved: qkv (bf16, q pre-scaled by hd^-0.5 * log2 e -- the base-2 softmax convention of the
// forward kernels) and O.  The N x N matrices are recomputed tile by tile with mma.sync.m16n8k16 and never leave registers;
// the row statistics (log-sum-exp) are recomputed in a first pass instead of being stored by the forward kernels.
//
// One persistent CTA walks (head, window) units; Q, K, V, dO of the unit live in shared memory (cp.async, 64-byte rows with
// the xor chunk swizzle of attn_window.cu).  Main loop: a warp OWNS a 16-key tile (dK, dV accumulate in registers across
// all query blocks; S^T = K Q^T and dP^T = V dO^T make P^T / dZ^T come out of the MMA already in A-fragment layout); a second
// pass with a warp owning 16 QUERY rows recomputes S / dP / dZ and accumulates dQ in registers (a first version reduced dQ^T =
// K^T dZ^T across the key-owning warps with shared fp32 atomics: 36 ms per training step vs the recomputation's cost).  The
// relative-position-bias gradient accumulates per unit in fixed point (scale from a per-unit bound) with native integer shared atomics (fp32 shared
// atomics are CAS loops) and per CTA in an fp32 table copy that is flushed when the head changes.
#include "kernels.cuh"

#include <cstdlib>

namespace lavt {

constexpr int AB_HD = 32;
constexpr float AB_LOG2E = 1.4426950408889634f;
constexpr float AB_MASKV = -100.0f * AB_LOG2E;
constexpr int AB_WARPS = 16;

__device__ __forceinline__ int ab_off(int row, int chunk) { return row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4); }
__device__ __forceinline__ float ab_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t movmatrix_trans(uint32_t a) {
  uint32_t d;
  asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(d) : "r"(a));
  return d;
}

struct AbTok {        // per-token record: one LDS.128 in the main loop
  int code;           // linearised position in the configured window (rel-pos index closed form)
  int rid;            // shifted-window region id
  float lse;          // log2-sum-exp2 of the token's score row
  float delta;        // sum_c dO[i,c] * O[i,c]
};

__global__ void __launch_bounds__(AB_WARPS * 32, 1) window_attn_bwd_kernel(const AttnBwdParams p, const int NP, const int units) {
  extern __shared__ __align__(16) uint8_t ab_smem[];
  const int N = p.win.N, C = p.C, L = p.L;
  uint8_t* sQ = ab_smem;
  uint8_t* sK = sQ + NP * 64;
  uint8_t* sV = sK + NP * 64;
  uint8_t* sD = sV + NP * 64;
  AbTok* tok = reinterpret_cast<AbTok*>(sD + NP * 64);               // [NP]
  float* tab = reinterpret_cast<float*>(tok + NP);                   // [L]  table * log2 e of the current head
  float* dtab = tab + L;                                             // [L]  gradient accumulator of the current head
  int* itab = reinterpret_cast<int*>(dtab + L);                      // [L]  this unit's table gradient in 16.16 fixed point (below)
  int* work_ctr = itab + L;                                          // dynamic work-list cursor of the current unit
  int* umax = work_ctr + 1;                                          // [2] bit patterns of max |dO|, max |V| of the current unit

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int nwin = p.win.B * p.win.nwd * p.win.nwh * p.win.nww;
  const bool need_mask = (p.win.sd | p.win.sh | p.win.sw) != 0;
  const int rc = rel_const(p.win);
  const int u_begin = static_cast<int>(1LL * units * blockIdx.x / gridDim.x);
  const int u_end = static_cast<int>(1LL * units * (blockIdx.x + 1) / gridDim.x);
  int cur_head = -1;
  // Shared-memory fp32 atomicAdd compiles to an LDS / FADD / ATOMS.CAST.SPIN retry loop (ncu source page: those loops were the top
  // stall sites, and neighbouring lanes hit the SAME table entry); only 32-bit integer ATOMS.ADD is native.  The per-unit table
  // gradient is therefore accumulated in fixed point and folded into the fp32 table after each unit.  The scale is chosen per unit
  // from a rigorous bound: |dZ| <= |dP| + |delta| <= 64 max|dO| max|V| and an entry receives at most N terms, so
  // scale = 2^30 / (64 N max|dO| max|V|) cannot overflow int32 and keeps ~1e-7 of the bound as resolution (order-independent sums).
  for (int i = threadIdx.x; i < L; i += blockDim.x) itab[i] = 0;

  for (int u = u_begin; u < u_end; ++u) {
    const int head = u / nwin, win = u - head * nwin;
    const long long row0 = static_cast<long long>(win) * N;
    __syncthreads();                                       // previous unit finished with every buffer
    if (threadIdx.x == 0) { *work_ctr = 0; umax[0] = 0; umax[1] = 0; }
    if (head != cur_head) {
      if (cur_head >= 0 && p.dtable_t)
        for (int i = threadIdx.x; i < L; i += blockDim.x) atomicAdd(p.dtable_t + static_cast<long long>(cur_head) * L + i, dtab[i]);
      for (int i = threadIdx.x; i < L; i += blockDim.x) {
        tab[i] = __ldg(p.table_t + static_cast<long long>(head) * L + i) * AB_LOG2E;
        dtab[i] = 0.f;
      }
      cur_head = head;
    }
    // ---- stage Q, K, V, dO (rows >= N zero-filled), zero the dQ accumulator, per-token codes / region ids
    for (int i = threadIdx.x; i < NP * 16; i += blockDim.x) {
      const int row = i >> 4, which = (i >> 2) & 3, ch = i & 3;
      const bool in = row < N;
      const long long r = row0 + (in ? row : 0);
      const __nv_bfloat16* src = (which < 3) ? p.qkv + r * (3 * C) + which * C + head * AB_HD + ch * 8
                                             : p.dout + r * C + head * AB_HD + ch * 8;
      cp_async_16(ab_smem + which * NP * 64 + ab_off(row, ch), src, in);
    }
    cp_async_commit();
    for (int i = threadIdx.x; i < NP; i += blockDim.x) {
      AbTok a;
      a.code = 0; a.rid = -1; a.lse = 0.f; a.delta = 0.f;
      if (i < N) {
        const WinTok w = win_token(p.win, row0 + i);
        a.code = w.code;
        a.rid = w.rid;
        if (p.lse) a.lse = __ldg(p.lse + (row0 + i) * p.nH + head);      // saved by the forward kernel: pass 0 is skipped
      }
      tok[i] = a;
    }
    cp_async_wait<0>();
    __syncthreads();
    // ---- unit maxima of |dO| and |V| for the fixed-point scale of the table gradient
    {
      float mdo = 0.f, mv = 0.f;
      for (int i = threadIdx.x; i < N * 4; i += blockDim.x) {
        const uint4 a = *reinterpret_cast<const uint4*>(sD + ab_off(i >> 2, i & 3));
        const uint4 b = *reinterpret_cast<const uint4*>(sV + ab_off(i >> 2, i & 3));
        const uint32_t aa[4] = {a.x, a.y, a.z, a.w}, bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 x = unpack_bf16x2(aa[j]), y = unpack_bf16x2(bb[j]);
          mdo = fmaxf(mdo, fmaxf(fabsf(x.x), fabsf(x.y)));
          mv = fmaxf(mv, fmaxf(fabsf(y.x), fabsf(y.y)));
        }
      }
      mdo = warp_max(mdo);
      mv = warp_max(mv);
      if (lane == 0) {       // non-negative floats order like their bit patterns
        atomicMax(umax, __float_as_int(mdo));
        atomicMax(umax + 1, __float_as_int(mv));
      }
    }
    // ---- delta_i = dO_i . O_i  (O from global: 64 contiguous bytes per row)
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      const uint4* o4 = reinterpret_cast<const uint4*>(p.out + (row0 + i) * C + head * AB_HD);
      float acc = 0.f;
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const uint4 a = __ldg(o4 + ch);
        const uint4 b = *reinterpret_cast<const uint4*>(sD + ab_off(i, ch));
        const uint32_t aa[4] = {a.x, a.y, a.z, a.w}, bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 x = unpack_bf16x2(aa[j]), y = unpack_bf16x2(bb[j]);
          acc += x.x * y.x + x.y * y.y;
        }
      }
      tok[i].delta = acc;
    }
    // ---- pass 0: log2-sum-exp2 of every score row (warp = 16 query rows, all keys)
    for (int qt = warp; qt < (p.lse ? 0 : NP / 16); qt += AB_WARPS) {
      const int i0 = qt * 16;
      uint32_t qf[2][4];
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) ldmatrix_x4(qf[ks], sQ + ab_off(i0 + (lane & 7) + ((lane >> 3) & 1) * 8, 2 * ks + (lane >> 4)));
      const AbTok q0 = tok[i0 + g], q1 = tok[i0 + g + 8];
      const float* tq0 = tab + q0.code + rc;
      const float* tq1 = tab + q1.code + rc;
      float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
      for (int j0 = 0; j0 < NP; j0 += 8) {
        uint32_t kf[4];
        ldmatrix_x4(kf, sK + ab_off(j0 + (lane & 7), lane >> 3));
        float s[4] = {0.f, 0.f, 0.f, 0.f};
        mma_bf16_16816(s, qf[0], kf[0], kf[1]);
        mma_bf16_16816(s, qf[1], kf[2], kf[3]);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int j = j0 + 2 * t + e;
          if (j < N) {
            const AbTok kj = tok[j];
            s[e] += tq0[-kj.code];
            s[2 + e] += tq1[-kj.code];
            if (need_mask) {
              if (kj.rid != q0.rid) s[e] += AB_MASKV;
              if (kj.rid != q1.rid) s[2 + e] += AB_MASKV;
            }
          } else {
            s[e] = -INFINITY;
            s[2 + e] = -INFINITY;
          }
        }
        const float n0 = fmaxf(m0, fmaxf(s[0], s[1])), n1 = fmaxf(m1, fmaxf(s[2], s[3]));
        if (n0 > -INFINITY) { l0 = l0 * ab_ex2(m0 - n0) + ab_ex2(s[0] - n0) + ab_ex2(s[1] - n0); m0 = n0; }
        if (n1 > -INFINITY) { l1 = l1 * ab_ex2(m1 - n1) + ab_ex2(s[2] - n1) + ab_ex2(s[3] - n1); m1 = n1; }
      }
      // merge the four lanes of a quad (each saw a quarter of the keys)
#pragma unroll
      for (int o = 1; o <= 2; o <<= 1) {
        const float om0 = __shfl_xor_sync(0xffffffffu, m0, o), ol0 = __shfl_xor_sync(0xffffffffu, l0, o);
        const float om1 = __shfl_xor_sync(0xffffffffu, m1, o), ol1 = __shfl_xor_sync(0xffffffffu, l1, o);
        const float n0 = fmaxf(m0, om0), n1 = fmaxf(m1, om1);
        l0 = (m0 > -INFINITY ? l0 * ab_ex2(m0 - n0) : 0.f) + (om0 > -INFINITY ? ol0 * ab_ex2(om0 - n0) : 0.f);
        l1 = (m1 > -INFINITY ? l1 * ab_ex2(m1 - n1) : 0.f) + (om1 > -INFINITY ? ol1 * ab_ex2(om1 - n1) : 0.f);
        m0 = n0;
        m1 = n1;
      }
      if (t == 0) {
        tok[i0 + g].lse = m0 + log2f(l0);
        tok[i0 + g + 8].lse = m1 + log2f(l1);
      }
    }
    __syncthreads();
    // ---- main pass (items 0 .. T-1: a warp owns a 16-key tile) and pass 2 (items T .. 2T-1: a warp owns 16 query rows) share one
    //      dynamically scheduled work list: the two passes are independent of each other, and T = 25 tiles over 16 warps would
    //      otherwise idle 7 warps for half of each pass (ncu: barrier was the second largest stall reason)
    const int T = NP / 16;
    const float ubound = 64.0f * static_cast<float>(N) * __int_as_float(umax[0]) * __int_as_float(umax[1]);
    const float fix = (ubound > 0.f && isfinite(ubound)) ? 1073741824.0f / ubound : 1.0f;
    for (;;) {
      int item = 0;
      if (lane == 0) item = atomicAdd(work_ctr, 1);
      item = __shfl_sync(0xffffffffu, item, 0);
      if (item >= 2 * T) break;
      if (item < T) {
      const int jt = item;
      const int j0 = jt * 16;
      uint32_t kA[2][4], vA[2][4];
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        ldmatrix_x4(kA[ks], sK + ab_off(j0 + (lane & 7) + ((lane >> 3) & 1) * 8, 2 * ks + (lane >> 4)));
        ldmatrix_x4(vA[ks], sV + ab_off(j0 + (lane & 7) + ((lane >> 3) & 1) * 8, 2 * ks + (lane >> 4)));
      }
      const AbTok k0 = tok[j0 + g], k1 = tok[j0 + g + 8];
      const bool kv0 = j0 + g < N, kv1 = j0 + g + 8 < N;
      float dK[4][4], dV[4][4];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) { dK[a][b] = 0.f; dV[a][b] = 0.f; }

      for (int qb = 0; qb < NP / 16; ++qb) {
        uint32_t pP[2][2], pZ[2][2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int i0 = qb * 16 + h * 8;
          uint32_t qf[4], df[4];
          ldmatrix_x4(qf, sQ + ab_off(i0 + (lane & 7), lane >> 3));
          ldmatrix_x4(df, sD + ab_off(i0 + (lane & 7), lane >> 3));
          float s[4] = {0.f, 0.f, 0.f, 0.f}, dp[4] = {0.f, 0.f, 0.f, 0.f};
          mma_bf16_16816(s, kA[0], qf[0], qf[1]);
          mma_bf16_16816(s, kA[1], qf[2], qf[3]);
          mma_bf16_16816(dp, vA[0], df[0], df[1]);
          mma_bf16_16816(dp, vA[1], df[2], df[3]);
          float pv[4], zv[4];
#pragma unroll
          for (int e = 0; e < 2; ++e) {            // query i0 + 2t + e
            const int i = i0 + 2 * t + e;
            const AbTok qi = tok[i];
            const bool iv = i < N;
            const int ib = qi.code + rc;
#pragma unroll
            for (int r = 0; r < 2; ++r) {          // key j0 + g + 8r
              const AbTok& kj = r ? k1 : k0;
              const bool ok = iv && (r ? kv1 : kv0);
              const int idx = ok ? ib - kj.code : 0;
              float z = s[2 * r + e] + tab[idx] - qi.lse;
              if (need_mask && kj.rid != qi.rid) z += AB_MASKV;
              const float pr = ok ? ab_ex2(z) : 0.f;
              const float dz = pr * (dp[2 * r + e] - qi.delta);
              pv[2 * r + e] = pr;
              zv[2 * r + e] = dz;
              if (ok && p.dtable_t) atomicAdd(itab + idx, __float2int_rn(dz * fix));
            }
          }
          pP[h][0] = pack_bf16x2(pv[0], pv[1]);
          pP[h][1] = pack_bf16x2(pv[2], pv[3]);
          pZ[h][0] = pack_bf16x2(zv[0], zv[1]);
          pZ[h][1] = pack_bf16x2(zv[2], zv[3]);
        }
        // dV += P^T dO, dK += dZ^T Q   (A = 16 keys x 16 queries from the two accumulator halves)
        const uint32_t aP[4] = {pP[0][0], pP[0][1], pP[1][0], pP[1][1]};
        const uint32_t aZ[4] = {pZ[0][0], pZ[0][1], pZ[1][0], pZ[1][1]};
#pragma unroll
        for (int dpair = 0; dpair < 2; ++dpair) {
          uint32_t bf[4];
          ldmatrix_x4_trans(bf, sD + ab_off(qb * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, dpair * 2 + (lane >> 4)));
          mma_bf16_16816(dV[dpair * 2 + 0], aP, bf[0], bf[1]);
          mma_bf16_16816(dV[dpair * 2 + 1], aP, bf[2], bf[3]);
          ldmatrix_x4_trans(bf, sQ + ab_off(qb * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, dpair * 2 + (lane >> 4)));
          mma_bf16_16816(dK[dpair * 2 + 0], aZ, bf[0], bf[1]);
          mma_bf16_16816(dK[dpair * 2 + 1], aZ, bf[2], bf[3]);
        }
      }
      // dy_k = dZ^T q' / log2 e  (q' = y_q hd^-0.5 log2 e),  dy_v = P^T dO
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int j = j0 + g + 8 * r;
        if (j >= N) continue;
        __nv_bfloat16* dst = p.dqkv + (row0 + j) * (3 * C) + head * AB_HD + 2 * t;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          *reinterpret_cast<uint32_t*>(dst + C + nt * 8) = pack_bf16x2(dK[nt][2 * r] * (1.0f / AB_LOG2E), dK[nt][2 * r + 1] * (1.0f / AB_LOG2E));
          *reinterpret_cast<uint32_t*>(dst + 2 * C + nt * 8) = pack_bf16x2(dV[nt][2 * r], dV[nt][2 * r + 1]);
        }
      }
      } else {
      // ---- pass 2: dy_q = hd^-0.5 dZ K with a warp OWNING 16 query rows (S, dP, dZ recomputed; dQ accumulates in registers --
      //      reducing dQ across the key-owning warps of the main pass with shared fp32 atomics cost more than this recomputation)
      const int qt = item - T;
      const int i0 = qt * 16;
      uint32_t qf[2][4], df[2][4];
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        ldmatrix_x4(qf[ks], sQ + ab_off(i0 + (lane & 7) + ((lane >> 3) & 1) * 8, 2 * ks + (lane >> 4)));
        ldmatrix_x4(df[ks], sD + ab_off(i0 + (lane & 7) + ((lane >> 3) & 1) * 8, 2 * ks + (lane >> 4)));
      }
      const AbTok q0 = tok[i0 + g], q1 = tok[i0 + g + 8];
      const float* tq0 = tab + q0.code + rc;
      const float* tq1 = tab + q1.code + rc;
      float dQ[4][4];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) dQ[a][b] = 0.f;
      for (int jb = 0; jb < NP / 16; ++jb) {
        uint32_t aZ[4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int j0 = jb * 16 + h * 8;
          uint32_t kf[4], vf[4];
          ldmatrix_x4(kf, sK + ab_off(j0 + (lane & 7), lane >> 3));
          ldmatrix_x4(vf, sV + ab_off(j0 + (lane & 7), lane >> 3));
          float s[4] = {0.f, 0.f, 0.f, 0.f}, dp[4] = {0.f, 0.f, 0.f, 0.f};
          mma_bf16_16816(s, qf[0], kf[0], kf[1]);
          mma_bf16_16816(s, qf[1], kf[2], kf[3]);
          mma_bf16_16816(dp, df[0], vf[0], vf[1]);
          mma_bf16_16816(dp, df[1], vf[2], vf[3]);
          float zv[4];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int j = j0 + 2 * t + e;
            const AbTok kj = tok[j];
            const bool ok = j < N;
            float z0 = s[e] + tq0[-kj.code] - q0.lse, z1 = s[2 + e] + tq1[-kj.code] - q1.lse;
            if (need_mask) {
              if (kj.rid != q0.rid) z0 += AB_MASKV;
              if (kj.rid != q1.rid) z1 += AB_MASKV;
            }
            zv[e] = ok ? ab_ex2(z0) * (dp[e] - q0.delta) : 0.f;
            zv[2 + e] = ok ? ab_ex2(z1) * (dp[2 + e] - q1.delta) : 0.f;
          }
          aZ[2 * h] = pack_bf16x2(zv[0], zv[1]);
          aZ[2 * h + 1] = pack_bf16x2(zv[2], zv[3]);
        }
#pragma unroll
        for (int dpair = 0; dpair < 2; ++dpair) {
          uint32_t bf[4];
          ldmatrix_x4_trans(bf, sK + ab_off(jb * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, dpair * 2 + (lane >> 4)));
          mma_bf16_16816(dQ[dpair * 2 + 0], aZ, bf[0], bf[1]);
          mma_bf16_16816(dQ[dpair * 2 + 1], aZ, bf[2], bf[3]);
        }
      }
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int i = i0 + g + 8 * r;
        if (i >= N) continue;
        __nv_bfloat16* dst = p.dqkv + (row0 + i) * (3 * C) + head * AB_HD + 2 * t;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
          *reinterpret_cast<uint32_t*>(dst + nt * 8) = pack_bf16x2(dQ[nt][2 * r] * p.qscale, dQ[nt][2 * r + 1] * p.qscale);
      }
      }
    }
    __syncthreads();
    if (p.dtable_t)
      for (int i = threadIdx.x; i < L; i += blockDim.x) {
        dtab[i] += static_cast<float>(itab[i]) / fix;
        itab[i] = 0;
      }
  }
  __syncthreads();
  if (cur_head >= 0 && p.dtable_t)
    for (int i = threadIdx.x; i < L; i += blockDim.x) atomicAdd(p.dtable_t + static_cast<long long>(cur_head) * L + i, dtab[i]);
}

int attn_bwd_impl_setting(int set) {
  static int impl = -1;
  if (impl < 0) {
    // "mma" = mma.sync kernel only, "tc" = attn_bwd_tc.cu where it applies (= auto), "tc2" = attn_bwd_tc2.cu wherever it applies
    const char* e = getenv("LAVT_ATTN_BWD_IMPL");
    impl = !e ? 0 : e[0] == 'm' ? 1 : (e[0] == 't' && e[1] == 'c' && e[2] == '2') ? 3 : e[0] == 't' ? 2 : 0;
  }
  const int prev = impl;
  if (set >= 0) impl = set <= 3 ? set : 0;
  return prev;
}

static size_t ab_smem_bytes(const AttnBwdParams& p) {
  const int NP = (p.win.N + 15) / 16 * 16;
  return static_cast<size_t>(NP) * 64 * 4 + static_cast<size_t>(NP) * sizeof(AbTok) + static_cast<size_t>(p.L) * 12 + 32;
}

AttnBwdKernel window_attn_bwd_choose(const AttnBwdParams& p) {
  const WinGeom& w = p.win;
  if (p.C != p.nH * AB_HD || w.N <= 0 || w.N != w.wd * w.wh * w.ww) return AttnBwdKernel::NONE;
  const int impl = attn_bwd_impl_setting(-1);
  if (impl == 3 && window_attn_bwd_tc2_supported(p)) return AttnBwdKernel::TC2;
  if (impl != 1 && window_attn_bwd_tc_supported(p)) return AttnBwdKernel::TC;
  if (ab_smem_bytes(p) <= 227 * 1024) return AttnBwdKernel::MMA;
  if (impl != 1 && window_attn_bwd_tc2_supported(p)) return AttnBwdKernel::TC2;
  return AttnBwdKernel::NONE;
}

long long window_attn_bwd_workspace_floats(const AttnBwdParams& p) {
  return window_attn_bwd_choose(p) == AttnBwdKernel::TC2 ? window_attn_bwd_tc2_workspace_floats(p) : 0;
}

int window_attn_bwd_dispatch(const AttnBwdParams& p, float* workspace, long long workspace_floats, cudaStream_t st) {
  const WinGeom& w = p.win;
  LAVT_REQUIRE(p.C == p.nH * AB_HD, "attention backward: head_dim must be 32 (C=%d, heads=%d)", p.C, p.nH);
  LAVT_REQUIRE(w.N > 0 && w.N == w.wd * w.wh * w.ww, "attention backward: bad window geometry");
  const AttnBwdKernel k = window_attn_bwd_choose(p);
  if (k == AttnBwdKernel::TC) return window_attn_bwd_tc_dispatch(p, st);
  if (k == AttnBwdKernel::TC2) return window_attn_bwd_tc2_dispatch(p, workspace, workspace_floats, st);
  const size_t smem = ab_smem_bytes(p);
  LAVT_REQUIRE(k == AttnBwdKernel::MMA, "attention backward: no kernel for a window of %d tokens (table %d, %s): the mma.sync kernel "
               "needs %zu B of shared memory, the tcgen05 kernels need 16 ... 1152 tokens and the forward's saved lse%s", w.N, p.L,
               p.lse ? "lse saved" : "no lse", smem, attn_bwd_impl_setting(-1) == 1 ? " (mma.sync only was selected)" : "");
  const int NP = (w.N + 15) / 16 * 16;
  static size_t configured = 0;
  if (smem > configured) {
    LAVT_CUDA(cudaFuncSetAttribute(window_attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    configured = smem;
  }
  const int nwin = w.B * w.nwd * w.nwh * w.nww;
  const long long units = 1LL * nwin * p.nH;
  LAVT_REQUIRE(units < (1LL << 30), "attention backward: too many (window, head) units");
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int grid = static_cast<int>(units < sms ? units : sms);
  window_attn_bwd_kernel<<<grid, AB_WARPS * 32, smem, st>>>(p, NP, static_cast<int>(units));
  LAVT_LAUNCH_CHECK("window_attn_bwd_kernel");
  return LAVT_OK;
}

}  // namespace lavt
