// CQAttention (models/layers.py:402-437) + its cqa_linear projection on tcgen05 tensor cores, both directions
// (models/SeqPAN.py:73-74), one CTA per (sample, direction).  C = context rows [F,128], Q = query rows [S,128]:
//   S    = (C*w4mlu).Q^T + C.w4C (+) (Q.w4Q)^T            trilinear score             UMMA  [128 x Sp], K = 128
//   S^T  = Q.(C*w4mlu)^T + ...                            the same scores, transposed  UMMA  [128 x Fp], K = 128
//   P1   = exp(S  + mask_q - rowmax)   (rows = context)    row softmax over the query axis   (unnormalised, bf16)
//   P2   = exp(S^T + mask_c - rowmax)  (rows = query)      column softmax of S = row softmax of S^T
//   c2q  = P1.Q / sum1            R = P2.C / sum2          UMMA with Q / C as MN-major B operands (no transposition)
//   q2c  = P1.R / sum1            (= S1.S2^T.C, re-associated; R goes back to shared memory as a bf16 B operand)
//   out  = W.[C, c2q, C*c2q, C*q2c] + b                    4 accumulating UMMAs, the 512-wide concat never exists
// Both softmaxes are thread-per-row sweeps over TMEM (tcgen05.ld): warps 1-4 take the rows of S, warps 5-8 the rows of
// S^T.  Every epilogue splits a row's 128 columns between two warps.  Shared-memory tiles are recycled as their
// consumers retire (5 x 32 KB operand tiles + one 32 KB weight slot).  Needs L <= 128 and T <= 128.
#include <cstdio>

#include "chain_tc.cuh"
#include "tc_common.cuh"

using namespace tcx;

namespace {

constexpr int KBB = 16384;
constexpr int TILE_B = 2 * KBB;
constexpr int CQ_TC_THREADS = 288;
constexpr float MASKV = -1e30f;
constexpr float LOG2E = 1.4426950408889634f;

struct CqTcParams {
  const float* x;       // joint rows [M,128] fp32: B*L video rows, then B*T text rows
  const float* vmask;   // [B,L]
  const float* tmask;   // [B,T]
  const float* w4c[2]; const float* w4q[2]; const float* w4mlu[2]; const float* bias[2];
  float* out[2];        // dir 0: [B*L, ldo[0]] (context = video), dir 1: [B*T, ldo[1]] (context = text)
  int ldo[2];
  int B, L, T;
};

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// bf16 pair of (a, b) and the bf16 pair of the rounding remainders: a ~ hi + lo to ~16 mantissa bits
__device__ __forceinline__ uint32_t pack_hi_lo(float a, float b, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  const float2 f = __bfloat1622float2(h);
  const __nv_bfloat162 l = __floats2bfloat162_rn(a - f.x, b - f.y);
  lo = *reinterpret_cast<const uint32_t*>(&l);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ void store_a16(uint32_t abuf, int row, int col, const float (&v)[16]) {
  st_shared_v4(abuf + sw128_chunk_offset<KBB>(row, col), pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]),
               pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
  st_shared_v4(abuf + sw128_chunk_offset<KBB>(row, col + 8), pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]),
               pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
}

__global__ void __launch_bounds__(CQ_TC_THREADS, 1)
cq_tc_kernel(const __grid_constant__ CUtensorMap tm_w0, const __grid_constant__ CUtensorMap tm_w1, CqTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t Ct = base;                   // C (bf16)                                   A of out, B (MN) of R
  const uint32_t Cw = base + TILE_B;          // C*w4mlu; later R (bf16)                    A of S / B of S^T; B (MN) of q2c
  const uint32_t Qt = base + 2 * TILE_B;      // Q; later C*c2q                              B of S / A of S^T, B (MN) of c2q
  const uint32_t P1 = base + 3 * TILE_B;      // first the bf16 remainders of C*w4mlu; then exp(S) rows; later C*q2c
  const uint32_t P2 = base + 4 * TILE_B;      // first the bf16 remainders of Q; then exp(S^T) rows; later c2q
  const uint32_t Wb = base + 5 * TILE_B;      // weight slot: two k-blocks of cqa_linear's [128,512] matrix
  uint8_t* tail = gen + 6 * TILE_B;
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail);  // 0 wfull, 1 wfree, 2 bar_a, 3 bar_mma
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tail + 64);
  float* fsm = reinterpret_cast<float*>(tail + 128);
  float* sub0 = fsm;          // [128] C.w4C
  float* sub1 = fsm + 128;    // [128] Q.w4Q
  float* cbS = fsm + 256;     // [128] per query column j of S:   sub1[j] + mask_q, -inf beyond S
  float* cbT = fsm + 384;     // [128] per context column i of S^T: sub0[i] + mask_c, -inf beyond F
  float* inv1 = fsm + 512;    // [128] 1 / row sums of P1
  float* inv2 = fsm + 640;    // [128] 1 / row sums of P2
  float* fbias = fsm + 768;   // [128] cqa_linear bias

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x, dir = blockIdx.y;
  const int F = dir == 0 ? p.L : p.T, S = dir == 0 ? p.T : p.L;
  const int Fp = (F + 15) & ~15, Sp = (S + 15) & ~15;
  const long long Mv = (long long)p.B * p.L;
  const long long crow0 = dir == 0 ? (long long)b * p.L : Mv + (long long)b * p.T;
  const long long qrow0 = dir == 0 ? Mv + (long long)b * p.T : (long long)b * p.L;
  const float* cmask = dir == 0 ? p.vmask + (long long)b * p.L : p.tmask + (long long)b * p.T;
  const float* qmask = dir == 0 ? p.tmask + (long long)b * p.T : p.vmask + (long long)b * p.L;

  if (threadIdx.x == 0) {
    mbar_init(smem_u32(bars + 0), 1);
    mbar_init(smem_u32(bars + 1), 1);
    mbar_init(smem_u32(bars + 2), 256);
    mbar_init(smem_u32(bars + 3), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x < 128) fbias[threadIdx.x] = __ldg(p.bias[dir] + threadIdx.x);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  const uint32_t wfull = smem_u32(bars + 0), wfree = smem_u32(bars + 1), bar_a = smem_u32(bars + 2), bar_mma = smem_u32(bars + 3);
  const uint32_t T_S = tmem, T_ST = tmem + 128, T_OUT = tmem + 256;

  if (warp == 0) {
    if (lane == 0) {
      const CUtensorMap* wm = dir == 0 ? &tm_w0 : &tm_w1;
      auto load_w = [&](int kb0) {
        mbar_expect_tx(wfull, TILE_B);
        tma_load_2d(Wb, wm, wfull, kb0 * 64, 0);
        tma_load_2d(Wb + KBB, wm, wfull, (kb0 + 1) * 64, 0);
      };
      // D[128, N] (+)= A-tile (K-major, 128 columns) . B-tile^T (K-major, N rows)
      auto mma_kmajor = [&](uint32_t d, uint32_t a, uint32_t bt, int N, bool acc) {
        const uint32_t idesc = make_idesc(128, N);
        const uint64_t ad = make_sw128_desc(a), bd = make_sw128_desc(bt);
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(d, desc_add(ad, kb * KBB + k * 32), desc_add(bd, kb * KBB + k * 32), idesc,
                      (acc || kb || k) ? 1u : 0u);
      };
      // D[128, 128] = P-tile (K-major, Kp columns) . B-tile (row-major [Kp rows][128] = MN-major)
      auto mma_mnmajor = [&](uint32_t d, uint32_t a, uint32_t bm, int Kp) {
        const uint32_t idesc = make_idesc(128, 128) | IDESC_B_MN_MAJOR;
        const uint64_t ad = make_sw128_desc(a), bd = make_mn_sw128_desc(bm, KBB);
        for (int ks = 0; ks < Kp / 16; ++ks)
          umma_bf16(d, desc_add(ad, (ks >> 2) * KBB + (ks & 3) * 32), desc_add(bd, ks * 2048), idesc, ks ? 1u : 0u);
      };
      load_w(0);
      mbar_wait(bar_a, 0); tcgen05_fence_after();            // Ct, Cw, Qt built
      mma_kmajor(T_S, Cw, Qt, Sp, false);                    // S   = (C*w).Q^T          hi.hi
      mma_kmajor(T_S, Cw, P2, Sp, true);                     //                          + hi.lo  (P2 region = Q remainders)
      mma_kmajor(T_S, P1, Qt, Sp, true);                     //                          + lo.hi  (P1 region = C*w remainders)
      mma_kmajor(T_ST, Qt, Cw, Fp, false);                   // S^T = Q.(C*w)^T
      mma_kmajor(T_ST, P2, Cw, Fp, true);
      mma_kmajor(T_ST, Qt, P1, Fp, true);
      umma_commit(bar_mma);                                  // #0 -> softmaxes
      mbar_wait(wfull, 0);
      mma_kmajor(T_OUT, Ct, Wb, 128, false);                 // out  = W[:, 0:128].C
      umma_commit(wfree);
      mbar_wait(wfree, 0);
      load_w(2);
      mbar_wait(bar_a, 1); tcgen05_fence_after();            // P1, P2 written
      mma_mnmajor(T_S, P1, Qt, Sp);                          // c2q_raw = P1.Q
      mma_mnmajor(T_ST, P2, Ct, Fp);                         // R_raw   = P2.C
      umma_commit(bar_mma);                                  // #1 -> epilogue 1
      mbar_wait(bar_a, 0); tcgen05_fence_after();            // R (in Cw), c2q (in P2), C*c2q (in Qt) written
      mma_mnmajor(T_ST, P1, Cw, Sp);                         // q2c_raw = P1.R
      umma_commit(bar_mma);                                  // #2 -> epilogue 2
      mbar_wait(wfull, 1);
      mma_kmajor(T_OUT, P2, Wb, 128, true);                  // out += W[:, 128:256].c2q
      umma_commit(wfree);
      mbar_wait(wfree, 1);
      load_w(4);
      mbar_wait(wfull, 0);
      mma_kmajor(T_OUT, Qt, Wb, 128, true);                  // out += W[:, 256:384].(C*c2q)
      umma_commit(wfree);
      mbar_wait(wfree, 0);
      load_w(6);
      mbar_wait(bar_a, 1); tcgen05_fence_after();            // C*q2c (in P1) written
      mbar_wait(wfull, 1);
      mma_kmajor(T_OUT, P1, Wb, 128, true);                  // out += W[:, 384:512].(C*q2c)
      umma_commit(bar_mma);                                  // #3 -> final epilogue
    }
  } else {
    const int w8 = warp - 1, q = warp & 3, half = w8 >> 2;
    const int row = q * 32 + lane;
    const uint32_t tq = tmem + ((uint32_t)(q * 32) << 16);
    auto publish = [&]() { tcgen05_fence_before(); fence_proxy_async(); mbar_arrive(bar_a); };
    // ---- load phase: 16 context rows + 16 query rows per warp (coalesced 512-byte rows, 8 loads in flight) ----
    {
      const int col = lane * 4;
      const float4 wc = __ldg(reinterpret_cast<const float4*>(p.w4c[dir] + col));
      const float4 wq = __ldg(reinterpret_cast<const float4*>(p.w4q[dir] + col));
      const float4 wm = __ldg(reinterpret_cast<const float4*>(p.w4mlu[dir] + col));
#pragma unroll 1
      for (int gg = 0; gg < 2; ++gg) {         // gg 0: this warp's 16 context rows; gg 1: its 16 query rows -- all 16 loads in flight
        const bool isq = gg == 1;
        const int n = isq ? S : F;
        const float* src = p.x + (isq ? qrow0 : crow0) * 128 + col;
        float4 xw[16];
#pragma unroll
        for (int i = 0; i < 16; ++i)
          xw[i] = (w8 * 16 + i) < n ? __ldg(reinterpret_cast<const float4*>(src + (long long)(w8 * 16 + i) * 128)) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 ws = isq ? wq : wc;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
        const int r0 = w8 * 16 + hh * 8;
        float d[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = r0 + i;
          const float4 v = xw[hh * 8 + i];
          d[i] = v.x * ws.x + v.y * ws.y + v.z * ws.z + v.w * ws.w;
          const uint32_t off = sw128_chunk_offset<KBB>(r, col & ~7) + (col & 7) * 2;
          // The trilinear scores feed exp(): an absolute score error IS the relative error of the attention weight, and the scores
          // are unscaled 128-term dot products.  Both score operands therefore carry a second bf16 tile with the rounding
          // remainders (hi + lo ~ 16 mantissa bits; S = hi.hi + hi.lo + lo.hi, three accumulating UMMAs).  The remainder tiles
          // live in the P1 / P2 regions, which are dead until the softmax writes them.
          if (isq) {
            uint32_t l0, l1;
            const uint32_t h0 = pack_hi_lo(v.x, v.y, l0), h1 = pack_hi_lo(v.z, v.w, l1);
            st_shared_v2(Qt + off, h0, h1);
            st_shared_v2(P2 + off, l0, l1);
          } else {
            st_shared_v2(Ct + off, pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
            uint32_t l0, l1;
            const uint32_t h0 = pack_hi_lo(v.x * wm.x, v.y * wm.y, l0), h1 = pack_hi_lo(v.z * wm.z, v.w * wm.w, l1);
            st_shared_v2(Cw + off, h0, h1);
            st_shared_v2(P1 + off, l0, l1);
          }
        }
        // 8 row sums over the 32 lanes in 9 shuffles (instead of 8 x 5): halve the rows a lane carries while halving the
        // lanes that share a row (lane bits 4, 3, 2 select the row), then two plain butterfly steps
        {
          const bool h4 = lane & 16, h3 = lane & 8, h2 = lane & 4;
          float e[4], f2[2], g1;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float keep = h4 ? d[i + 4] : d[i], send = h4 ? d[i] : d[i + 4];
            e[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
          }
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const float keep = h3 ? e[i + 2] : e[i], send = h3 ? e[i] : e[i + 2];
            f2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
          }
          {
            const float keep = h2 ? f2[1] : f2[0], send = h2 ? f2[0] : f2[1];
            g1 = keep + __shfl_xor_sync(0xffffffffu, send, 4);
          }
          g1 += __shfl_xor_sync(0xffffffffu, g1, 2);
          g1 += __shfl_xor_sync(0xffffffffu, g1, 1);
          if ((lane & 3) == 0) {
            const int r = r0 + (h4 ? 4 : 0) + (h3 ? 2 : 0) + (h2 ? 1 : 0);
            (isq ? sub1 : sub0)[r] = g1;
          }
        }
        }
      }
    }
    publish();                                               // bar_a #0
    asm volatile("bar.sync 1, 256;" ::: "memory");           // sub0 / sub1 complete
    {
      const int t = w8 * 32 + lane;                          // 0..255
      if (t < 128) {       // column bias of S (query axis): mask_logits adds (1 - m) * -1e30 (models/layers.py:9-12)
        cbS[t] = t < S ? sub1[t] + (1.0f - __ldg(qmask + t)) * MASKV : -INFINITY;
      } else {             // column bias of S^T (context axis)
        const int i = t - 128;
        cbT[i] = i < F ? sub0[i] + (1.0f - __ldg(cmask + i)) * MASKV : -INFINITY;
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    // residual context values of this thread's (row, 64-column half), loaded while the score MMAs run
    float4 cv[16];
    {
      const bool has = row < F;
      const float* src = p.x + (crow0 + row) * 128 + half * 64;
#pragma unroll
      for (int i = 0; i < 16; ++i) cv[i] = has ? __ldg(reinterpret_cast<const float4*>(src + i * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // ---- softmaxes: half 0 = rows of S (context rows, softmax over the query axis), half 1 = rows of S^T ----
    mbar_wait(bar_mma, 0);
    tcgen05_fence_after();
    {
      const int nrow = half == 0 ? F : S, ncol = half == 0 ? Sp : Fp;
      if (q * 32 < nrow) {                                   // warp-uniform: tcgen05.ld is warp-collective
        const uint32_t tcol = half == 0 ? T_S : T_ST;
        const float* cb = half == 0 ? cbS : cbT;
        const float a = half == 0 ? sub0[row] : sub1[row];
        const uint32_t Pt = half == 0 ? P1 : P2;
        const uint32_t tr = tcol + ((uint32_t)(q * 32) << 16);
        float m0 = -INFINITY, m1 = -INFINITY;
        tmem_pipe16_rt(tr, ncol / 16, [&](int c, uint32_t (&r0)[16]) {
#pragma unroll
          for (int j = 0; j < 16; j += 2) {
            m0 = fmaxf(m0, (__uint_as_float(r0[j]) + a) + cb[c * 16 + j]);
            m1 = fmaxf(m1, (__uint_as_float(r0[j + 1]) + a) + cb[c * 16 + j + 1]);
          }
        });
        const float mx = fmaxf(m0, m1);
        float s0 = 0.f, s1 = 0.f;
        tmem_pipe16_rt(tr, ncol / 16, [&](int c, uint32_t (&r0)[16]) {
          float e[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) e[j] = ex2_approx((((__uint_as_float(r0[j]) + a) + cb[c * 16 + j]) - mx) * LOG2E);
#pragma unroll
          for (int j = 0; j < 16; j += 2) { s0 += e[j]; s1 += e[j + 1]; }
          store_a16(Pt, row, c * 16, e);
        });
        (half == 0 ? inv1 : inv2)[row] = 1.0f / (s0 + s1);
      }
    }
    publish();                                               // bar_a #1
    asm volatile("bar.sync 1, 256;" ::: "memory");           // inv1 / inv2 visible to both halves
    // ---- epilogue 1: c2q -> tiles (c2q, C*c2q), R -> bf16 B operand ----
    mbar_wait(bar_mma, 1);
    tcgen05_fence_after();
    {
      // rows beyond F / S hold whatever the unused lanes accumulated (possibly NaN): they are written as exact zeros,
      // because R's padding rows are inside the K extent of the q2c product
      const bool okF = row < F, okS = row < S;
      const float i1 = okF ? inv1[row] : 0.f, i2 = okS ? inv2[row] : 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t ra[16], rb[16];
        tmem_ld16(tq + (T_S - tmem) + half * 64 + c * 16, ra);
        tmem_ld16(tq + (T_ST - tmem) + half * 64 + c * 16, rb);
        tmem_ld_wait();
        float c2q[16], cc[16], rr[16];
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const float4 cx = cv[c * 4 + j4];
          const float xs[4] = {cx.x, cx.y, cx.z, cx.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int j = j4 * 4 + e;
            c2q[j] = okF ? __uint_as_float(ra[j]) * i1 : 0.f;
            cc[j] = xs[e] * c2q[j];
            rr[j] = okS ? __uint_as_float(rb[j]) * i2 : 0.f;
          }
        }
        store_a16(P2, row, half * 64 + c * 16, c2q);
        store_a16(Qt, row, half * 64 + c * 16, cc);
        store_a16(Cw, row, half * 64 + c * 16, rr);
      }
    }
    publish();                                               // bar_a #2
    // ---- epilogue 2: q2c -> tile C*q2c ----
    mbar_wait(bar_mma, 0);
    tcgen05_fence_after();
    {
      const bool okF = row < F;
      const float i1 = okF ? inv1[row] : 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t ra[16];
        tmem_ld16(tq + (T_ST - tmem) + half * 64 + c * 16, ra);
        tmem_ld_wait();
        float cq[16];
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const float4 cx = cv[c * 4 + j4];
          cq[j4 * 4 + 0] = okF ? cx.x * (__uint_as_float(ra[j4 * 4 + 0]) * i1) : 0.f;
          cq[j4 * 4 + 1] = okF ? cx.y * (__uint_as_float(ra[j4 * 4 + 1]) * i1) : 0.f;
          cq[j4 * 4 + 2] = okF ? cx.z * (__uint_as_float(ra[j4 * 4 + 2]) * i1) : 0.f;
          cq[j4 * 4 + 3] = okF ? cx.w * (__uint_as_float(ra[j4 * 4 + 3]) * i1) : 0.f;
        }
        store_a16(P1, row, half * 64 + c * 16, cq);
      }
    }
    publish();                                               // bar_a #3
    // ---- final epilogue: out = acc + bias ----
    mbar_wait(bar_mma, 1);
    tcgen05_fence_after();
    {
      float* dst = p.out[dir] + ((dir == 0 ? (long long)b * p.L : (long long)b * p.T) + row) * p.ldo[dir] + half * 64;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t ra[16];
        tmem_ld16(tq + (T_OUT - tmem) + half * 64 + c * 16, ra);
        tmem_ld_wait();
        if (row < F) {
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            float4 v;
            v.x = __uint_as_float(ra[j4 * 4 + 0]) + fbias[half * 64 + c * 16 + j4 * 4 + 0];
            v.y = __uint_as_float(ra[j4 * 4 + 1]) + fbias[half * 64 + c * 16 + j4 * 4 + 1];
            v.z = __uint_as_float(ra[j4 * 4 + 2]) + fbias[half * 64 + c * 16 + j4 * 4 + 2];
            v.w = __uint_as_float(ra[j4 * 4 + 3]) + fbias[half * 64 + c * 16 + j4 * 4 + 3];
            *reinterpret_cast<float4*>(dst + c * 16 + j4 * 4) = v;
          }
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
  }
}

constexpr size_t CQ_TC_SMEM = 1024 + 6 * TILE_B + 128 + 7 * 128 * sizeof(float);

}  // namespace

bool cq_tc_supported(int L, int T) { return L >= 1 && L <= 128 && T >= 1 && T <= 128; }

int cq_attention_tc(const TcArena& a, const float* x, const float* vmask, const float* tmask, const float* const* w4c,
                    const float* const* w4q, const float* const* w4mlu, const float* const* bias, float* out_v, int ldo_v,
                    float* out_t, int ldo_t, int B, int L, int T, cudaStream_t st) {
  if (!cq_tc_supported(L, T)) return SEQPAN_E_INVALID;
  static SqSmemOptIn optin;
  if (optin.ensure((const void*)cq_tc_kernel, CQ_TC_SMEM) != cudaSuccess) return SEQPAN_E_CUDA;
  CqTcParams p;
  p.x = x; p.vmask = vmask; p.tmask = tmask;
  for (int d = 0; d < 2; ++d) { p.w4c[d] = w4c[d]; p.w4q[d] = w4q[d]; p.w4mlu[d] = w4mlu[d]; p.bias[d] = bias[d]; }
  p.out[0] = out_v; p.out[1] = out_t; p.ldo[0] = ldo_v; p.ldo[1] = ldo_t;
  p.B = B; p.L = L; p.T = T;
  cq_tc_kernel<<<dim3(B, 2), CQ_TC_THREADS, CQ_TC_SMEM, st>>>(*reinterpret_cast<const CUtensorMap*>(a.slot[TC_Q2V_LIN].tmap),
                                                           *reinterpret_cast<const CUtensorMap*>(a.slot[TC_V2Q_LIN].tmap), p);
  return cudaGetLastError() == cudaSuccess ? SEQPAN_OK : SEQPAN_E_CUDA;
}
