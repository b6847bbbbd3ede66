// bf16 mixed-precision version of the training GEMM (seqpan_t_gemm_bf16) on 5th-generation tensor cores (sm_100a).
// Same contract as seqpan_t_gemm (train_ops.cu): C[b0,b1] = alpha * A.B + bias + beta * C over strided fp32 operands, two
// batch dims, split-K.  Every element of A and B is rounded to bf16 (round-to-nearest-even) on its way into shared memory;
// the products accumulate in fp32 in TMEM; C, bias, alpha and beta stay fp32.
//
// One CTA of 128 threads computes one 128 x BN tile of one (batch, K-split) slice:
//   * all four warps stage a 64-wide k-block of A ([128 rows][64 k]) and B ([BN rows][64 k]) with plain global loads along
//     the operand's unit-stride dimension, round to bf16 and store K-major 128-byte-swizzled tiles (make_sw128_desc).  An
//     operand whose unit stride runs along M / N (gᵀ of dW, row-major B of dx = g.W and P.V) is transposed on the way: each
//     thread gathers the 8 k-values of one row -- lanes take consecutive rows, so every global load is coalesced -- and
//     writes them as one 16-byte chunk.  No cast pass, no TMA: operands need no alignment and no tensor map per call.
//   * thread 0 issues UMMA 128xBNx16 (kind::f16) on the staged k-block and commits to that stage's barrier; two stages, so
//     the staging of k-block kb + 1 overlaps the MMAs of kb.  Edges (M, N, K) are zero-padded in shared memory.
//   * epilogue: tcgen05.ld (one TMEM lane = one output row per thread), transposed through shared memory so that each warp
//     stores 32 consecutive columns of a row at once; alpha, bias (K-split 0 only), beta; atomicAdd when split-K.  The
//     deterministic entry point (seqpan_t_gemm_bf16_det) instead stores each K-split's raw tile to scratch [split][M][N] and
//     leaves alpha, bias and beta to the ordered reduction of train_ops.cu.
// No synchronisation and no allocation on the host side: TrainStep(graph=True) captures it like the fp32 kernel.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "tc_common.cuh"
#include "train_ops.cuh"

using namespace tcx;

namespace {

constexpr int TB_M = 128, TB_K = 64;              // BK bf16 = 128 bytes = one swizzle span
constexpr int TB_THREADS = 128;
constexpr int TB_STAGE_A = TB_M * TB_K * 2;       // 16 KB
constexpr int TB_STAGE_B = 128 * TB_K * 2;        // 16 KB (BN <= 128)
constexpr int TB_STAGES = 2;
constexpr int TB_TMEM_COLS = 128;
constexpr int TB_SMEM = 1024 + TB_STAGES * (TB_STAGE_A + TB_STAGE_B) + 64;

struct TbParams {
  SeqpanGemm g;
  int bn;              // N tile: multiple of 16, <= 128
  int split;
  long long kchunk;    // K range of one split: multiple of TB_K
  int a_kmaj, b_kmaj;  // the operand has unit stride along K
  int a_vec, b_vec;    // ... and every row start is 16-byte aligned: 8 k-values = two float4 loads
  float* part;         // deterministic split-K: raw partial tiles [split][M][N] instead of C (NULL: write / add into C)
};

// One k-block [k0, min(k0 + 64, kend)) of an operand with `rows` tile rows (rows_valid of them inside the matrix): element
// (r, k) at src[r * rs + k * ks].  Writes every chunk of the tile, zeros outside the matrix.
template <int G>
__device__ __forceinline__ void stage_kblock(uint32_t dst, const float* __restrict__ src, long long rs, long long ks, int rows,
                                             long long rows_valid, long long k0, long long kend, bool kmaj, bool vec) {
  const int nch = rows * 8;   // 16-byte bf16 chunks: 8 per row
#pragma unroll 1
  for (int c0 = threadIdx.x; c0 < nch; c0 += G * TB_THREADS) {
    float v[G][8];
#pragma unroll
    for (int i = 0; i < G; ++i) {
      const int c = c0 + i * TB_THREADS;
      // K-major source: 8 lanes walk the k-chunks of one row; otherwise lanes walk consecutive rows at fixed k
      const int r = kmaj ? (c >> 3) : (c % rows), kc = kmaj ? (c & 7) : (c / rows);
      const long long k = k0 + kc * 8;
      const bool rok = c < nch && r < rows_valid;
      const float* p = src + (long long)r * rs + k * ks;
      if (vec && rok && k + 8 <= kend) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(p)), y = __ldg(reinterpret_cast<const float4*>(p + 4));
        v[i][0] = x.x; v[i][1] = x.y; v[i][2] = x.z; v[i][3] = x.w;
        v[i][4] = y.x; v[i][5] = y.y; v[i][6] = y.z; v[i][7] = y.w;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[i][j] = (rok && k + j < kend) ? __ldg(p + j * ks) : 0.f;
      }
    }
#pragma unroll
    for (int i = 0; i < G; ++i) {
      const int c = c0 + i * TB_THREADS;
      if (c >= nch) break;
      const int r = kmaj ? (c >> 3) : (c % rows), kc = kmaj ? (c & 7) : (c / rows);
      st_shared_v4_nc(dst + sw128_chunk_offset<0>(r, kc * 8), pack_bf16(v[i][0], v[i][1]), pack_bf16(v[i][2], v[i][3]),
                      pack_bf16(v[i][4], v[i][5]), pack_bf16(v[i][6], v[i][7]));
    }
  }
}

__global__ void __launch_bounds__(TB_THREADS) t_gemm_bf16_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                                                 float* __restrict__ C, const float* __restrict__ bias,
                                                                 const TbParams p) {
  const SeqpanGemm& g = p.g;
  const int z = blockIdx.z;
  const int ks = z % p.split, bz = z / p.split;
  const int b1 = bz % g.batch1, b0 = bz / g.batch1;
  const long long kbeg = ks * p.kchunk, kend = min((long long)g.K, kbeg + p.kchunk);
  const int nkb = kbeg < kend ? (int)((kend - kbeg + TB_K - 1) / TB_K) : 0;
  const bool add_bias = bias && ks == 0;
  if (nkb == 0 && p.split > 1 && !add_bias && !p.part) return;   // an empty K-split adds nothing (its partial tile is zeros)
  A += b0 * g.a_b0 + b1 * g.a_b1;
  B += b0 * g.b_b0 + b1 * g.b_b1;
  C += b0 * g.c_b0 + b1 * g.c_b1;
  const long long m0 = (long long)blockIdx.y * TB_M, n0 = (long long)blockIdx.x * p.bn;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;   // 128-byte-swizzled tiles need 1024-byte alignment
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t a_smem = base, b_smem = base + TB_STAGES * TB_STAGE_A;
  uint8_t* tail = gen + TB_STAGES * (TB_STAGE_A + TB_STAGE_B);
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail);              // empty[TB_STAGES], tmem_full
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tail + 8 * (TB_STAGES + 1));
  const uint32_t empty0 = smem_u32(bars), tfull = smem_u32(bars + TB_STAGES);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < TB_STAGES; ++s) mbar_init(empty0 + 8 * s, 1);
    mbar_init(tfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TB_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_d = *reinterpret_cast<volatile uint32_t*>(tmem_slot);

  const uint32_t idesc = make_idesc(TB_M, p.bn);
  const uint64_t ad0 = make_sw128_desc(a_smem), bd0 = make_sw128_desc(b_smem);
#pragma unroll 1
  for (int kb = 0; kb < nkb; ++kb) {
    const int s = kb & 1;
    if (kb >= TB_STAGES) mbar_wait(empty0 + 8 * s, ((kb >> 1) - 1) & 1);   // the MMAs of k-block kb - 2 have read stage s
    const long long k0 = kbeg + (long long)kb * TB_K;
    stage_kblock<8>(a_smem + s * TB_STAGE_A, A + m0 * g.a_rs, g.a_rs, g.a_cs, TB_M, g.M - m0, k0, kend, p.a_kmaj, p.a_vec);
    stage_kblock<8>(b_smem + s * TB_STAGE_B, B + n0 * g.b_cs, g.b_cs, g.b_rs, p.bn, g.N - n0, k0, kend, p.b_kmaj, p.b_vec);
    fence_proxy_async();          // st.shared -> visible to the tensor core's operand reads
    __syncthreads();
    if (threadIdx.x == 0) {
      tcgen05_fence_after();
      const uint64_t ad = desc_add(ad0, s * TB_STAGE_A), bd = desc_add(bd0, s * TB_STAGE_B);
#pragma unroll
      for (int k = 0; k < TB_K / 16; ++k)   // UMMA_K = 16 bf16 = 32 bytes inside the 128-byte swizzle span
        umma_bf16(tmem_d, desc_add(ad, k * 32), desc_add(bd, k * 32), idesc, (kb | k) != 0);
      umma_commit(empty0 + 8 * s);
      if (kb == nkb - 1) umma_commit(tfull);
    }
  }

  // ---- epilogue: warp w owns TMEM lanes (tile rows) 32w..32w+31; 32-column chunks are transposed through shared memory so
  // that lane = column for the global accesses (coalesced along a row-major C) ----
  if (nkb > 0) {
    mbar_wait(tfull, 0);
    tcgen05_fence_after();
  }
  float* stg = reinterpret_cast<float*>(gen) + warp * (32 * 33);   // aliases stage 0: every MMA has completed
  const long long mrow = m0 + warp * 32;
#pragma unroll 1
  for (int c = 0; c < (p.bn + 31) / 32; ++c) {
    uint32_t r[32];
    if (nkb > 0) {
      tmem_ld32(tmem_d + ((uint32_t)(warp * 32) << 16) + c * 32, r);
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) r[j] = 0u;
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) stg[lane * 33 + j] = __uint_as_float(r[j]);
    __syncwarp();
    const int jn = c * 32 + lane;
    const long long n = n0 + jn;
    const bool nok = jn < p.bn && n < g.N;
    const float bv = (add_bias && nok) ? __ldg(bias + n) : 0.f;
#pragma unroll 4
    for (int i = 0; i < 32; ++i) {
      const long long m = mrow + i;
      if (!nok || m >= g.M) continue;
      if (p.part) { p.part[(ks * g.M + m) * g.N + n] = stg[i * 33 + lane]; continue; }
      float* cp = C + m * g.c_rs + n * g.c_cs;
      const float v = g.alpha * stg[i * 33 + lane] + bv;
      if (p.split > 1) atomicAdd(cp, v);                         // C was pre-scaled by beta (0: zeroed) by the launcher
      else *cp = v + (g.beta != 0.f ? g.beta * *cp : 0.f);
    }
    __syncwarp();
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(TB_TMEM_COLS) : "memory");
  }
}

bool aligned16(const float* base, long long rs, long long s0, long long s1) {
  return ((uintptr_t)base & 15) == 0 && rs % 4 == 0 && s0 % 4 == 0 && s1 % 4 == 0;
}

}  // namespace

// part == NULL: seqpan_t_gemm_bf16; otherwise the K-splits of a split-K product store their raw tiles to `part`
static int t_gemm_bf16_launch(const float* A, const float* B, float* C, const float* bias, const SeqpanGemm* gp, int split, long long gz,
                       float* part, cudaStream_t st) {
  static SqSmemOptIn optin;
  if (optin.ensure((const void*)t_gemm_bf16_kernel, TB_SMEM) != cudaSuccess) return tcheck();
  TbParams p;
  p.g = *gp;
  const SeqpanGemm& g = p.g;
  p.split = split;
  p.part = part;
  p.kchunk = ((g.K + split - 1) / split + TB_K - 1) / TB_K * TB_K;
  // N tile: the smallest legal UMMA N that covers N, at most 128; halved to 64 when 128-wide tiles leave most SMs idle
  const long long mt = (g.M + TB_M - 1) / TB_M;
  p.bn = (int)(g.N >= 128 ? 128 : (g.N + 15) / 16 * 16);
  if (p.bn == 128 && mt * ((g.N + 127) / 128) * gz < 148) p.bn = 64;
  p.a_kmaj = g.a_cs == 1;
  p.b_kmaj = g.b_rs == 1;
  p.a_vec = p.a_kmaj && aligned16(A, g.a_rs, g.a_b0, g.a_b1);
  p.b_vec = p.b_kmaj && aligned16(B, g.b_cs, g.b_b0, g.b_b1);
  dim3 grid((unsigned)((g.N + p.bn - 1) / p.bn), (unsigned)mt, (unsigned)gz);
  t_gemm_bf16_kernel<<<grid, TB_THREADS, TB_SMEM, st>>>(A, B, C, bias, p);
  return tcheck();
}

extern "C" int seqpan_t_gemm_bf16(const float* A, const float* B, float* C, const float* bias, const SeqpanGemm* gp, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  int split = 1;
  long long gz = 0;
  const int rc = t_gemm_prepare(A, B, C, gp, st, split, gz);
  if (rc != SEQPAN_OK || gz == 0) return rc;
  return t_gemm_bf16_launch(A, B, C, bias, gp, split, gz, nullptr, st);
}

extern "C" int seqpan_t_gemm_bf16_det(const float* A, const float* B, float* C, const float* bias, const SeqpanGemm* gp,
                                      void* scratch, size_t scratch_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  int split = 1;
  long long gz = 0;
  int rc = t_gemm_prepare(A, B, C, gp, st, split, gz, false);
  if (rc != SEQPAN_OK || gz == 0) return rc;
  if (split == 1) return t_gemm_bf16_launch(A, B, C, bias, gp, split, gz, nullptr, st);   // already one writer per element
  if ((rc = t_gemm_det_check(*gp, scratch, scratch_bytes)) != SEQPAN_OK) return rc;
  if ((rc = t_gemm_bf16_launch(A, B, C, nullptr, gp, split, gz, (float*)scratch, st)) != SEQPAN_OK) return rc;
  return t_gemm_splitk_reduce(C, (const float*)scratch, bias, *gp, split, st);
}
