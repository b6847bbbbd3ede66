// Fused tcgen05 "chain" kernels of the bf16 mode: a CTA owns 128 rows of the joint row buffer and runs a whole
// chain of row-local 128-wide projections on them without leaving the SM.  Activations between projections live
// in TMEM (fp32 accumulators, 4 x 128 columns) and in shared memory (bf16 operand tiles, 128-byte swizzle);
// weights stream through a 2-slot ring by TMA.  Thread layout: warp 0 = control (one elected thread issues the
// weight TMA loads and every tcgen05.mma), the other warps = workers (TMEM lane = row of the thread): they build
// the first operand tiles cooperatively (coalesced global reads, LayerNorm by warp shuffles) and run every
// epilogue, each of which produces the next operand tile.  Control and workers hand over through two mbarriers
// (operand tiles ready / accumulators ready) whose phases alternate step by step.
// (The DualAttentionBlock post-attention chain, the FEP tail + logit head and the concat + match head live in tail_tc.cu.)
#include "chain_tc.cuh"

#include <cstdio>
#include <cstring>
#include <cstdlib>

#include "tc_common.cuh"

using namespace tcx;

namespace {

constexpr int KBB = 16384;          // one k-block of an operand tile: [128 rows][64 bf16]
constexpr int TILE_B = 2 * KBB;     // [128][128] bf16
constexpr int CB_THREADS = 288;   // warp 0 control + 8 worker warps

__device__ __forceinline__ void mma_tile(uint32_t tmem_d, uint32_t abuf, uint32_t wbuf, uint32_t idesc, bool accumulate) {
  const uint64_t ad = make_sw128_desc(abuf), wd = make_sw128_desc(wbuf);
#pragma unroll
  for (int kb = 0; kb < 2; ++kb)
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma_bf16(tmem_d, desc_add(ad, kb * KBB + k * 32), desc_add(wd, kb * KBB + k * 32), idesc,
                (accumulate || kb || k) ? 1u : 0u);
}

// 16 fp32 values of one row -> bf16 -> operand tile (two 16-byte chunks), swizzled
__device__ __forceinline__ void store_a16(uint32_t abuf, int row, int col, const float (&v)[16]) {
  st_shared_v4(abuf + sw128_chunk_offset<KBB>(row, col), pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]),
               pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
  st_shared_v4(abuf + sw128_chunk_offset<KBB>(row, col + 8), pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]),
               pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
}

// ------------------------------------------------------------------------------------------------------------
// Shared pieces of the chain kernels
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void chain_end(uint32_t tmem, int tmem_cols) {
  tcgen05_fence_before();
  __syncthreads();
  if ((threadIdx.x >> 5) == 0) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(tmem_cols) : "memory");
  }
}

// Cooperative operand construction: the calling warp turns its 32 rows (q*32..q*32+31 of the tile starting at m0)
// of an fp32 [M,128] matrix into bf16 operand tiles: tileA = LN(x; gA,bA) (or plain x when gA == nullptr) and,
// if tileB != 0, tileB = LN(x; gB,bB).  16 coalesced 512-byte row loads are in flight per warp.
template <int ROWS = 32>
__device__ __forceinline__ void rows_to_tiles(const float* __restrict__ x, long long M, long long m0, int rbase, int lane,
                                              float eps, const float* gA, const float* bA, uint32_t tileA,
                                              const float* gB, const float* bB, uint32_t tileB) {
  const int col = lane * 4;
  float4 ga = make_float4(1.f, 1.f, 1.f, 1.f), ba = make_float4(0.f, 0.f, 0.f, 0.f), gb = ga, bb = ba;
  if (gA) { ga = __ldg(reinterpret_cast<const float4*>(gA + col)); ba = __ldg(reinterpret_cast<const float4*>(bA + col)); }
  if (tileB) { gb = __ldg(reinterpret_cast<const float4*>(gB + col)); bb = __ldg(reinterpret_cast<const float4*>(bB + col)); }
#pragma unroll 1
  for (int r0 = 0; r0 < ROWS; r0 += 16) {
    float4 xv[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const long long gr = m0 + rbase + r0 + i;
      xv[i] = gr < M ? __ldg(reinterpret_cast<const float4*>(x + gr * 128 + col)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int r = rbase + r0 + i;
      const float4 v = xv[i];
      const uint32_t off = sw128_chunk_offset<KBB>(r, col & ~7) + (col & 7) * 2;
      if (!gA) {
        st_shared_v2(tileA + off, pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
        continue;
      }
      float mean = v.x + v.y + v.z + v.w;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mean += __shfl_xor_sync(0xffffffffu, mean, o);
      mean *= (1.0f / 128.0f);
      const float dx = v.x - mean, dy = v.y - mean, dz = v.z - mean, dw = v.w - mean;
      float var = dx * dx + dy * dy + dz * dz + dw * dw;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) var += __shfl_xor_sync(0xffffffffu, var, o);
      const float rstd = rsqrtf(var * (1.0f / 128.0f) + eps);
      st_shared_v2(tileA + off, pack_bf16(dx * rstd * ga.x + ba.x, dy * rstd * ga.y + ba.y),
                   pack_bf16(dz * rstd * ga.z + ba.z, dw * rstd * ga.w + ba.w));
      if (tileB)
        st_shared_v2(tileB + off, pack_bf16(dx * rstd * gb.x + bb.x, dy * rstd * gb.y + bb.y),
                     pack_bf16(dz * rstd * gb.z + bb.z, dw * rstd * gb.w + bb.w));
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// LayerNorm + multi-output projection: out_A = LN_A(x) . W_A^T + b_A  (nA 128-wide column tiles) and optionally
// out_B = LN_B(x) . W_B^T + b_B (nB tiles) from ONE read of x.  DualAttentionBlock: LN1 -> query|f_key|f_value and
// LNt -> t_key|t_value (models/layers.py:282-283, 339-344); FeatureEncoderPredict: layer_norm_1 -> in_proj
// (models/layers.py:630-632).  Two TMEM accumulators ping-pong so the epilogue of tile t overlaps the MMA of t+1.
// ------------------------------------------------------------------------------------------------------------
struct ProjLnParams {
  const float* x;
  long long M;
  float eps;
  const float* gA; const float* bA; const float* gB; const float* bB;
  float* outA; float* outB;   // [M, nA*128], [M, nB*128]
  const float* biasA; const float* biasB;
  int nA, nB;
  // optional head-blocked bf16 outputs of the A tiles (q, k, v of nn.MultiheadAttention's in_proj) for the batch-axis
  // attention kernel: tile t -> hb[t][((l*4 + head)*hbB + b) * hb_stride[t] + d], row m = b*hbL + l
  void* hb[3];
  int hb_stride[3];
  int hbL, hbB;
  int out_bf16;          // 1: outA/outB are bf16 row-major matrices (operands of the tcgen05 dual attention)
  const float* hb_mask;  // [B*L] additive key mask: written as column 32 of every k row (column 32 of q rows = 1),
                         // so the tensor core adds the mask:  [q*scale, 1] . [k, mask] = scale q.k + mask
};

__global__ void __launch_bounds__(CB_THREADS)
proj_ln_kernel(const __grid_constant__ CUtensorMap tm_wA, const __grid_constant__ CUtensorMap tm_wB, ProjLnParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t PA = base, PB = base + TILE_B, Wt = base + 2 * TILE_B;
  uint8_t* tail = gen + 3 * TILE_B;
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail);  // 0 wfull, 1 wempty, 2 bar_a, 3/4 tfull[2], 5/6 tfree[2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tail + 64);
  float* fb = reinterpret_cast<float*>(tail + 128);    // biases of all tiles [ntiles][128]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long m0 = (long long)blockIdx.x * 128;
  const int ntiles = p.nA + p.nB;
  for (int i = threadIdx.x; i < ntiles * 128; i += CB_THREADS)
    fb[i] = i < p.nA * 128 ? __ldg(p.biasA + i) : __ldg(p.biasB + (i - p.nA * 128));
  if (threadIdx.x == 0) {
    for (int i = 0; i < 7; ++i) mbar_init(smem_u32(bars + i), (i == 2 || i >= 5) ? 256u : 1u);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(256)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  const uint32_t wfull = smem_u32(bars), wempty = smem_u32(bars + 1), bar_a = smem_u32(bars + 2);

  if (warp == 0) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc(128, 128);
      for (int t = 0; t < ntiles; ++t) {
        const bool isB = t >= p.nA;
        const CUtensorMap* map = isB ? &tm_wB : &tm_wA;
        const int row0 = (isB ? t - p.nA : t) * 128;
        if (t > 0) mbar_wait(wempty, (t - 1) & 1);           // previous MMA finished reading the weight slot
        mbar_expect_tx(wfull, TILE_B);
        tma_load_2d(Wt, map, wfull, 0, row0);
        tma_load_2d(Wt + KBB, map, wfull, 64, row0);
        if (t == 0) { mbar_wait(bar_a, 0); tcgen05_fence_after(); }
        if (t >= 2) { mbar_wait(smem_u32(bars + 5 + (t & 1)), ((t >> 1) - 1) & 1); tcgen05_fence_after(); }
        mbar_wait(wfull, t & 1);
        mma_tile(tmem + (t & 1) * 128, isB ? PB : PA, Wt, idesc, false);
        umma_commit(wempty);
        umma_commit(smem_u32(bars + 3 + (t & 1)));
      }
    }
  } else {
    // 8 worker warps: each builds 16 rows of the operand tiles, then owns (row, 64-column half) of every epilogue
    const int w8 = warp - 1, q = warp & 3, half = w8 >> 2;
    rows_to_tiles<16>(p.x, p.M, m0, w8 * 16, lane, p.eps, p.gA, p.bA, PA, p.gB, p.bB, p.nB > 0 ? PB : 0u);
    tcgen05_fence_before();
    fence_proxy_async();
    mbar_arrive(bar_a);
    const int row = q * 32 + lane;
    const long long grow = m0 + row;
    const bool valid = grow < p.M;
    const uint32_t tq = tmem + ((uint32_t)(q * 32) << 16) + half * 64;
    const int bb = (int)(grow / p.hbL), ll = (int)(grow % p.hbL);
    const float hmask = (p.hb[0] && valid) ? __ldg(p.hb_mask + grow) : 0.f;
    for (int t = 0; t < ntiles; ++t) {
      const bool isB = t >= p.nA;
      const int tt = isB ? t - p.nA : t;
      const float* bias = fb + t * 128 + half * 64;
      mbar_wait(smem_u32(bars + 3 + (t & 1)), (t >> 1) & 1);
      tcgen05_fence_after();
      // two 16-column chunks per TMEM round trip (tcgen05.wait::ld covers every outstanding load of the thread)
      auto emit = [&](int c, const uint32_t (&r0)[16], const float4 (&bq)[4]) {
        float v[16];
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const float4 bv = bq[j4];
          v[j4 * 4 + 0] = __uint_as_float(r0[j4 * 4 + 0]) + bv.x; v[j4 * 4 + 1] = __uint_as_float(r0[j4 * 4 + 1]) + bv.y;
          v[j4 * 4 + 2] = __uint_as_float(r0[j4 * 4 + 2]) + bv.z; v[j4 * 4 + 3] = __uint_as_float(r0[j4 * 4 + 3]) + bv.w;
        }
        const int cg = half * 4 + c;       // 16-column chunk index within the 128-wide tile
        if (valid && p.hb[0] && !isB) {
          // q is pre-scaled by sqrt(1/head_dim) like F.multi_head_attention_forward does before the q.k product
          if (tt == 0) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] *= 0.17677669529663687f;
          }
          __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.hb[tt]) +
                               ((long long)(ll * 4 + (cg >> 1)) * p.hbB + bb) * p.hb_stride[tt] + (cg & 1) * 16;
          uint4 lo, hi;
          lo.x = pack_bf16(v[0], v[1]); lo.y = pack_bf16(v[2], v[3]); lo.z = pack_bf16(v[4], v[5]); lo.w = pack_bf16(v[6], v[7]);
          hi.x = pack_bf16(v[8], v[9]); hi.y = pack_bf16(v[10], v[11]); hi.z = pack_bf16(v[12], v[13]); hi.w = pack_bf16(v[14], v[15]);
          *reinterpret_cast<uint4*>(dst) = lo;
          *reinterpret_cast<uint4*>(dst + 8) = hi;
          if (tt < 2 && (cg & 1)) {  // columns 32..47 of this head's row: [1 | mask, 0, ..., 0]
            const float m = tt == 0 ? 1.0f : hmask;
            *reinterpret_cast<uint4*>(dst + 16) = make_uint4(pack_bf16(m, 0.f), 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(dst + 24) = make_uint4(0u, 0u, 0u, 0u);
          }
        } else if (valid && p.out_bf16) {
          __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(isB ? p.outB : p.outA) +
                               grow * (long long)((isB ? p.nB : p.nA) * 128) + tt * 128 + cg * 16;
          uint4 lo, hi;
          lo.x = pack_bf16(v[0], v[1]); lo.y = pack_bf16(v[2], v[3]); lo.z = pack_bf16(v[4], v[5]); lo.w = pack_bf16(v[6], v[7]);
          hi.x = pack_bf16(v[8], v[9]); hi.y = pack_bf16(v[10], v[11]); hi.z = pack_bf16(v[12], v[13]); hi.w = pack_bf16(v[14], v[15]);
          *reinterpret_cast<uint4*>(dst) = lo;
          *reinterpret_cast<uint4*>(dst + 8) = hi;
        } else if (valid) {
          float* out = (isB ? p.outB : p.outA) + grow * (long long)((isB ? p.nB : p.nA) * 128) + tt * 128 + cg * 16;
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4)
            *reinterpret_cast<float4*>(out + j4 * 4) = make_float4(v[j4 * 4], v[j4 * 4 + 1], v[j4 * 4 + 2], v[j4 * 4 + 3]);
        }
      };
#pragma unroll 1
      for (int cp = 0; cp < 2; ++cp) {
        uint32_t ra[16], rb[16];
        tmem_ld16(tq + (t & 1) * 128 + cp * 32, ra);
        tmem_ld16(tq + (t & 1) * 128 + cp * 32 + 16, rb);
        float4 ba[4], bb[4];                     // biases fetched while the TMEM loads are in flight
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          ba[j4] = *reinterpret_cast<const float4*>(bias + cp * 32 + j4 * 4);
          bb[j4] = *reinterpret_cast<const float4*>(bias + cp * 32 + 16 + j4 * 4);
        }
        tmem_wait16(ra);
        tmem_wait16(rb);
        emit(cp * 2, ra, ba);
        emit(cp * 2 + 1, rb, bb);
      }
      tcgen05_fence_before();
      mbar_arrive(smem_u32(bars + 5 + (t & 1)));   // accumulator drained
    }
  }
  chain_end(tmem, 256);
}
constexpr size_t PROJ_LN_SMEM = 1024 + 3 * TILE_B + 128 + 5 * 128 * sizeof(float);

// ------------------------------------------------------------------------------------------------------------
// Whole DepthwiseSeparableConvBlock (4 layers, models/layers.py:139-148) + the position add of FeatureEncoder
// (models/layers.py:396-399) in ONE launch for segments of at most 128 rows, optionally followed by the LayerNorm +
// projections that consume the block's output (DualAttentionBlock's LN1 -> query|f_key|f_value and LNt -> t_key|t_value,
// models/layers.py:282-283,339-344; FeatureEncoderPredict's layer_norm_1 -> in_proj, models/layers.py:630-632).
// A CTA owns G = floor(128/len) whole segments, so the depthwise conv never needs rows of another CTA.
//   * the fp32 residual stream lives in REGISTERS: worker thread (row, 64-column half) keeps its 64 values for all four
//     layers; every epilogue (ReLU/bias/residual) updates them in place, produces the next layer's LayerNorm statistics
//     (the two halves of a row meet through shared memory) and writes the normalised row n^ = (x - mean) * rstd to the
//     fp32 tile Nt;
//   * operand tile of a layer: warp w builds rows [16w, 16w+16): A[r][c] = sum_j (w[c,j] g[c]) n^[r+j-3][c] + b[c] sum_j w[c,j]
//     over the taps inside the row's segment (LayerNorm's affine folded into the tap weights), register sliding window;
//   * one UMMA 128x128x128 per layer against the TMA-streamed pointwise weight.
// ------------------------------------------------------------------------------------------------------------
constexpr int LPR = 17;           // rows of the per-layer parameter table (see conv_block4_kernel)
constexpr int CB_HALO = 12, CB_OWN = 128 - 2 * CB_HALO;   // long segments: rows a tile recomputes per side / rows it owns
constexpr int XLD = 132;          // fp32 row stride of Nt (conflict-free float4 access by row or by column)

constexpr int CONV_TAB_FLOATS = 512 + 4 * LPR * 128;
// tab = [4][128] pointwise biases | [4 layers][17][128]: rows 0..6 = tap_j * g (LayerNorm's affine folded into the depthwise
// taps: n = n^ g + b  =>  conv = sum_j (w_j g) n^_j + b sum_j w_j), 7 = b * sum(taps), 8 = b, 9..16 = prefix sums PS[0..7]
__global__ void __launch_bounds__(512) conv_tables_kernel(const float* g0, const float* g1, const float* g2, const float* g3,
                                                          const float* b0, const float* b1, const float* b2, const float* b3,
                                                          const float* d0, const float* d1, const float* d2, const float* d3,
                                                          const float* p0, const float* p1, const float* p2, const float* p3,
                                                          float* __restrict__ tab) {
  const int layer = threadIdx.x >> 7, c = threadIdx.x & 127;
  const float* g = layer == 0 ? g0 : (layer == 1 ? g1 : (layer == 2 ? g2 : g3));
  const float* b = layer == 0 ? b0 : (layer == 1 ? b1 : (layer == 2 ? b2 : b3));
  const float* d = layer == 0 ? d0 : (layer == 1 ? d1 : (layer == 2 ? d2 : d3));
  const float* pb = layer == 0 ? p0 : (layer == 1 ? p1 : (layer == 2 ? p2 : p3));
  tab[threadIdx.x] = pb[c];
  float* lpar = tab + 512;
  const float gmm = g[c], btt = b[c];
  float ws = 0.f;
  for (int j = 0; j < 7; ++j) {
    const float wv = d[c * 7 + j];
    lpar[(layer * LPR + j) * 128 + c] = wv * gmm;
    lpar[(layer * LPR + 9 + j) * 128 + c] = ws;       // PS[j] = sum of taps < j
    ws += wv;
  }
  lpar[(layer * LPR + 16) * 128 + c] = ws;            // PS[7]
  lpar[(layer * LPR + 7) * 128 + c] = btt * ws;
  lpar[(layer * LPR + 8) * 128 + c] = btt;
}

struct ConvBlockParams {
  const float* x;      // [Mtot,128] block input
  const float* pos;    // position table [>=len,128]
  float* out;          // [Mtot,128] (may alias x: a CTA only touches its own rows)
  const float* tab;    // CONV_TAB_FLOATS floats built once per weight set by conv_tables_kernel: pointwise biases + tap tables
  long long R1;        // rows of group 0 (= nseg0 * len0); group 1 rows start here
  int nseg0, nseg1, len0, len1;
  int tiles0;          // CTAs of group 0
  int nlayers;         // 2 or 4 conv layers (BaseFast's shared encoder has 2)
  int halo0;           // > 0: group-0 segments are longer than a tile: `halo0` tiles per segment, each owning CB_OWN rows and
                       //      recomputing CB_HALO rows of its neighbours (3 rows of context per layer x 4 layers)
  int pair;            // > 0: CTA c owns segment c of group 0 followed by `pair` segments [c*pair, (c+1)*pair) of group 1
};                     //      (one video clip + its query in one 128-row tile: no separate text CTAs, no third wave)
struct ProjTail {      // LN + projections fused behind the block (nA == 0: none)
  int nA, nB;          // 128-wide output tiles computed from LN_A(x) / LN_B(x)
  float eps;
  const float* gA; const float* bA; const float* gB; const float* bB;
  const float* biasA; const float* biasB;
  void* outA; void* outB;     // bf16 row-major [Mtot, nA*128] / [Mtot, nB*128]   (used when hb[0] == nullptr)
  void* hb[3];                // head-blocked bf16 q/k/v [L][4][B][64|64|32] (see ProjLnParams)
  int hb_stride[3];
  int hbL, hbB;
  const float* hb_mask;
  int hb_tma;                 // 1: head-blocked outputs (and the mask columns of the q / k rows) leave through TMA stores
};                            //    (one segment = one sample per tile; tm_hq/hk/hv/hq16/hk16 valid)

// bf16 output of one 16-column chunk of a projection tile (shared by proj_ln_kernel's layouts)
__device__ __forceinline__ void proj_store_chunk(const ProjTail& t, bool isB, int tt, int cg, long long grow, int bb, int ll,
                                                 float hmask, float (&v)[16]) {
  if (t.hb[0] && !isB) {
    if (tt == 0) {
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] *= 0.17677669529663687f;   // q / sqrt(head_dim)
    }
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(t.hb[tt]) +
                         ((long long)(ll * 4 + (cg >> 1)) * t.hbB + bb) * t.hb_stride[tt] + (cg & 1) * 16;
    *reinterpret_cast<uint4*>(dst) = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
    *reinterpret_cast<uint4*>(dst + 8) = make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
    if (tt < 2 && (cg & 1)) {  // columns 32..47 of this head's row: [1 | mask, 0, ..., 0]
      const float m = tt == 0 ? 1.0f : hmask;
      *reinterpret_cast<uint4*>(dst + 16) = make_uint4(pack_bf16(m, 0.f), 0u, 0u, 0u);
      *reinterpret_cast<uint4*>(dst + 24) = make_uint4(0u, 0u, 0u, 0u);
    }
  } else {
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(isB ? t.outB : t.outA) +
                         grow * (long long)((isB ? t.nB : t.nA) * 128) + tt * 128 + cg * 16;
    *reinterpret_cast<uint4*>(dst) = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
    *reinterpret_cast<uint4*>(dst + 8) = make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
  }
}

// Operand tile rows [w*8, w*8+8) of one conv-block layer (see conv_block4_kernel): tile rows rb..rb+13 stream through an
// 8-slot register window (slot = k & 7), branch-free so that consecutive output rows overlap.  Packed fp32x2 FMAs
// (FFMA2): lane = 4 channels = 2 pairs.  Taps outside the row's segment are the conv's zero padding: with one segment per
// tile (MULTI = false) they read exact zeros anyway (rows before the tile are skipped, rows behind the segment are kept at
// n^ = 0), so only the LayerNorm-bias term b * (PS[hi+1] - PS[lo]) sees the edge; with several segments per tile the
// window value is masked per tap.
template <bool MULTI>
__device__ __forceinline__ void conv_build_rows(const float* __restrict__ Nt, const float* __restrict__ lp /* + col */, uint32_t A,
                                                int r0, int col, int l, int len, int len_next) {
  // (l, len): position of output row r0 inside its segment and that segment's length; len_next: length of the segments
  // that follow it in the tile (a mixed tile is one long segment followed by short ones)
  f32x2 wg[2][7];
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    const float4 t = *reinterpret_cast<const float4*>(lp + j * 128);
    wg[0][j] = pack2(t.x, t.y); wg[1][j] = pack2(t.z, t.w);
  }
  const float4 btf = *reinterpret_cast<const float4*>(lp + 8 * 128);
  const f32x2 bt0 = pack2(btf.x, btf.y), bt1 = pack2(btf.z, btf.w);
  const float4 fullf = *reinterpret_cast<const float4*>(lp + 7 * 128);          // b * sum(taps): the bias term of interior rows
  const f32x2 full0 = pack2(fullf.x, fullf.y), full1 = pack2(fullf.z, fullf.w);
  f32x2 win[8][2];
  const int rb = r0 - 3;
  const uint32_t a_col = (uint32_t)((col >> 6) * KBB + (col & 7) * 2);
  const int chunk = (col & 63) >> 3;
#pragma unroll
  for (int k = 0; k < 14; ++k) {
    const int rr = rb + k;
    {
      const float4 v = (rr >= 0 && rr < 128) ? *reinterpret_cast<const float4*>(Nt + rr * XLD + col) : make_float4(0.f, 0.f, 0.f, 0.f);
      win[k & 7][0] = pack2(v.x, v.y); win[k & 7][1] = pack2(v.z, v.w);
    }
    if (k >= 6) {
      const int r = rr - 3;                // output row (tile-local); taps j = 0..6 are rows r-3..r+3
      const int lo = max(0, 3 - l), hi = min(6, len + 2 - l);
      f32x2 acc0, acc1;
      if (lo == 0 && hi == 6) {
        // interior row (warp-uniform test: every lane of a warp works on the same rows): all 7 taps are inside the segment,
        // the LayerNorm-bias term is the per-channel constant b * sum(taps) -- no prefix-sum lookups (they were the largest
        // single consumer of shared-memory bandwidth in this kernel: 2 x 512 B per warp and output row)
        acc0 = full0; acc1 = full1;
#pragma unroll
        for (int j = 0; j < 7; ++j) {
          acc0 = fma2(wg[0][j], win[(k - 6 + j) & 7][0], acc0);
          acc1 = fma2(wg[1][j], win[(k - 6 + j) & 7][1], acc1);
        }
      } else {
        const float4 p1 = *reinterpret_cast<const float4*>(lp + (10 + hi) * 128);
        const float4 p0 = *reinterpret_cast<const float4*>(lp + (9 + lo) * 128);
        acc0 = mul2(bt0, pack2(p1.x - p0.x, p1.y - p0.y)); acc1 = mul2(bt1, pack2(p1.z - p0.z, p1.w - p0.w));
#pragma unroll
        for (int j = 0; j < 7; ++j) {
          f32x2 t0 = win[(k - 6 + j) & 7][0], t1 = win[(k - 6 + j) & 7][1];
          if (MULTI && (j < lo || j > hi)) { t0 = 0ull; t1 = 0ull; }
          acc0 = fma2(wg[0][j], t0, acc0);
          acc1 = fma2(wg[1][j], t1, acc1);
        }
      }
      float a0, a1, a2, a3;
      unpack2(acc0, a0, a1); unpack2(acc1, a2, a3);
      st_shared_v2_nc(A + a_col + (uint32_t)(r * 128 + ((chunk ^ (r & 7)) << 4)), pack_bf16(a0, a1), pack_bf16(a2, a3));
      if (++l == len) { l = 0; len = len_next; }
    }
  }
}

// (Round 2 measured an alternative mapping -- 16 rows x one 64-channel half per warp, two channels per lane, 22 window rows per 16
// output rows: half the LDS traffic per output row -- at +5 % kernel time (220.8 vs 206.7 us per step): the build is a dependent
// FFMA2 / issue chain, not a shared-memory-bandwidth problem.  The code was removed; DESIGN.md section 9 has the numbers.)
// 16 warps, no dedicated control warp: every phase ends in a CTA barrier after which ONE elected thread issues the
// tcgen05.mma chain (and the TMA load of the weight two layers ahead); all threads then wait on the commit barrier.
// Warp w: TMEM lane quadrant q = w & 3 (rows 32q..32q+31), column quarter cq = w >> 2 (columns 32cq..32cq+31).
constexpr int CB16_THREADS = 512;

__global__ void __launch_bounds__(CB16_THREADS, 1)
conv_block4_kernel(const __grid_constant__ CUtensorMap tm_w0, const __grid_constant__ CUtensorMap tm_w1,
                   const __grid_constant__ CUtensorMap tm_w2, const __grid_constant__ CUtensorMap tm_w3,
                   const __grid_constant__ CUtensorMap tm_pA, const __grid_constant__ CUtensorMap tm_pB,
                   const __grid_constant__ CUtensorMap tm_hq, const __grid_constant__ CUtensorMap tm_hk,
                   const __grid_constant__ CUtensorMap tm_hv, const __grid_constant__ CUtensorMap tm_hq16,
                   const __grid_constant__ CUtensorMap tm_hk16, ConvBlockParams p, ProjTail pt) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t A = base, Wb[2] = {base + TILE_B, base + 2 * TILE_B};
  float* Nt = reinterpret_cast<float*>(gen + 3 * TILE_B);             // [128][XLD] normalised rows (raw x at both ends)
  const uint32_t PB = base + 3 * TILE_B;                              // second operand tile of the tail: aliases Nt
  float* part = Nt + 128 * XLD;                                       // [4 quarters][128 rows][2]
  float* fbias = part + 1024;                                         // [4][128] pointwise biases
  float* lpar = fbias + 512;     // [4 layers][17][128]: 7 taps * g | b * sum(taps) | b | prefix sums PS[0..7] of the raw taps
  float* tbias = lpar + 4 * LPR * 128;                                // [<=5][128] projection biases of the tail
  uint8_t* tail = reinterpret_cast<uint8_t*>(tbias + 640);
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail);                 // 0/1 wfull, 2 bar_mma, 3..6 tfull[4]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tail + 64);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  TL(0);

  const int g = blockIdx.x >= (unsigned)p.tiles0;
  const int tile = blockIdx.x - (g ? p.tiles0 : 0);
  const bool pair = p.pair > 0;
  const bool halo = !g && p.halo0 > 0;                                // this tile is a window of a long group-0 segment
  const int len = (g && !pair) ? p.len1 : p.len0, nseg = (g && !pair) ? p.nseg1 : p.nseg0;
  const int G = (pair || halo) ? 2 : 128 / len;                       // segments per CTA (pair / halo: > 1 selects the masked taps)
  const int hseg = halo ? tile / p.halo0 : 0, ht = halo ? tile % p.halo0 : 0;
  const int l0 = halo ? max(0, ht * CB_OWN - CB_HALO) : 0;            // segment position of tile row 0
  const int seg0 = halo ? hseg : (pair ? tile : tile * G);
  const int split = pair ? p.len0 : 128;                              // first tile row of the group-1 segments (pair mode)
  const int lenB = pair ? p.len1 : len;                               // length of the segments behind the first one
  const int n1 = pair ? max(0, min(p.pair, p.nseg1 - tile * p.pair)) : 0;
  const int nrows = halo ? min(128, len - l0) : (pair ? p.len0 + n1 * p.len1 : min(G, nseg - seg0) * len);   // valid rows of this tile
  // rows this tile stores / projects: everything valid, or the owned window of a long segment
  const int own_lo = halo ? ht * CB_OWN - l0 : 0, own_hi = halo ? min(len, (ht + 1) * CB_OWN) - l0 : nrows;
  const long long row0 = ((g && !pair) ? p.R1 : 0) + (long long)seg0 * len + l0;
  const long long row1 = p.R1 + (long long)tile * p.pair * p.len1 - split;    // global row of tile row r >= split: row1 + r
  auto grow_of = [&](int r) -> long long { return r >= split ? row1 + r : row0 + r; };
  auto seg_pos = [&](int r) -> int { return r >= split ? (r - split) % lenB : (l0 + r) % len; };
  const int ntail = pt.nA + pt.nB;
  const bool issuer = threadIdx.x == 0;
  const CUtensorMap* maps[4] = {&tm_w0, &tm_w1, &tm_w2, &tm_w3};
  auto load_tile = [&](int slot, const CUtensorMap* map, int row) {
    const uint32_t full = smem_u32(bars + slot);
    mbar_expect_tx(full, TILE_B);
    tma_load_2d(Wb[slot], map, full, 0, row);
    tma_load_2d(Wb[slot] + KBB, map, full, 64, row);
  };
  auto tail_map = [&](int t, int& row) -> const CUtensorMap* {
    const bool isB = t >= pt.nA;
    row = (isB ? t - pt.nA : t) * 128;
    return isB ? &tm_pB : &tm_pA;
  };

  if (issuer) {
    for (int i = 0; i < 7; ++i) mbar_init(smem_u32(bars + i), 1u);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    load_tile(0, maps[0], 0);
    load_tile(1, maps[1], 0);
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  TL(28);
  // ---- tile load with cp.async (8 rows per warp, all in flight) ----
  const int col = lane * 4;
  {
    const uint32_t nt_s = smem_u32(Nt);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = warp * 8 + i;
      if (r < nrows) cp_async16(nt_s + (uint32_t)(r * XLD + col) * 4u, p.x + grow_of(r) * 128 + col);
      else *reinterpret_cast<float4*>(Nt + r * XLD + col) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  const int q = warp & 3, cq = warp >> 2;
  const int row = q * 32 + lane;           // this thread's residual row (TMEM lane)
  float* nrow = Nt + row * XLD + cq * 32;
  // position rows of this thread's (row, quarter) straight into registers
  float xr[32];
  {
    const float* pr = p.pos + (long long)seg_pos(row) * 128 + cq * 32;
    const bool has = row < nrows;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float4 v = has ? __ldg(reinterpret_cast<const float4*>(pr + i * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
      xr[i * 4] = v.x; xr[i * 4 + 1] = v.y; xr[i * 4 + 2] = v.z; xr[i * 4 + 3] = v.w;
    }
  }
  // pointwise biases + per-layer tap tables: identical for every CTA, built once per weight set (conv_tables_kernel);
  // one bulk copy in the same cp.async group as the row tile
  {
    const uint32_t dst = smem_u32(fbias);
    for (int i = threadIdx.x; i < CONV_TAB_FLOATS / 4; i += CB16_THREADS) cp_async16(dst + i * 16, p.tab + i * 4);
  }
  for (int i = threadIdx.x; i < ntail * 128; i += CB16_THREADS)
    tbias[i] = i < pt.nA * 128 ? __ldg(pt.biasA + i) : __ldg(pt.biasB + (i - pt.nA * 128));
  TL(29);
  cp_async_wait_all();
  TL(30);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  const uint32_t bar_mma = smem_u32(bars + 2);
  const uint32_t tq = tmem + ((uint32_t)(q * 32) << 16) + cq * 32;
  const uint32_t idesc = make_idesc(128, 128);
  TL(1);
  // ---- residual (row, quarter) into registers (+pos), LayerNorm statistics of layer 0 ----
  float sum = 0.f, sq = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4 v = *reinterpret_cast<const float4*>(nrow + i * 4);
    xr[i * 4] += v.x; xr[i * 4 + 1] += v.y; xr[i * 4 + 2] += v.z; xr[i * 4 + 3] += v.w;
    sum += (xr[i * 4] + xr[i * 4 + 1]) + (xr[i * 4 + 2] + xr[i * 4 + 3]);
    sq = fmaf(xr[i * 4], xr[i * 4], fmaf(xr[i * 4 + 1], xr[i * 4 + 1], fmaf(xr[i * 4 + 2], xr[i * 4 + 2], fmaf(xr[i * 4 + 3], xr[i * 4 + 3], sq))));
  }
  // row statistics from the four quarter sums; returns (mean, rstd)
  auto row_stats = [&](float eps, float& mean, float& rstd) {
    part[(cq * 128 + row) * 2] = sum;
    part[(cq * 128 + row) * 2 + 1] = sq;
    __syncthreads();
    float s = 0.f, s2 = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) { s += part[(k * 128 + row) * 2]; s2 += part[(k * 128 + row) * 2 + 1]; }
    mean = s * (1.0f / 128.0f);
    rstd = rsqrtf(fmaxf(s2 * (1.0f / 128.0f) - mean * mean, 0.f) + eps);
  };
  // writes n^ = (x - mean) * rstd of this (row, quarter) to Nt; rows behind the tile's last segment stay exact zeros:
  // they are the zero padding of the depthwise conv
  auto normalise = [&]() {
    float mean, rstd;
    row_stats(1e-6f, mean, rstd);
    if (row >= nrows) rstd = 0.f;
    const float off = -mean * rstd;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      *reinterpret_cast<float4*>(nrow + i * 4) = make_float4(fmaf(xr[i * 4], rstd, off), fmaf(xr[i * 4 + 1], rstd, off),
                                                             fmaf(xr[i * 4 + 2], rstd, off), fmaf(xr[i * 4 + 3], rstd, off));
    __syncthreads();
  };
  normalise();
  TL(2);
  uint32_t nfull[2] = {0, 0};
  const int bl0 = seg_pos(warp * 8), bl_len = warp * 8 >= split ? lenB : len;   // this warp's first output row in its segment
  const int nl = p.nlayers;
  for (int layer = 0; layer < nl; ++layer) {
    // ---- operand tile: A[r] = DW7(LN(X))[r] for this warp's 8 rows ----
    if (G > 1) conv_build_rows<true>(Nt, lpar + layer * LPR * 128 + col, A, warp * 8, col, bl0, bl_len, lenB);
    else conv_build_rows<false>(Nt, lpar + layer * LPR * 128 + col, A, warp * 8, col, bl0, bl_len, lenB);
    TL(3 + layer * 4);
    tcgen05_fence_before();
    fence_proxy_async();
    __syncthreads();
    const int sl = layer & 1;
    if (issuer) {
      tcgen05_fence_after();
      mbar_wait(smem_u32(bars + sl), nfull[sl]++ & 1);
      mma_tile(tmem, A, Wb[sl], idesc, false);
      umma_commit(bar_mma);
    }
    // ---- epilogue: x += ReLU(acc + b) on this thread's (row, 32-column quarter), kept in registers ----
    mbar_wait(bar_mma, layer & 1);
    tcgen05_fence_after();
    TL(4 + layer * 4);
    if (issuer) {   // the weight slot is free again: next-but-one layer, or the first projection tiles of the tail
      const int nxt = layer + 2;
      if (nxt < nl) load_tile(sl, maps[nxt], 0);
      else if (nxt - nl < ntail) { int wrow; const CUtensorMap* m = tail_map(nxt - nl, wrow); load_tile(sl, m, wrow); }
    }
    sum = 0.f; sq = 0.f;
    const float* bl = fbias + layer * 128 + cq * 32;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      uint32_t r0[16];
      tmem_ld16(tq + c * 16, r0);
      tmem_wait16(r0);
#pragma unroll
      for (int j4 = 0; j4 < 4; ++j4) {
        const float4 bv = *reinterpret_cast<const float4*>(bl + c * 16 + j4 * 4);
        float* x4 = xr + c * 16 + j4 * 4;
        x4[0] += fmaxf(__uint_as_float(r0[j4 * 4 + 0]) + bv.x, 0.f);
        x4[1] += fmaxf(__uint_as_float(r0[j4 * 4 + 1]) + bv.y, 0.f);
        x4[2] += fmaxf(__uint_as_float(r0[j4 * 4 + 2]) + bv.z, 0.f);
        x4[3] += fmaxf(__uint_as_float(r0[j4 * 4 + 3]) + bv.w, 0.f);
        sum += (x4[0] + x4[1]) + (x4[2] + x4[3]);
        sq = fmaf(x4[0], x4[0], fmaf(x4[1], x4[1], fmaf(x4[2], x4[2], fmaf(x4[3], x4[3], sq))));
      }
    }
    tcgen05_fence_before();
    TL(5 + layer * 4);
    if (layer < nl - 1) normalise();
    TL(6 + layer * 4);
  }
  // ---- block output: through Nt for coalesced 512-byte row stores ----
#pragma unroll
  for (int i = 0; i < 8; ++i)
    *reinterpret_cast<float4*>(nrow + i * 4) = make_float4(xr[i * 4], xr[i * 4 + 1], xr[i * 4 + 2], xr[i * 4 + 3]);
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = warp * 8 + i;
    if (r >= own_lo && r < own_hi)
      *reinterpret_cast<float4*>(p.out + grow_of(r) * 128 + col) = *reinterpret_cast<const float4*>(Nt + r * XLD + col);
  }
  TL(19);
  if (ntail > 0) {
    // ---- fused LayerNorm + projections of the consumer: operand tiles from the register-resident rows ----
    float mean, rstd;
    row_stats(pt.eps, mean, rstd);                     // its barrier also orders the Nt reads above before PB (alias) writes
    {
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        float va[16], vb[16];
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const int cc = cq * 32 + c * 16 + j4 * 4;
          const float4 ga = __ldg(reinterpret_cast<const float4*>(pt.gA + cc)), ba = __ldg(reinterpret_cast<const float4*>(pt.bA + cc));
          const float n0 = (xr[c * 16 + j4 * 4] - mean) * rstd, n1 = (xr[c * 16 + j4 * 4 + 1] - mean) * rstd,
                      n2 = (xr[c * 16 + j4 * 4 + 2] - mean) * rstd, n3 = (xr[c * 16 + j4 * 4 + 3] - mean) * rstd;
          va[j4 * 4] = fmaf(n0, ga.x, ba.x); va[j4 * 4 + 1] = fmaf(n1, ga.y, ba.y);
          va[j4 * 4 + 2] = fmaf(n2, ga.z, ba.z); va[j4 * 4 + 3] = fmaf(n3, ga.w, ba.w);
          if (pt.nB > 0) {
            const float4 gb = __ldg(reinterpret_cast<const float4*>(pt.gB + cc)), bb4 = __ldg(reinterpret_cast<const float4*>(pt.bB + cc));
            vb[j4 * 4] = fmaf(n0, gb.x, bb4.x); vb[j4 * 4 + 1] = fmaf(n1, gb.y, bb4.y);
            vb[j4 * 4 + 2] = fmaf(n2, gb.z, bb4.z); vb[j4 * 4 + 3] = fmaf(n3, gb.w, bb4.w);
          }
        }
        store_a16(A, row, cq * 32 + c * 16, va);
        if (pt.nB > 0) store_a16(PB, row, cq * 32 + c * 16, vb);
      }
    }
    const long long grow = grow_of(row);
    const bool valid = row >= own_lo && row < own_hi;
    const int bb = (int)(grow / pt.hbL), ll = (int)(grow % pt.hbL);
    const float hmask = (pt.hb[0] && valid) ? __ldg(pt.hb_mask + grow) : 0.f;
    // columns 32..47 of the head-blocked q / k rows ([1 | key mask, 0 x 15]: the additive key mask rides in the score MMA;
    // columns 48..63 are never read): two [128 positions][16] blocks in the dead tap-table region, stored once per head
    const uint32_t MQ = smem_u32(lpar), MK = MQ + 4096;
    if (pt.hb_tma && cq == 0) {
      st_shared_v4(MQ + row * 32, pack_bf16(1.0f, 0.f), 0u, 0u, 0u); st_shared_v4(MQ + row * 32 + 16, 0u, 0u, 0u, 0u);
      st_shared_v4(MK + row * 32, pack_bf16(hmask, 0.f), 0u, 0u, 0u); st_shared_v4(MK + row * 32 + 16, 0u, 0u, 0u, 0u);
    }
    tcgen05_fence_before();
    fence_proxy_async();
    for (int t = 0; t <= ntail; ++t) {
      // Four TMEM accumulators (tile t -> columns (t & 3) * 128): no accumulator is reused before tile 4, so the only CTA
      // barriers are the one that publishes the operand tiles (t == 0) and the one before tile 4 overwrites accumulator 0
      // (every thread drained it in iteration 1).  The weight slot of tile t was refilled by the issuer once tile t-2's
      // MMA had signalled completion (below), so MMA t only waits for its TMA.
      if (t == 0 || t == 4) __syncthreads();
      if (issuer && t < ntail) {
        const int sl = t & 1;
        tcgen05_fence_after();
        mbar_wait(smem_u32(bars + sl), nfull[sl]++ & 1);
        mma_tile(tmem + (t & 3) * 128, t >= pt.nA ? PB : A, Wb[sl], idesc, false);
        umma_commit(smem_u32(bars + 3 + (t & 3)));
      }
      if (t == 0) continue;
      const int u = t - 1;                              // epilogue of tile u overlaps the MMA of tile u + 1
      const bool isB = u >= pt.nA;
      const int tt = isB ? u - pt.nA : u;
      const float* bias = tbias + u * 128 + cq * 32;
      mbar_wait(smem_u32(bars + 3 + (u & 3)), (u >> 2) & 1);
      tcgen05_fence_after();
      TL(21 + u);
      if (issuer && u + 2 < ntail) {                    // tile u's MMA has finished reading its weight slot
        int wrow; const CUtensorMap* m = tail_map(u + 2, wrow);
        load_tile(u & 1, m, wrow);
      }
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        uint32_t r0[16];
        tmem_ld16(tq + (u & 3) * 128 + c * 16, r0);
        tmem_wait16(r0);
        float v[16];
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) {
          const float4 bv = *reinterpret_cast<const float4*>(bias + c * 16 + j4 * 4);
          v[j4 * 4 + 0] = __uint_as_float(r0[j4 * 4 + 0]) + bv.x; v[j4 * 4 + 1] = __uint_as_float(r0[j4 * 4 + 1]) + bv.y;
          v[j4 * 4 + 2] = __uint_as_float(r0[j4 * 4 + 2]) + bv.z; v[j4 * 4 + 3] = __uint_as_float(r0[j4 * 4 + 3]) + bv.w;
        }
        if (pt.hb_tma) {
          // staging tile of this projection: 4 head boxes of [128 positions][32 d] bf16 (64-byte rows, 64-byte swizzle);
          // this thread's quarter cq IS head cq, its two chunks are the 16-byte chunks 2c, 2c+1 of the head's row
          if (tt == 0) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] *= 0.17677669529663687f;   // q / sqrt(head_dim)
          }
          const uint32_t sb = PB + (u & 1) * TILE_B + cq * 8192 + row * 64;
          const int sx = (row >> 1) & 3;
          st_shared_v4(sb + (((2 * c) ^ sx) << 4), pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
          st_shared_v4(sb + (((2 * c + 1) ^ sx) << 4), pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
        } else if (valid) {
          proj_store_chunk(pt, isB, tt, cq * 2 + c, grow, bb, ll, hmask, v);
        }
      }
      tcgen05_fence_before();
      if (pt.hb_tma) {
        fence_proxy_async();
        __syncthreads();                                  // staging tile of projection u complete
        if (issuer) {
          const CUtensorMap* hm = tt == 0 ? &tm_hq : (tt == 1 ? &tm_hk : &tm_hv);
          const int bsmp = (int)(row0 / pt.hbL);          // one segment (sample) per tile
#pragma unroll
          for (int hd = 0; hd < 4; ++hd) tma_store_4d(hm, PB + (u & 1) * TILE_B + hd * 8192, 0, bsmp, hd, 0);
          if (tt < 2) {
#pragma unroll
            for (int hd = 0; hd < 4; ++hd) tma_store_4d(tt == 0 ? &tm_hq16 : &tm_hk16, tt == 0 ? MQ : MK, 32, bsmp, hd, 0);
          }
          tma_store_commit();
          tma_store_wait_read1();                         // the other staging buffer (projection u-1) has been read
        }
      }
    }
    if (pt.hb_tma && issuer) tma_store_wait_read();
  }
  TL(26);
  tcgen05_fence_before();
  __syncthreads();
  TL(27);
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
  }
}
constexpr size_t CONV_BLOCK_SMEM = 1024 + 3 * TILE_B + (128 * XLD + 1024 + 512 + 640 + 4 * LPR * 128) * sizeof(float) + 128;


thread_local char g_chain_err[256] = "";

}  // namespace

const char* chain_last_error() { return g_chain_err; }

int chain_read_timeline(long long* out64) { return tl_read(out64); }

static int chain_set_smem(SqSmemOptIn& optin, const void* fn, size_t bytes) {
  cudaError_t e = optin.ensure(fn, bytes);
  if (e != cudaSuccess) { snprintf(g_chain_err, sizeof(g_chain_err), "%s", cudaGetErrorString(e)); return SEQPAN_E_CUDA; }
  return SEQPAN_OK;
}
static int chain_check_launch() {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { snprintf(g_chain_err, sizeof(g_chain_err), "%s", cudaGetErrorString(e)); return SEQPAN_E_CUDA; }
  return SEQPAN_OK;
}

int chain_proj_ln(const TcArena& a, int slotA, int slotB, const float* x, long long M, float eps, const float* gA,
                  const float* bA, const float* gB, const float* bB, float* outA, const float* biasA, float* outB,
                  const float* biasB, cudaStream_t st, void* const* hb, int hbL, int hbB, const float* hb_mask,
                  bool out_bf16) {
  if (M <= 0) return SEQPAN_OK;
  static SqSmemOptIn optin;
  { int rc = chain_set_smem(optin, (const void*)proj_ln_kernel, PROJ_LN_SMEM); if (rc) return rc; }
  ProjLnParams p;
  p.x = x; p.M = M; p.eps = eps; p.gA = gA; p.bA = bA; p.gB = gB; p.bB = bB; p.outA = outA; p.outB = outB;
  p.biasA = biasA; p.biasB = biasB;
  p.nA = a.slot[slotA].N / 128;
  p.nB = slotB >= 0 ? a.slot[slotB].N / 128 : 0;
  for (int i = 0; i < 3; ++i) { p.hb[i] = hb ? hb[i] : nullptr; p.hb_stride[i] = i < 2 ? 64 : 32; }
  p.hbL = hbL > 0 ? hbL : 1; p.hbB = hbB; p.hb_mask = hb_mask; p.out_bf16 = out_bf16 ? 1 : 0;
  const CUtensorMap& mA = *reinterpret_cast<const CUtensorMap*>(a.slot[slotA].tmap);
  const CUtensorMap& mB = *reinterpret_cast<const CUtensorMap*>(a.slot[slotB >= 0 ? slotB : slotA].tmap);
  proj_ln_kernel<<<(unsigned)((M + 127) / 128), CB_THREADS, PROJ_LN_SMEM, st>>>(mA, mB, p);
  return chain_check_launch();
}

size_t chain_conv_tab_floats() { return CONV_TAB_FLOATS; }

int chain_conv_tables(const float* const* ln_g, const float* const* ln_b, const float* const* dw, const float* const* bias,
                      float* tab, cudaStream_t st) {
  conv_tables_kernel<<<1, 512, 0, st>>>(ln_g[0], ln_g[1], ln_g[2], ln_g[3], ln_b[0], ln_b[1], ln_b[2], ln_b[3], dw[0], dw[1], dw[2],
                                        dw[3], bias[0], bias[1], bias[2], bias[3], tab);
  return chain_check_launch();
}

int chain_conv_block(const TcArena& a, int slot0, const float* x, const float* pos, float* out, const float* tab, int nseg0,
                     int len0, int nseg1, int len1, cudaStream_t st, const ChainProjTail* tail, int nlayers) {
  if (nlayers != 2 && nlayers != 4) { snprintf(g_chain_err, sizeof(g_chain_err), "conv block: 2 or 4 layers"); return SEQPAN_E_INVALID; }
  // group 0 may hold long segments (tiled with halos, at most SEQPAN_MAX_VLEN rows); group 1 segments must fit one tile
  if (len0 < 1 || len0 > SEQPAN_MAX_VLEN || len1 > 128) {
    snprintf(g_chain_err, sizeof(g_chain_err), "conv block: segment lengths %d / %d outside [1,%d] / [0,128]", len0, len1, SEQPAN_MAX_VLEN);
    return SEQPAN_E_INVALID;
  }
  static SqSmemOptIn optin;
  { int rc = chain_set_smem(optin, (const void*)conv_block4_kernel, CONV_BLOCK_SMEM); if (rc) return rc; }
  ConvBlockParams p;
  p.x = x; p.pos = pos; p.out = out; p.tab = tab; p.nlayers = nlayers;
  p.nseg0 = nseg0; p.nseg1 = nseg1; p.len0 = len0; p.len1 = len1 > 0 ? len1 : 1;
  p.R1 = (long long)nseg0 * len0;
  const int G0 = len0 <= 128 ? 128 / len0 : 1, G1 = len1 > 0 ? 128 / len1 : 1;
  p.halo0 = len0 > 128 ? (len0 + CB_OWN - 1) / CB_OWN : 0;   // long segments: windows of CB_OWN owned rows + halos
  p.tiles0 = p.halo0 ? nseg0 * p.halo0 : (nseg0 + G0 - 1) / G0;
  int tiles1 = (len1 > 0 && nseg1 > 0) ? (nseg1 + G1 - 1) / G1 : 0;
  // pair mode: one long segment + the short segments that fit behind it in the same 128-row tile (a clip and its query)
  p.pair = 0;
  if (tiles1 > 0 && G0 == 1 && !p.halo0 && len0 + len1 <= 128) {
    const int g1 = (128 - len0) / len1;
    if ((long long)nseg0 * g1 >= nseg1) { p.pair = g1; tiles1 = 0; }
  }
  if (p.tiles0 + tiles1 <= 0) return SEQPAN_OK;
  auto tm = [&](int i) { return *reinterpret_cast<const CUtensorMap*>(a.slot[slot0 + (i < nlayers ? i : 0)].tmap); };
  ProjTail pt{};
  int sA = slot0, sB = slot0;
  pt.hbL = 1;
  if (tail) {
    sA = tail->slotA; sB = tail->slotB >= 0 ? tail->slotB : tail->slotA;
    pt.nA = a.slot[tail->slotA].N / 128;
    pt.nB = tail->slotB >= 0 ? a.slot[tail->slotB].N / 128 : 0;
    if (pt.nA + pt.nB > 5) { snprintf(g_chain_err, sizeof(g_chain_err), "conv block tail: more than 5 projection tiles"); return SEQPAN_E_INVALID; }
    pt.eps = tail->eps; pt.gA = tail->gA; pt.bA = tail->bA; pt.gB = tail->gB; pt.bB = tail->bB;
    pt.biasA = tail->biasA; pt.biasB = tail->biasB; pt.outA = tail->outA; pt.outB = tail->outB;
    for (int i = 0; i < 3; ++i) { pt.hb[i] = tail->hb ? tail->hb[i] : nullptr; pt.hb_stride[i] = i < 2 ? 64 : 32; }
    pt.hbL = tail->hbL > 0 ? tail->hbL : 1; pt.hbB = tail->hbB; pt.hb_mask = tail->hb_mask;
    // head-blocked outputs by TMA: one whole sample per tile (so a tile is one (b, all l) block) and no second operand tile
    pt.hb_tma = (tail->hb && G0 == 1 && !p.halo0 && nseg1 == 0 && pt.nB == 0 && len0 == pt.hbL) ? 1 : 0;
  }
  CUtensorMap hq, hk, hv, hq16, hk16;
  memset(&hq, 0, sizeof(hq)); memset(&hk, 0, sizeof(hk)); memset(&hv, 0, sizeof(hv)); memset(&hq16, 0, sizeof(hq16)); memset(&hk16, 0, sizeof(hk16));
  if (pt.hb_tma) {
    if (tc_make_hb_tmap(&hq, pt.hb[0], pt.hbB, pt.hbL, 64) != SEQPAN_OK || tc_make_hb_tmap(&hk, pt.hb[1], pt.hbB, pt.hbL, 64) != SEQPAN_OK ||
        tc_make_hb_tmap(&hv, pt.hb[2], pt.hbB, pt.hbL, 32) != SEQPAN_OK || tc_make_hb_tmap(&hq16, pt.hb[0], pt.hbB, pt.hbL, 64, 16) != SEQPAN_OK ||
        tc_make_hb_tmap(&hk16, pt.hb[1], pt.hbB, pt.hbL, 64, 16) != SEQPAN_OK) {
      snprintf(g_chain_err, sizeof(g_chain_err), "%s", tc_last_error());
      return SEQPAN_E_CUDA;
    }
  }
  conv_block4_kernel<<<p.tiles0 + tiles1, CB16_THREADS, CONV_BLOCK_SMEM, st>>>(
      tm(0), tm(1), tm(2), tm(3), *reinterpret_cast<const CUtensorMap*>(a.slot[sA].tmap),
      *reinterpret_cast<const CUtensorMap*>(a.slot[sB].tmap), hq, hk, hv, hq16, hk16, p, pt);
  return chain_check_launch();
}
