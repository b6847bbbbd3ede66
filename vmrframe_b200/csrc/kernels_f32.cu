// fp32 CUDA-core kernels of the SeqPAN hot path (sm_100a).  These carry the rtol-1e-4 parity gate and every
// non-GEMM block of both precision modes: masking, softmax, LayerNorm, depthwise conv, attention, span decode.
// Reference formulas: SURVEY.md Appendix A; each kernel cites the reference lines it replaces.
#include <cstdlib>
#include "kernels.cuh"

#include <cuda_bf16.h>

namespace sq {

// ------------------------------------------------------------------------------------------------
// Linear: y = act(x . w^T + bias) (+ residual)      replaces Conv1D(k=1) (models/layers.py:15-26)
// 128x128x32 tiles, 256 threads, 8x8 register micro-tiles, register prefetch of the next k-tile.
// Thread (tx,ty) owns rows ty*8+i and columns tx+16*j so that both shared-memory operand reads are
// conflict-free LDS.128 (row stride 36 floats).
// ------------------------------------------------------------------------------------------------
constexpr int LBM = 128, LBN = 128, LBK = 32, LPAD = 36;

__global__ void __launch_bounds__(256) linear_f32_kernel(LinearArgs a) {
  __shared__ __align__(16) float Xs[LBM][LPAD];
  __shared__ __align__(16) float Ws[LBN][LPAD];
  const int z = blockIdx.z;
  const float* __restrict__ X = a.x[z];
  const float* __restrict__ W = a.w[z];
  const float* __restrict__ bias = a.bias[z];
  const float* R = a.res[z];  // may alias Y (in-place residual update): no __restrict__
  float* Y = a.y[z];
  const long long M = a.M;
  const int N = a.N, K = a.K;
  const long long m0 = (long long)blockIdx.x * LBM;
  const int n0 = blockIdx.y * LBN;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  float4 xr[4], wr[4];
  auto load_tile = [&](int k0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int id = tid + 256 * i, r = id >> 3, c = (id & 7) * 4;
      const int k = k0 + c;
      const long long m = m0 + r;
      const int n = n0 + r;
      xr[i] = (m < M && k < K) ? ldg4(X + m * a.ldx + k) : make_float4(0.f, 0.f, 0.f, 0.f);
      wr[i] = (n < N && k < K) ? ldg4(W + (long long)n * a.ldw + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  load_tile(0);
  for (int k0 = 0; k0 < K; k0 += LBK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int id = tid + 256 * i, r = id >> 3, c = (id & 7) * 4;
      st4(&Xs[r][c], xr[i]);
      st4(&Ws[r][c], wr[i]);
    }
    __syncthreads();
    if (k0 + LBK < K) load_tile(k0 + LBK);
#pragma unroll
    for (int kk = 0; kk < LBK; kk += 4) {
      float4 wb[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) wb[j] = ld4(&Ws[tx + 16 * j][kk]);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 xa = ld4(&Xs[ty * 8 + i][kk]);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc[i][j] = fmaf(xa.x, wb[j].x, acc[i][j]);
          acc[i][j] = fmaf(xa.y, wb[j].y, acc[i][j]);
          acc[i][j] = fmaf(xa.z, wb[j].z, acc[i][j]);
          acc[i][j] = fmaf(xa.w, wb[j].w, acc[i][j]);
        }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const long long m = m0 + ty * 8 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int n = n0 + tx + 16 * j;
      if (n >= N) continue;
      float v = acc[i][j] + (bias ? __ldg(bias + n) : 0.f);
      if (a.relu) v = fmaxf(v, 0.f);
      if (R) v += R[m * a.ldr + n];
      Y[m * a.ldy + n] = v;
    }
  }
}

cudaError_t launch_linear_f32(const LinearArgs& a, cudaStream_t st) {
  if (a.M <= 0) return cudaSuccess;
  dim3 grid((unsigned)((a.M + LBM - 1) / LBM), (unsigned)((a.N + LBN - 1) / LBN), (unsigned)a.count);
  linear_f32_kernel<<<grid, 256, 0, st>>>(a);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// LayerNorm over 128 columns, one warp per row, up to two affine outputs from one read of x
// (DualAttentionBlock.layer_norm_1 / layer_norm_t, models/layers.py:282-283), optional side copy of a
// second 128-wide row into columns [128,256) of y1 (torch.concat([LN(feat), x]), models/layers.py:666-667).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, int ldx, long long M,
                                                        const float* __restrict__ g1, const float* __restrict__ b1,
                                                        float eps, float* __restrict__ y1, int ldy1,
                                                        const float* __restrict__ g2, const float* __restrict__ b2,
                                                        float* __restrict__ y2, int ldy2,
                                                        const float* __restrict__ copy_src, float* __restrict__ copy_dst,
                                                        int ldcopy) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float4 v = ldg4(x + row * ldx + lane * 4);
  float mean, rstd;
  row_stats(v, eps, mean, rstd);
  st4(y1 + row * ldy1 + lane * 4, ln_apply(v, mean, rstd, ldg4(g1 + lane * 4), ldg4(b1 + lane * 4)));
  if (y2) st4(y2 + row * ldy2 + lane * 4, ln_apply(v, mean, rstd, ldg4(g2 + lane * 4), ldg4(b2 + lane * 4)));
  if (copy_dst) st4(copy_dst + row * ldcopy + lane * 4, ldg4(copy_src + row * SQ_D + lane * 4));
}

cudaError_t launch_layernorm(const float* x, int ldx, long long M, const float* g1, const float* b1, float eps,
                             float* y1, int ldy1, const float* g2, const float* b2, float* y2, int ldy2,
                             const float* copy_src, float* copy_dst, int ldcopy, cudaStream_t st) {
  if (M <= 0) return cudaSuccess;
  layernorm_kernel<<<(unsigned)((M + 7) / 8), 256, 0, st>>>(x, ldx, M, g1, b1, eps, y1, ldy1, g2, b2, y2, ldy2,
                                                            copy_src, copy_dst, ldcopy);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// z = DW7(LN(x (+pos)))   one layer of DepthwiseSeparableConvBlock up to the pointwise conv
// (models/layers.py:139-148: LayerNorm eps 1e-6 then depthwise k=7, padding 3 (zeros at the TENSOR edge,
// not the mask edge), no bias) with the PositionalEmbedding add of FeatureEncoder.forward (:396-399) fused
// into the first layer.  One CTA = 32 rows of one segment + 3 halo rows each side; LN is recomputed for
// the halo.  Padded rows are processed exactly like valid ones (SURVEY.md §0 #11).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ln_dwconv_kernel(const float* __restrict__ x, const float* __restrict__ pos,
                                                        float* __restrict__ x0_out, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, float eps,
                                                        const float* __restrict__ dw, float* __restrict__ z, Segs sg,
                                                        int nblk0, int chunks0, int chunks1) {
  __shared__ __align__(16) float tile[38][SQ_D];
  const int g = blockIdx.x >= (unsigned)nblk0;
  const int blk = blockIdx.x - (g ? nblk0 : 0);
  const int chunks = g ? chunks1 : chunks0;
  const int seg = blk / chunks, c0 = (blk % chunks) * 32;
  const int len = sg.len[g];
  const long long base = sg.row0[g] + (long long)seg * len;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float4 gm = ldg4(gamma + lane * 4), bt = ldg4(beta + lane * 4);
  for (int i = w; i < 38; i += 8) {
    const int r = c0 - 3 + i;
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r >= 0 && r < len) {
      float4 v = ldg4(x + (base + r) * SQ_D + lane * 4);
      if (pos) {
        const float4 p = ldg4(pos + (long long)r * SQ_D + lane * 4);
        v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
        if (i >= 3 && i < 35) st4(x0_out + (base + r) * SQ_D + lane * 4, v);
      }
      float mean, rstd;
      row_stats(v, eps, mean, rstd);
      o = ln_apply(v, mean, rstd, gm, bt);
    }
    st4(&tile[i][lane * 4], o);
  }
  __syncthreads();
  float wg[4][7];
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int j = 0; j < 7; ++j) wg[c][j] = __ldg(dw + (lane * 4 + c) * 7 + j);
  for (int rr = w; rr < 32; rr += 8) {
    const int r = c0 + rr;
    if (r >= len) break;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      const float4 t = ld4(&tile[rr + j][lane * 4]);
      acc.x = fmaf(wg[0][j], t.x, acc.x);
      acc.y = fmaf(wg[1][j], t.y, acc.y);
      acc.z = fmaf(wg[2][j], t.z, acc.z);
      acc.w = fmaf(wg[3][j], t.w, acc.w);
    }
    st4(z + (base + r) * SQ_D + lane * 4, acc);
  }
}

cudaError_t launch_ln_dwconv(const float* x, const float* pos, float* x0_out, const float* gamma, const float* beta,
                             float eps, const float* dw, float* z, const Segs& sg, cudaStream_t st) {
  const int chunks0 = (sg.len[0] + 31) / 32, chunks1 = (sg.len[1] + 31) / 32;
  const int nblk0 = sg.nseg[0] * chunks0, nblk1 = sg.nseg[1] * chunks1;
  if (nblk0 + nblk1 <= 0) return cudaSuccess;
  ln_dwconv_kernel<<<nblk0 + nblk1, 256, 0, st>>>(x, pos, x0_out, gamma, beta, eps, dw, z, sg, nblk0,
                                                  chunks0 > 0 ? chunks0 : 1, chunks1 > 0 ? chunks1 : 1);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Text embedding (models/layers.py:28-93).  Pack time: the char-CNN's Conv2d(100->ch,(1,k)) over the
// embedded characters is linear in the embedding, and the character vocabulary is tiny, so
// P[k][j][char][o] = sum_i Wk[o,i,0,j] * emb[char,i] is tabulated once per weight set (300*num_chars
// floats); the per-word work becomes k table adds per (position, channel) instead of 100*k MACs.
// Run time: gather the word vector from cat[pad, unk, glove] (never materialised) and evaluate
// max_p ReLU(b + sum_j P[k][j][char[p+j]]) per channel.   Output row = [word 300 | char 100].
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int char_tab_offset(int k, int nc) {  // start of kernel-size k's table (k = 1..4)
  return nc * 10 * ((k - 1) * k * (2 * k - 1) / 6);               // sum_{q<k} q * (10 q) * nc
}

__global__ void char_table_kernel(const float* __restrict__ w1, const float* __restrict__ w2,
                                  const float* __restrict__ w3, const float* __restrict__ w4,
                                  const float* __restrict__ emb, int nc, float* __restrict__ table) {
  const int total = 300 * nc;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  int k = 1;
  while (k < 4 && idx >= char_tab_offset(k + 1, nc)) ++k;
  const int ch = 10 * k;
  int rem = idx - char_tab_offset(k, nc);
  const int ol = rem % ch; rem /= ch;
  const int c = rem % nc;
  const int j = rem / nc;
  const float* W = k == 1 ? w1 : k == 2 ? w2 : k == 3 ? w3 : w4;  // [ch, 100, 1, k]
  float s = 0.f;
  for (int i = 0; i < 100; ++i) s = fmaf(W[(ol * 100 + i) * k + j], emb[c * 100 + i], s);
  table[idx] = s;
}

cudaError_t launch_char_table(const float* const conv_w[4], const float* char_emb, int num_chars, float* table,
                              cudaStream_t st) {
  const int total = 300 * num_chars;
  char_table_kernel<<<(total + 255) / 256, 256, 0, st>>>(conv_w[0], conv_w[1], conv_w[2], conv_w[3], char_emb,
                                                         num_chars, table);
  return cudaGetLastError();
}

// One work unit = (kernel size K, channel pair, position p): K float2 table reads summed in tap order (the same order as
// a per-channel loop), ReLU, then a shared-memory max over the positions (non-negative floats order like their bit
// patterns, so an integer atomicMax is exact).  Units are dealt to the 128 threads per kernel size, K compile-time:
// no divergent trip counts, 17 load instructions per warp and word instead of up to 36 serial ones per thread.
template <int K>
__device__ __forceinline__ void char_cnn_units(const float* __restrict__ ctab, const float* __restrict__ cbias,
                                               const int* __restrict__ ch, int C, int nc, int tid, int* __restrict__ mx) {
  constexpr int CHN = 10 * K, NP2 = CHN / 2;     // output channels of this kernel size, in pairs
  constexpr int COFF = 5 * K * (K - 1);          // first output channel: 0, 10, 30, 60
  const float* T = ctab + char_tab_offset(K, nc);
  const int units = NP2 * (C - K + 1);
  for (int u = tid; u < units; u += 128) {
    const int p = u / NP2, o2 = u - p * NP2;
    float2 v = __ldg(reinterpret_cast<const float2*>(cbias + COFF) + o2);
#pragma unroll
    for (int j = 0; j < K; ++j) {
      const float2 t = __ldg(reinterpret_cast<const float2*>(T + (j * nc + ch[p + j]) * CHN) + o2);
      v.x += t.x; v.y += t.y;
    }
    atomicMax(mx + COFF + 2 * o2, __float_as_int(fmaxf(v.x, 0.f)));
    atomicMax(mx + COFF + 2 * o2 + 1, __float_as_int(fmaxf(v.y, 0.f)));
  }
}

__global__ void __launch_bounds__(128) embed_text_kernel(const int64_t* __restrict__ word_ids,
                                                         const int64_t* __restrict__ char_ids, int C,
                                                         const float* __restrict__ pad, const float* __restrict__ unk,
                                                         const float* __restrict__ glove,
                                                         const float* __restrict__ table, int num_words, int nc,
                                                         const float* __restrict__ ctab,
                                                         const float* __restrict__ cbias, float* __restrict__ out) {
  __shared__ int ch[64];
  __shared__ int mx[100];
  const long long word = blockIdx.x;
  const int tid = threadIdx.x;
  if (tid < C) {
    long long c = char_ids[word * C + tid];
    ch[tid] = (int)(c < 0 ? 0 : (c >= nc ? nc - 1 : c));
  }
  if (tid < 100) mx[tid] = 0;   // max over positions of ReLU(.) is >= 0 and at least one position exists (C >= 4)
  long long id = word_ids[word];
  id = id < 0 ? 0 : (id >= num_words ? num_words - 1 : id);
  const float* src = table ? table + id * 300 : (id == 0 ? pad : (id == 1 ? unk : glove + (id - 2) * 300));
  float wv[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) wv[i] = tid + i * 128 < 300 ? __ldg(src + tid + i * 128) : 0.f;   // in flight under the char CNN
  __syncthreads();
  char_cnn_units<4>(ctab, cbias, ch, C, nc, tid, mx);
  char_cnn_units<3>(ctab, cbias, ch, C, nc, tid, mx);
  char_cnn_units<2>(ctab, cbias, ch, C, nc, tid, mx);
  char_cnn_units<1>(ctab, cbias, ch, C, nc, tid, mx);
#pragma unroll
  for (int i = 0; i < 3; ++i)
    if (tid + i * 128 < 300) out[word * 400 + tid + i * 128] = wv[i];
  __syncthreads();
  if (tid < 100) out[word * 400 + 300 + tid] = __int_as_float(mx[tid]);
}

cudaError_t launch_embed_text(const int64_t* word_ids, const int64_t* char_ids, long long n_words, int C,
                              const float* pad, const float* unk, const float* glove, const float* table,
                              int num_words, int num_chars, const float* ctab, const float* cbias, float* out,
                              cudaStream_t st) {
  if (n_words <= 0) return cudaSuccess;
  if ((reinterpret_cast<uintptr_t>(ctab) | reinterpret_cast<uintptr_t>(cbias)) & 7) return cudaErrorMisalignedAddress;
  embed_text_kernel<<<(unsigned)n_words, 128, 0, st>>>(word_ids, char_ids, C, pad, unk, glove, table, num_words,
                                                       num_chars, ctab, cbias, out);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Warp-cooperative attention core shared by DualMultiAttention and the predictor's batch-axis attention.
// A warp processes 4 query rows against `nk` keys held in shared memory:
//   Kt [32][ldk]  keys transposed (d-major)   -> scores: lane owns 4 consecutive keys of a 128-key tile,
//                                               one LDS.128 of keys + one broadcast LDS.128 of the 4 queries
//                                               feed 16 FMAs
//   V  [nk][32]                               -> P.V: lane = (4 dims, key residue mod 4), 2 LDS.128 per 16 FMAs,
//                                               then a 2-step butterfly over the key residues
// score(qi, j, dot) supplies the model-specific scaling and additive mask.  Softmax is fp32 exp/sum like
// torch.softmax; a fully masked row (all scores == -1e30) yields the uniform distribution.
// ------------------------------------------------------------------------------------------------
template <class ScoreFn>
__device__ __forceinline__ void warp_attend4(const float* __restrict__ qt /*[32][4]*/, const float* __restrict__ Kt,
                                             int ldk, const float* __restrict__ V, int nk,
                                             float* __restrict__ ps /*[nk][4]*/, ScoreFn score, int lane,
                                             float4& out /* dims 4*(lane&7).. of query (lane>>3) */) {
  for (int j0 = 0; j0 < nk; j0 += 128) {
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
#pragma unroll 8
    for (int d = 0; d < SQ_HD; ++d) {
      const float4 k4 = ld4(Kt + d * ldk + j0 + 4 * lane);
      const float4 q4 = ld4(qt + d * 4);
      const float kk[4] = {k4.x, k4.y, k4.z, k4.w};
      const float qq[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = fmaf(qq[a], kk[b], acc[a][b]);
    }
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int j = j0 + 4 * lane + b;
      if (j < nk)
        st4(ps + j * 4, make_float4(score(0, j, acc[0][b]), score(1, j, acc[1][b]), score(2, j, acc[2][b]),
                                    score(3, j, acc[3][b])));
    }
  }
  __syncwarp();
  // softmax over keys for the 4 queries at once (component q of each float4)
  float4 mx = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  for (int j = lane; j < nk; j += 32) {
    const float4 s = ld4(ps + j * 4);
    mx.x = fmaxf(mx.x, s.x); mx.y = fmaxf(mx.y, s.y); mx.z = fmaxf(mx.z, s.z); mx.w = fmaxf(mx.w, s.w);
  }
  mx.x = warp_max(mx.x); mx.y = warp_max(mx.y); mx.z = warp_max(mx.z); mx.w = warp_max(mx.w);
  float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int j = lane; j < nk; j += 32) {
    float4 s = ld4(ps + j * 4);
    s.x = expf(s.x - mx.x); s.y = expf(s.y - mx.y); s.z = expf(s.z - mx.z); s.w = expf(s.w - mx.w);
    sum.x += s.x; sum.y += s.y; sum.z += s.z; sum.w += s.w;
    st4(ps + j * 4, s);
  }
  sum.x = warp_sum(sum.x); sum.y = warp_sum(sum.y); sum.z = warp_sum(sum.z); sum.w = warp_sum(sum.w);
  __syncwarp();
  // P.V
  const int dg = lane & 7, jg = lane >> 3;
  float o[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) o[a][b] = 0.f;
  for (int j = jg; j < nk; j += 4) {
    const float4 p4 = ld4(ps + j * 4);
    const float4 v4 = ld4(V + j * SQ_HD + 4 * dg);
    const float pp[4] = {p4.x, p4.y, p4.z, p4.w};
    const float vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) o[a][b] = fmaf(pp[a], vv[b], o[a][b]);
  }
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      o[a][b] += __shfl_xor_sync(0xffffffffu, o[a][b], 8);
      o[a][b] += __shfl_xor_sync(0xffffffffu, o[a][b], 16);
    }
  const float sm[4] = {sum.x, sum.y, sum.z, sum.w};
  float r[4];
#pragma unroll
  for (int b = 0; b < 4; ++b) {  // lane group jg publishes query jg
    r[b] = jg == 0 ? o[0][b] : (jg == 1 ? o[1][b] : (jg == 2 ? o[2][b] : o[3][b]));
  }
  const float inv = 1.0f / (jg == 0 ? sm[0] : (jg == 1 ? sm[1] : (jg == 2 ? sm[2] : sm[3])));
  out = make_float4(r[0] * inv, r[1] * inv, r[2] * inv, r[3] * inv);
  __syncwarp();
}

__device__ __forceinline__ int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Stage keys (transposed) and values of one head from a row-major projection buffer into shared memory.
__device__ __forceinline__ void stage_kv(const float* __restrict__ src, long long row0, long long row_stride, int ld,
                                         int kcol, int vcol, int n, float* Kt, int ldk, float* V) {
  for (int idx = threadIdx.x; idx < n * SQ_HD; idx += blockDim.x) {
    const int j = idx >> 5, d = idx & 31;
    const float* rowp = src + (row0 + (long long)j * row_stride) * ld;
    Kt[d * ldk + j] = __ldg(rowp + kcol + d);
    V[j * SQ_HD + d] = __ldg(rowp + vcol + d);
  }
}

// ------------------------------------------------------------------------------------------------
// DualMultiAttention core (models/layers.py:339-367): for every (sample, head, direction)
//   self : softmax_j(q.fk_j / sqrt(32) + (1 - m_f[i] m_f[j]) * -1e30) . fv
//   cross: softmax_j(q.tk_j / sqrt(32) + (1 - m_f[i] m_t[j]) * -1e30) . tv
// direction 0: from = video rows, to = text rows; direction 1 the reverse (models/SeqPAN.py:64-70; both
// directions share the block's weights, so their projections live in the same joint row buffers).
// ------------------------------------------------------------------------------------------------
size_t dual_attention_smem(int L, int T) {
  const int mx = L > T ? L : T;
  auto rup = [](int x) { return (x + 127) / 128 * 128 + 4; };
  size_t fl = (size_t)32 * rup(L) + (size_t)L * 32 + (size_t)32 * rup(T) + (size_t)T * 32 + L + T + 4;
  fl += 8 * (128 + (size_t)4 * mx);
  return fl * sizeof(float);
}

__global__ void __launch_bounds__(256) dual_attention_kernel(DualAttnArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int b = blockIdx.x, h = blockIdx.y, dir = blockIdx.z;
  const int F = dir == 0 ? a.L : a.T, S = dir == 0 ? a.T : a.L;
  const long long Mv = (long long)a.B * a.L;
  const long long frow0 = dir == 0 ? (long long)b * a.L : Mv + (long long)b * a.T;
  const long long trow0 = dir == 0 ? Mv + (long long)b * a.T : (long long)b * a.L;
  const float* fmask = dir == 0 ? a.vmask + (long long)b * a.L : a.tmask + (long long)b * a.T;
  const float* tmask = dir == 0 ? a.tmask + (long long)b * a.T : a.vmask + (long long)b * a.L;
  const int ldF = round_up(F, 128) + 4, ldS = round_up(S, 128) + 4;
  const int mxk = F > S ? F : S;
  float* Kts = smem;
  float* Vs = Kts + 32 * ldF;
  float* Ktx = Vs + F * 32;
  float* Vx = Ktx + 32 * ldS;
  float* mf = Vx + S * 32;
  float* mt = mf + F;
  float* wbase = mt + S;
  wbase += (4 - ((wbase - smem) & 3)) & 3;  // 16-byte align the per-warp area
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* qt = wbase + w * (128 + 4 * mxk);
  float* ps = qt + 128;

  stage_kv(a.qkv, frow0, 1, 384, 128 + h * SQ_HD, 256 + h * SQ_HD, F, Kts, ldF, Vs);
  stage_kv(a.tkv, trow0, 1, 256, h * SQ_HD, 128 + h * SQ_HD, S, Ktx, ldS, Vx);
  for (int i = threadIdx.x; i < F; i += blockDim.x) mf[i] = fmask[i];
  for (int i = threadIdx.x; i < S; i += blockDim.x) mt[i] = tmask[i];
  __syncthreads();

  const float sqrt_hd = sqrtf((float)SQ_HD);
  for (int i0 = w * 4; i0 < F; i0 += 32) {
    {  // this warp's 4 queries, transposed to [d][q]
      const int qi = lane >> 3, d4 = (lane & 7) * 4;
      const int i = min(i0 + qi, F - 1);
      const float4 q = ldg4(a.qkv + (frow0 + i) * 384 + h * SQ_HD + d4);
      qt[(d4 + 0) * 4 + qi] = q.x; qt[(d4 + 1) * 4 + qi] = q.y;
      qt[(d4 + 2) * 4 + qi] = q.z; qt[(d4 + 3) * 4 + qi] = q.w;
    }
    __syncwarp();
    float mq[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) mq[q] = mf[min(i0 + q, F - 1)];
    const int qi = lane >> 3, d4 = (lane & 7) * 4;
    float4 o;
    warp_attend4(qt, Kts, ldF, Vs, F, ps,
                 [&](int q, int j, float dot) { return dot / sqrt_hd + (1.0f - mq[q] * mf[j]) * SQ_MASK; }, lane, o);
    auto put = [&](float* f32, void* bf, float4 v) {
      const long long off = (frow0 + i0 + qi) * SQ_D + h * SQ_HD + d4;
      if (bf) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&lo);
        pk.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(bf) + off) = pk;
      } else {
        st4(f32 + off, v);
      }
    };
    if (i0 + qi < F) put(a.sa, a.sa_bf16, o);
    warp_attend4(qt, Ktx, ldS, Vx, S, ps,
                 [&](int q, int j, float dot) { return dot / sqrt_hd + (1.0f - mq[q] * mt[j]) * SQ_MASK; }, lane, o);
    if (i0 + qi < F) put(a.xa, a.xa_bf16, o);
  }
}

cudaError_t launch_dual_attention(const DualAttnArgs& a, cudaStream_t st) {
  const size_t smem = dual_attention_smem(a.L, a.T);
  cudaError_t e = cudaFuncSetAttribute(dual_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  dual_attention_kernel<<<dim3(a.B, SQ_H, 2), 256, smem, st>>>(a);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Cross gating and the masked sigmoid gate of DualMultiAttention (models/layers.py:374, 380)
// ------------------------------------------------------------------------------------------------
__global__ void gate_combine_kernel(const float4* __restrict__ sg, const float4* __restrict__ x,
                                    const float4* __restrict__ xg, const float4* __restrict__ s,
                                    float4* __restrict__ out, long long n4) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const float4 a = sg[i], b = x[i], c = xg[i], d = s[i];
  out[i] = make_float4(a.x * b.x + c.x * d.x, a.y * b.y + c.y * d.y, a.z * b.z + c.z * d.z, a.w * b.w + c.w * d.w);
}
cudaError_t launch_gate_combine(const float* sg, const float* x, const float* xg, const float* s, float* out,
                                long long n4, cudaStream_t st) {
  if (n4 <= 0) return cudaSuccess;
  gate_combine_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>((const float4*)sg, (const float4*)x,
                                                                    (const float4*)xg, (const float4*)s,
                                                                    (float4*)out, n4);
  return cudaGetLastError();
}

// y = sigmoid(scores + (-1e30)(1 - m_f)) * values, scva = [scores | values] per row (256 columns)
__global__ void sigmoid_gate_kernel(const float* __restrict__ scva, const float* __restrict__ rowmask,
                                    float* __restrict__ y, long long M) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float mk = SQ_MASK * (1.0f - rowmask[row]);
  const float4 sc = ldg4(scva + row * 256 + lane * 4), va = ldg4(scva + row * 256 + 128 + lane * 4);
  auto sig = [&](float v) { return 1.0f / (1.0f + expf(-(v + mk))); };
  st4(y + row * SQ_D + lane * 4, make_float4(sig(sc.x) * va.x, sig(sc.y) * va.y, sig(sc.z) * va.z, sig(sc.w) * va.w));
}
cudaError_t launch_sigmoid_gate(const float* scva, const float* rowmask, float* y, long long M, cudaStream_t st) {
  if (M <= 0) return cudaSuccess;
  sigmoid_gate_kernel<<<(unsigned)((M + 7) / 8), 256, 0, st>>>(scva, rowmask, y, M);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// CQAttention up to the concat (models/layers.py:417-437): trilinear scores, row softmax under the query
// mask, column softmax under the context mask, c2q = S1.Q, q2c = S1.S2^T.C, and the 512-wide
// [C, c2q, C*c2q, C*q2c] row handed to cqa_linear.  One CTA per (sample, direction); score matrices live in
// shared memory, the 128-wide rows are streamed through L1 (each warp reads whole 512-byte rows).
// q2c is evaluated as S1.(S2^T.C) when the context is the long side and as (S1.S2^T).C otherwise.
// ------------------------------------------------------------------------------------------------
constexpr int CQLD = 132;  // padded fp32 row stride of the staged context/query rows (conflict-free float4 by row)
static size_t cq_smem_floats(int F, int S, int staged_rows) {
  const size_t ext = F >= S ? (size_t)S * 128 : (size_t)F * F;  // R[S][128] or G[F][F]
  return (size_t)staged_rows * CQLD + 2 * (size_t)F * (S + 1) + F + S + 8 + 128 + ext;
}
static size_t cq_smem_bytes(int L, int T, bool stage_video) {
  const int rows = T + (stage_video ? L : 0);
  const size_t a = cq_smem_floats(L, T, rows), b = cq_smem_floats(T, L, rows);
  return (a > b ? a : b) * sizeof(float);
}
// smallest configuration that must fit: text rows staged, video rows streamed through L1
size_t cq_attention_smem(int L, int T) { return cq_smem_bytes(L, T, false); }

// Work is dealt by warp / thread index with the block size as stride, so the result does not depend on the block size:
// 256 threads when several CTAs fit an SM, 1024 when the staged rows (L > 128) leave room for one CTA only.
template <int NT>
__global__ void __launch_bounds__(NT) cq_attention_kernel(CqArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int b = blockIdx.x, dir = blockIdx.y;
  const int F = dir == 0 ? a.L : a.T, S = dir == 0 ? a.T : a.L;
  const long long Mv = (long long)a.B * a.L;
  const float* C = a.x + (dir == 0 ? (long long)b * a.L : Mv + (long long)b * a.T) * SQ_D;
  const float* Q = a.x + (dir == 0 ? Mv + (long long)b * a.T : (long long)b * a.L) * SQ_D;
  const float* cmask = dir == 0 ? a.vmask + (long long)b * a.L : a.tmask + (long long)b * a.T;
  const float* qmask = dir == 0 ? a.tmask + (long long)b * a.T : a.vmask + (long long)b * a.L;
  float* out = a.cat[dir] + (dir == 0 ? (long long)b * a.L : (long long)b * a.T) * 512;
  const bool reassoc = F >= S;
  const int lds = S + 1;
  // the video rows are the context in direction 0 and the query in direction 1
  const bool stageC = dir == 1 || a.stage_video, stageQ = dir == 0 || a.stage_video;
  float* Cst = smem;                                   // [F][CQLD] context rows (if staged)
  float* Qst = Cst + (stageC ? F * CQLD : 0);          // [S][CQLD] query rows (if staged)
  float* A = Qst + (stageQ ? S * CQLD : 0);            // [F][S+1] raw scores, then row softmax S1
  const float* Cs = stageC ? Cst : C;
  const float* Qs = stageQ ? Qst : Q;
  const int cld = stageC ? CQLD : SQ_D, qld = stageQ ? CQLD : SQ_D;
  float* Bm = A + F * lds;           // [F][S+1] column softmax S2
  float* sub0 = Bm + F * lds;        // [F] C.w4C
  float* sub1 = sub0 + F;            // [S] Q.w4Q
  float* wms = sub1 + S;
  wms += (4 - ((wms - smem) & 3)) & 3;  // [128] w4mlu (16-byte aligned)
  float* ext = wms + 128;               // R [S][128] or G [F][F]
  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
  constexpr int nt = NT, nw = NT >> 5;
  const float4 w4c = ldg4(a.w4c[dir] + lane * 4), w4q = ldg4(a.w4q[dir] + lane * 4);
  if (tid < 128) wms[tid] = __ldg(a.w4mlu[dir] + tid);

  // stage both row sets once (coalesced 512-byte rows) and form the rank-1 terms of the trilinear score
  for (int i = w; i < F; i += nw) {
    const float4 c = ldg4(C + (long long)i * SQ_D + lane * 4);
    if (stageC) st4(Cst + i * CQLD + lane * 4, c);
    const float s0 = warp_sum(dot4(c, w4c));
    if (lane == 0) sub0[i] = s0;
  }
  for (int j = w; j < S; j += nw) {
    const float4 qv = ldg4(Q + (long long)j * SQ_D + lane * 4);
    if (stageQ) st4(Qst + j * CQLD + lane * 4, qv);
    const float s1 = warp_sum(dot4(qv, w4q));
    if (lane == 0) sub1[j] = s1;
  }
  __syncthreads();
  // scores: four context rows x one query row per thread iteration (the query row and the weights are read once for
  // the four pairs), 128-long dot products out of shared memory; every pair sums in the same order as alone
  {
    const float* wm = wms;
    const int F4 = (F + 3) >> 2;
    for (int pidx = tid; pidx < F4 * S; pidx += nt) {
      const int i4 = pidx / S, j = pidx - i4 * S;
      const int i0 = i4 * 4;
      const float* cr[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) cr[u] = Cs + min(i0 + u, F - 1) * cld;   // rows behind F: recomputed, not stored
      const float* qr = Qs + j * qld;
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
      for (int d = 0; d < SQ_D; d += 4) {
        const float4 qv = ld4(qr + d), wv = ld4(wm + d);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float4 c = ld4(cr[u] + d);
          acc[u] = fmaf(c.x * wv.x, qv.x, acc[u]);
          acc[u] = fmaf(c.y * wv.y, qv.y, acc[u]);
          acc[u] = fmaf(c.z * wv.z, qv.z, acc[u]);
          acc[u] = fmaf(c.w * wv.w, qv.w, acc[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i0 + u < F) A[(i0 + u) * lds + j] = (sub0[i0 + u] + sub1[j]) + acc[u];
    }
  }
  __syncthreads();
  // S2 = softmax over the context axis (dim=1) of scores + mask_c   (models/layers.py:420)
  for (int j = w; j < S; j += nw) {
    float mx = -INFINITY;
    for (int i = lane; i < F; i += 32) mx = fmaxf(mx, A[i * lds + j] + SQ_MASK * (1.0f - cmask[i]));
    mx = warp_max(mx);
    float sum = 0.f;
    for (int i = lane; i < F; i += 32) {
      const float e = expf(A[i * lds + j] + SQ_MASK * (1.0f - cmask[i]) - mx);
      Bm[i * lds + j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    for (int i = lane; i < F; i += 32) Bm[i * lds + j] = Bm[i * lds + j] / sum;
  }
  __syncthreads();
  // S1 = softmax over the query axis (dim=2) of scores + mask_q, in place   (models/layers.py:419)
  for (int i = w; i < F; i += nw) {
    float mx = -INFINITY;
    for (int j = lane; j < S; j += 32) mx = fmaxf(mx, A[i * lds + j] + SQ_MASK * (1.0f - qmask[j]));
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < S; j += 32) {
      const float e = expf(A[i * lds + j] + SQ_MASK * (1.0f - qmask[j]) - mx);
      A[i * lds + j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    for (int j = lane; j < S; j += 32) A[i * lds + j] = A[i * lds + j] / sum;
  }
  __syncthreads();
  if (reassoc) {
    float* R = ext;  // R[j] = sum_i S2[i][j] C[i]; four j per warp: one read of C[i] serves four rows of R
    for (int j0 = w * 4; j0 < S; j0 += nw * 4) {
      float4 r[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) r[u] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
      for (int i = 0; i < F; ++i) {
        const float4 c = ld4(Cs + i * cld + lane * 4);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float p = Bm[i * lds + min(j0 + u, S - 1)];
          r[u].x = fmaf(p, c.x, r[u].x); r[u].y = fmaf(p, c.y, r[u].y); r[u].z = fmaf(p, c.z, r[u].z); r[u].w = fmaf(p, c.w, r[u].w);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (j0 + u < S) st4(R + (j0 + u) * SQ_D + lane * 4, r[u]);
    }
  } else {
    float* G = ext;  // G[i][i'] = sum_j S1[i][j] S2[i'][j]
    for (int idx = tid; idx < F * F; idx += nt) {
      const int i = idx / F, ip = idx % F;
      float g = 0.f;
      for (int j = 0; j < S; ++j) g = fmaf(A[i * lds + j], Bm[ip * lds + j], g);
      G[idx] = g;
    }
  }
  __syncthreads();
  // four context rows per warp: one read of Q[j] (and R[j]) serves the four rows
  for (int i0 = w * 4; i0 < F; i0 += nw * 4) {
    float4 c2q[4], q2c[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { c2q[u] = make_float4(0.f, 0.f, 0.f, 0.f); q2c[u] = make_float4(0.f, 0.f, 0.f, 0.f); }
#pragma unroll 2
    for (int j = 0; j < S; ++j) {
      const float4 qv = ld4(Qs + j * qld + lane * 4);
      float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
      if (reassoc) r = ld4(ext + j * SQ_D + lane * 4);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float p = A[min(i0 + u, F - 1) * lds + j];
        c2q[u].x = fmaf(p, qv.x, c2q[u].x); c2q[u].y = fmaf(p, qv.y, c2q[u].y); c2q[u].z = fmaf(p, qv.z, c2q[u].z); c2q[u].w = fmaf(p, qv.w, c2q[u].w);
        if (reassoc) {
          q2c[u].x = fmaf(p, r.x, q2c[u].x); q2c[u].y = fmaf(p, r.y, q2c[u].y); q2c[u].z = fmaf(p, r.z, q2c[u].z); q2c[u].w = fmaf(p, r.w, q2c[u].w);
        }
      }
    }
    if (!reassoc) {
      for (int ip = 0; ip < F; ++ip) {
        const float4 cc = ld4(Cs + ip * cld + lane * 4);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float g = ext[min(i0 + u, F - 1) * F + ip];
          q2c[u].x = fmaf(g, cc.x, q2c[u].x); q2c[u].y = fmaf(g, cc.y, q2c[u].y); q2c[u].z = fmaf(g, cc.z, q2c[u].z); q2c[u].w = fmaf(g, cc.w, q2c[u].w);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u;
      if (i >= F) break;
      const float4 c = ld4(Cs + i * cld + lane * 4);
      float* o = out + (long long)i * 512 + lane * 4;
      st4(o, c);
      st4(o + 128, c2q[u]);
      st4(o + 256, make_float4(c.x * c2q[u].x, c.y * c2q[u].y, c.z * c2q[u].z, c.w * c2q[u].w));
      st4(o + 384, make_float4(c.x * q2c[u].x, c.y * q2c[u].y, c.z * q2c[u].z, c.w * q2c[u].w));
    }
  }
}

cudaError_t launch_cq_attention(const CqArgs& a_in, cudaStream_t st) {
  CqArgs a = a_in;
  a.stage_video = cq_smem_bytes(a.L, a.T, true) <= 200 * 1024 ? 1 : 0;
  const size_t smem = cq_smem_bytes(a.L, a.T, a.stage_video != 0);
  const int nt = smem > 100 * 1024 ? 1024 : 256;   // block size 1024 when only one CTA fits an SM
  auto launch = [&](auto kern) -> cudaError_t {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    kern<<<dim3(a.B, 2), nt, smem, st>>>(a);
    return cudaSuccess;
  };
  cudaError_t e = nt == 256 ? launch(cq_attention_kernel<256>) : launch(cq_attention_kernel<1024>);
  if (e != cudaSuccess) return e;
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// WeightedPool + tile (models/layers.py:447-453, 463-466): pooled = sum_t softmax_t(x_t.w + mask) x_t,
// written into columns [128,256) of every row of the sample in the concat buffer.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) pool_tile_kernel(const float* __restrict__ v2t, const float* __restrict__ tmask,
                                                        const float* __restrict__ pw, float* __restrict__ cat2, int L,
                                                        int T) {
  __shared__ float al[SEQPAN_MAX_VLEN];
  const int b = blockIdx.x, tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
  const float* x = v2t + (long long)b * T * SQ_D;
  const float4 w4 = ldg4(pw + lane * 4);
  for (int t = w; t < T; t += 4) {
    const float s = warp_sum(dot4(ldg4(x + (long long)t * SQ_D + lane * 4), w4));
    if (lane == 0) al[t] = s + SQ_MASK * (1.0f - tmask[(long long)b * T + t]);
  }
  __syncthreads();
  float mx = -INFINITY;
  for (int t = 0; t < T; ++t) mx = fmaxf(mx, al[t]);
  float sum = 0.f;
  for (int t = 0; t < T; ++t) sum += expf(al[t] - mx);
  float p = 0.f;
  for (int t = 0; t < T; ++t) p = fmaf(expf(al[t] - mx) / sum, __ldg(x + (long long)t * SQ_D + tid), p);
  for (int l = 0; l < L; ++l) cat2[((long long)b * L + l) * 256 + 128 + tid] = p;
}
cudaError_t launch_pool_tile(const float* v2t, const float* tmask, const float* pool_w, float* cat2, int B, int L,
                             int T, cudaStream_t st) {
  pool_tile_kernel<<<B, 128, 0, st>>>(v2t, tmask, pool_w, cat2, L, T);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Match head (models/SeqPAN.py:78-82): Conv1D(128->4), gumbel softmax with injected noise and tau = 0.3,
// soft label embedding, (fuse + soft) * vmask.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) match_head_kernel(const float* __restrict__ fuse, const float* __restrict__ wm,
                                                         const float* __restrict__ bm, const float* __restrict__ gumbel,
                                                         const float* __restrict__ emb, const float* __restrict__ vmask,
                                                         float* __restrict__ match_score, float* __restrict__ fuse2,
                                                         long long M) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float4 f = ldg4(fuse + row * SQ_D + lane * 4);
  float y[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float ml = warp_sum(dot4(f, ldg4(wm + c * SQ_D + lane * 4))) + __ldg(bm + c);
    y[c] = (ml + __ldg(gumbel + row * 4 + c)) / 0.3f;
  }
  const float mx = fmaxf(fmaxf(y[0], y[1]), fmaxf(y[2], y[3]));
  float e[4], sum = 0.f;
#pragma unroll
  for (int c = 0; c < 4; ++c) { e[c] = expf(y[c] - mx); sum += e[c]; }
#pragma unroll
  for (int c = 0; c < 4; ++c) e[c] = e[c] / sum;
  if (lane < 4) match_score[row * 4 + lane] = lane == 0 ? e[0] : (lane == 1 ? e[1] : (lane == 2 ? e[2] : e[3]));
  const float mk = vmask[row];
  float o[4] = {f.x, f.y, f.z, f.w};
#pragma unroll
  for (int d = 0; d < 4; ++d) {
    const float4 le = ldg4(emb + (lane * 4 + d) * 4);  // label_embs [128,4]
    float soft = e[0] * le.x;
    soft = fmaf(e[1], le.y, soft);
    soft = fmaf(e[2], le.z, soft);
    soft = fmaf(e[3], le.w, soft);
    o[d] = (o[d] + soft) * mk;
  }
  st4(fuse2 + row * SQ_D + lane * 4, make_float4(o[0], o[1], o[2], o[3]));
}
cudaError_t launch_match_head(const float* fuse, const float* wm, const float* bm, const float* gumbel,
                              const float* label_embs, const float* vmask, float* match_score, float* fuse2,
                              long long M, cudaStream_t st) {
  if (M <= 0) return cudaSuccess;
  match_head_kernel<<<(unsigned)((M + 7) / 8), 256, 0, st>>>(fuse, wm, bm, gumbel, label_embs, vmask, match_score,
                                                             fuse2, M);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// TopSelfAttention2 core (models/layers.py:567-574): nn.MultiheadAttention(batch_first=False) applied to
// [B,L,D] attends ACROSS the batch for each (position l, head): softmax_b'((q_b/sqrt(32)).k_b' + vmask[b',l]).v
// One CTA per (l, head) keeps all B keys/values in shared memory.
// ------------------------------------------------------------------------------------------------
size_t batch_attention_smem(int B) {
  const int ldk = (B + 127) / 128 * 128 + 4;
  return ((size_t)32 * ldk + (size_t)B * 32 + B + 4 + 8 * (128 + (size_t)4 * B)) * sizeof(float);
}

__global__ void __launch_bounds__(256) batch_attention_kernel(const float* __restrict__ qkv,
                                                              const float* __restrict__ vmask,
                                                              float* __restrict__ out, void* out_bf16, int B, int L) {
  extern __shared__ __align__(16) float smem[];
  const int l = blockIdx.x, h = blockIdx.y;
  const int ldk = round_up(B, 128) + 4;
  float* Kt = smem;
  float* V = Kt + 32 * ldk;
  float* mb = V + B * 32;
  float* wbase = mb + B;
  wbase += (4 - ((wbase - smem) & 3)) & 3;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* qt = wbase + w * (128 + 4 * B);
  float* ps = qt + 128;
  stage_kv(qkv, l, L, 384, 128 + h * SQ_HD, 256 + h * SQ_HD, B, Kt, ldk, V);
  for (int j = threadIdx.x; j < B; j += blockDim.x) mb[j] = vmask[(long long)j * L + l];
  __syncthreads();
  const float scaling = 0.17677669529663687f;  // math.sqrt(1.0 / head_dim) in F.multi_head_attention_forward
  for (int i0 = w * 4; i0 < B; i0 += 32) {
    const int qi = lane >> 3, d4 = (lane & 7) * 4;
    {
      const int i = min(i0 + qi, B - 1);
      const float4 q = ldg4(qkv + ((long long)i * L + l) * 384 + h * SQ_HD + d4);
      qt[(d4 + 0) * 4 + qi] = q.x * scaling; qt[(d4 + 1) * 4 + qi] = q.y * scaling;
      qt[(d4 + 2) * 4 + qi] = q.z * scaling; qt[(d4 + 3) * 4 + qi] = q.w * scaling;
    }
    __syncwarp();
    float4 o;
    warp_attend4(qt, Kt, ldk, V, B, ps, [&](int, int j, float dot) { return dot + mb[j]; }, lane, o);
    if (i0 + qi < B) {
      const long long off = ((long long)(i0 + qi) * L + l) * SQ_D + h * SQ_HD + d4;
      if (out_bf16) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&lo);
        pk.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(out_bf16) + off) = pk;
      } else {
        st4(out + off, o);
      }
    }
  }
}
cudaError_t launch_batch_attention(const float* qkv, const float* vmask, float* out, void* out_bf16, int B, int L,
                                   cudaStream_t st) {
  const size_t smem = batch_attention_smem(B);
  cudaError_t e = cudaFuncSetAttribute(batch_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  batch_attention_kernel<<<dim3(L, SQ_H), 256, smem, st>>>(qkv, vmask, out, out_bf16, B, L);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Conv1D(128 -> 1) heads (models/layers.py:669-670) and the joint row mask
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rowdot_kernel(const float* __restrict__ x, int ldx, const float* __restrict__ w,
                                                     const float* __restrict__ b, float* __restrict__ out, long long M) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float s = warp_sum(dot4(ldg4(x + row * ldx + lane * 4), ldg4(w + lane * 4)));
  if (lane == 0) out[row] = s + __ldg(b);
}
cudaError_t launch_rowdot(const float* x, int ldx, const float* w, const float* b, float* out, long long M,
                          cudaStream_t st) {
  if (M <= 0) return cudaSuccess;
  rowdot_kernel<<<(unsigned)((M + 7) / 8), 256, 0, st>>>(x, ldx, w, b, out, M);
  return cudaGetLastError();
}

__global__ void build_rowmask_kernel(const float* __restrict__ vmask, long long nv, const float* __restrict__ tmask,
                                     long long nt, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nv) out[i] = vmask[i];
  else if (i < nv + nt) out[i] = tmask[i - nv];
}
cudaError_t launch_build_rowmask(const float* vmask, long long nv, const float* tmask, long long nt, float* out,
                                 cudaStream_t st) {
  build_rowmask_kernel<<<(unsigned)((nv + nt + 255) / 256), 256, 0, st>>>(vmask, nv, tmask, nt, out);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Span decode (utils/engine.py:28-44 infer_basic; models/layers.py:549-557 extract_index).
// The reference materialises outer[b,i,j] = sp[i]*ep[j], applies triu and takes two independent argmaxes.
// fp32 multiplication by a non-negative number is monotone, so max_{j>=i} sp[i]*ep[j] = sp[i]*max_{j>=i} ep[j]
// exactly: the decode is O(L) with a suffix max of ep and a prefix max of sp (SURVEY.md A.7).  Ties resolve to
// the lowest index like torch.max on CPU.  One warp per sample.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) span_decode_kernel(const float* __restrict__ s, const float* __restrict__ e,
                                                          const float* __restrict__ vmask, int B, int L,
                                                          int64_t* __restrict__ si, int64_t* __restrict__ ei,
                                                          float* __restrict__ fracs) {
  __shared__ float sp[4][SEQPAN_MAX_VLEN], ep[4][SEQPAN_MAX_VLEN], aux[4][SEQPAN_MAX_VLEN];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * 4 + w;
  if (b >= B) return;
  float ms = -INFINITY, me = -INFINITY, nvalid = 0.f;
  for (int i = lane; i < L; i += 32) {
    float a = s[(long long)b * L + i], c = e[(long long)b * L + i];
    if (vmask) {
      const float m = vmask[(long long)b * L + i];
      a = a + SQ_MASK * (1.0f - m);
      c = c + SQ_MASK * (1.0f - m);
      nvalid += m;
    }
    sp[w][i] = a; ep[w][i] = c;
    ms = fmaxf(ms, a); me = fmaxf(me, c);
  }
  ms = warp_max(ms); me = warp_max(me); nvalid = warp_sum(nvalid);
  float ss = 0.f, se = 0.f;
  for (int i = lane; i < L; i += 32) {
    const float a = expf(sp[w][i] - ms), c = expf(ep[w][i] - me);
    sp[w][i] = a; ep[w][i] = c;
    ss += a; se += c;
  }
  ss = warp_sum(ss); se = warp_sum(se);
  for (int i = lane; i < L; i += 32) { sp[w][i] = sp[w][i] / ss; ep[w][i] = ep[w][i] / se; }
  __syncwarp();
  // start index: argmax_i sp[i] * max_{j>=i} ep[j]
  {   // suffix max of ep, 32 positions per step: warp scan + carry from the chunk behind
    float carry = 0.f;
    for (int base = ((L - 1) >> 5) << 5; base >= 0; base -= 32) {
      const int i = base + lane;
      float v = i < L ? ep[w][i] : 0.f;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const float t = __shfl_down_sync(0xffffffffu, v, o); if (lane + o < 32) v = fmaxf(v, t); }
      v = fmaxf(v, carry);
      if (i < L) aux[w][i] = v;
      carry = __shfl_sync(0xffffffffu, v, 0);
    }
  }
  __syncwarp();
  float bv = -1.f; int bi = 0x7fffffff;
  for (int i = lane; i < L; i += 32) { const float v = sp[w][i] * aux[w][i]; if (v > bv) { bv = v; bi = i; } }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o); const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  const int start = bi;
  __syncwarp();
  // end index: argmax_j ep[j] * max_{i<=j} sp[i]
  {   // prefix max of sp
    float carry = 0.f;
    for (int base = 0; base < L; base += 32) {
      const int i = base + lane;
      float v = i < L ? sp[w][i] : 0.f;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const float t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v = fmaxf(v, t); }
      v = fmaxf(v, carry);
      if (i < L) aux[w][i] = v;
      carry = __shfl_sync(0xffffffffu, v, 31);
    }
  }
  __syncwarp();
  bv = -1.f; bi = 0x7fffffff;
  for (int i = lane; i < L; i += 32) { const float v = ep[w][i] * aux[w][i]; if (v > bv) { bv = v; bi = i; } }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o); const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  if (lane == 0) {
    if (si) si[b] = start;
    if (ei) ei[b] = bi;
    if (fracs) {
      const float n = vmask ? nvalid : (float)L;
      fracs[b * 2 + 0] = (float)start / n;
      fracs[b * 2 + 1] = (float)bi / n;
    }
  }
}
cudaError_t launch_span_decode(const float* s, const float* e, const float* vmask, int B, int L, int64_t* si,
                               int64_t* ei, float* fracs, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  span_decode_kernel<<<(B + 3) / 4, 128, 0, st>>>(s, e, vmask, B, L, si, ei, fracs);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// IoU counters (utils/utils.py:161-185, models/loss.py:83-109): temporal IoU of [s,e] fractions against
// ground truth, accumulated as {n, sum, #>=0.3, #>=0.5, #>=0.7} in fp64 so shards add exactly.
// ------------------------------------------------------------------------------------------------
__global__ void iou_counters_kernel(const float* __restrict__ fracs, const float* __restrict__ gt, int B,
                                    double* __restrict__ counters) {
  double c[5] = {0, 0, 0, 0, 0};
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    const float g0 = gt[b * 2], g1 = gt[b * 2 + 1], p0 = fracs[b * 2], p1 = fracs[b * 2 + 1];
    const float u0 = fminf(g0, p0), u1 = fmaxf(g1, p1), i0 = fmaxf(g0, p0), i1 = fminf(g1, p1);
    double iou = 0.0;
    if ((u1 - u0) != 0.0f) iou = (double)(i1 - i0) / (double)(u1 - u0);
    if (iou < 0.0) iou = 0.0;
    c[0] += 1.0; c[1] += iou; c[2] += iou >= 0.3; c[3] += iou >= 0.5; c[4] += iou >= 0.7;
  }
#pragma unroll
  for (int k = 0; k < 5; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c[k] += __shfl_xor_sync(0xffffffffu, c[k], o);
    if ((threadIdx.x & 31) == 0 && c[0] > 0) atomicAdd(counters + k, c[k]);
  }
}
cudaError_t launch_iou_counters(const float* fracs, const float* gt, int B, double* counters, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  int blocks = (B + 255) / 256;
  if (blocks > 148) blocks = 148;
  iou_counters_kernel<<<blocks, 256, 0, st>>>(fracs, gt, B, counters);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Device half of the ragged host->device feature copy (seqpan_h2d_ragged): BaseCollate zero-pads every
// clip to vlen rows (utils/BaseDataset.py:209); only the valid prefix of each sample crosses PCIe and the
// padding rows [valid[b], L) are written as zeros here.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) zero_tail_rows_kernel(float4* __restrict__ dst, const int32_t* __restrict__ valid,
                                                             int L, int row_vec4) {
  const int b = blockIdx.x;
  const int n = valid[b];
  const long long cnt = (long long)(L - n) * row_vec4;
  float4* p = dst + ((long long)b * L + n) * row_vec4;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long i = (long long)blockIdx.y * blockDim.x + threadIdx.x; i < cnt; i += (long long)gridDim.y * blockDim.x) p[i] = z;
}
// Zero-copy variant: the kernel itself reads the valid rows straight out of PINNED (UVA-mapped) host memory with
// coalesced 16-byte loads, 8 independent loads in flight per thread, and writes the padding rows as zeros: one launch
// per batch instead of one DMA descriptor per sample.  Work item = one 16-byte vector; a warp reads 512 contiguous bytes.
__global__ void __launch_bounds__(1024) h2d_ragged_kernel(float4* __restrict__ dst, const float4* __restrict__ src_host,
                                                         const int32_t* __restrict__ valid, int B, int L, int row_vec4) {
  const long long per_sample = (long long)L * row_vec4;
  const long long total = (long long)B * per_sample;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < total; i0 += stride * 8) {
    float4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const long long i = i0 + u * stride;
      v[u] = z;
      if (i < total) {
        const int b = (int)(i / per_sample);
        const long long r = (i - (long long)b * per_sample) / row_vec4;
        if (r < valid[b]) v[u] = __ldcs(src_host + i);
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const long long i = i0 + u * stride;
      if (i < total) dst[i] = v[u];
    }
  }
}
cudaError_t launch_h2d_ragged(float* dst, const float* src_host, const int32_t* valid_dev, int B, int L, int row_floats,
                              int ctas, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  const int threads = sq_env().h2d_threads;
  h2d_ragged_kernel<<<ctas, threads, 0, st>>>(reinterpret_cast<float4*>(dst), reinterpret_cast<const float4*>(src_host), valid_dev,
                                          B, L, row_floats / 4);
  return cudaGetLastError();
}

cudaError_t launch_zero_tail_rows(float* dst, const int32_t* valid_dev, int B, int L, int row_floats, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  zero_tail_rows_kernel<<<dim3(B, 4), 256, 0, st>>>(reinterpret_cast<float4*>(dst), valid_dev, L, row_floats / 4);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Clip resampling + padding + mask on the device (seqpan_collate_clips): the feature half of
// sample_vfeat_linear / interpolate_avrage (utils/data_utils.py:161-199), pad_video_seq (:70-84) and
// convert_length_to_mask for a whole batch of ragged clips that are already resident in HBM.
// One CTA per output row (sample b, position i): output row i of a resampled clip is the mean of the raw rows
// [idx(i), idx(i+1)) with idx(i) = round_half_even(fp32(i / size) * (n - 1)), idx(size) = n, or the single row
// idx(i) when that range is empty; every raw row is read once, 16 bytes per thread, 4 rows in flight.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int resample_idx(int i, int size, int n) {
  if (i >= size) return n;
  return (int)rintf(__fmul_rn(__fdiv_rn((float)i, (float)size), (float)(n - 1)));
}

template <typename VT>
__device__ __forceinline__ VT rs_zero();
template <> __device__ __forceinline__ float rs_zero<float>() { return 0.f; }
template <> __device__ __forceinline__ float4 rs_zero<float4>() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ void rs_add(float& a, float v) { a += v; }
__device__ __forceinline__ void rs_add(float4& a, const float4 v) { a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w; }
__device__ __forceinline__ void rs_div(float& a, float d) { a = __fdiv_rn(a, d); }
__device__ __forceinline__ void rs_div(float4& a, float d) {
  a.x = __fdiv_rn(a.x, d); a.y = __fdiv_rn(a.y, d); a.z = __fdiv_rn(a.z, d); a.w = __fdiv_rn(a.w, d);
}

template <typename VT>
__global__ void __launch_bounds__(256) collate_clips_kernel(const VT* __restrict__ raw, const int64_t* __restrict__ offs,
                                                            int vlen, int row_vec, int mode, VT* __restrict__ out,
                                                            float* __restrict__ vmask, int64_t* __restrict__ vlens) {
  const int i = blockIdx.x, b = blockIdx.y;
  const long long o0 = offs[b];
  const int n = (int)(offs[b + 1] - o0);
  const bool resample = mode == 2 || (mode == 1 && n > vlen);
  const int nout = resample ? vlen : min(n, vlen);
  if (threadIdx.x == 0) {
    if (vmask) vmask[(long long)b * vlen + i] = i < nout ? 1.f : 0.f;
    if (vlens && i == 0) vlens[b] = nout;
  }
  VT* dst = out + ((long long)b * vlen + i) * row_vec;
  if (i >= nout) {
    for (int c = threadIdx.x; c < row_vec; c += 256) dst[c] = rs_zero<VT>();
    return;
  }
  int s = i, e = i;
  if (resample) { s = resample_idx(i, vlen, n); e = resample_idx(i + 1, vlen, n); }
  const VT* src = raw + (o0 + s) * row_vec;
  if (s >= e) {
    for (int c = threadIdx.x; c < row_vec; c += 256) dst[c] = __ldcs(src + c);
    return;
  }
  const int cnt = e - s;
  for (int c = threadIdx.x; c < row_vec; c += 256) {
    VT acc = rs_zero<VT>();
    int r = 0;
    for (; r + 4 <= cnt; r += 4) {   // four independent loads in flight, summed in row order like the reference
      const VT v0 = __ldcs(src + (long long)r * row_vec + c), v1 = __ldcs(src + (long long)(r + 1) * row_vec + c);
      const VT v2 = __ldcs(src + (long long)(r + 2) * row_vec + c), v3 = __ldcs(src + (long long)(r + 3) * row_vec + c);
      rs_add(acc, v0); rs_add(acc, v1); rs_add(acc, v2); rs_add(acc, v3);
    }
    for (; r < cnt; ++r) rs_add(acc, __ldcs(src + (long long)r * row_vec + c));
    rs_div(acc, (float)cnt);
    dst[c] = acc;
  }
}

// Text half of BaseCollate (utils/BaseDataset.py:201-207): pad_seq (utils/data_utils.py:42-52) on the word ids and pad_char_seq
// (:55-68) on the character ids of a batch whose ragged id lists are resident in HBM, plus tmask = (word_ids != 0).  One thread per
// output element of char_ids [B,T,C]; the threads with c == 0 also write word_ids / tmask [B,T].
__global__ void __launch_bounds__(256) collate_text_kernel(const int64_t* __restrict__ words, const int64_t* __restrict__ woff,
                                                           const int64_t* __restrict__ chars, const int64_t* __restrict__ coff,
                                                           int B, int T, int C, int64_t* __restrict__ word_ids,
                                                           int64_t* __restrict__ char_ids, float* __restrict__ tmask) {
  const long long total = (long long)B * T * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const long long bt = i / C;
    const int t = (int)(bt % T), b = (int)(bt / T);
    const int64_t w0 = woff[b], nw = woff[b + 1] - w0;
    int64_t ch = 0, wid = 0;
    if (t < nw) {
      const int64_t w = w0 + t;
      wid = words[w];
      const int64_t c0 = coff[w], nc = coff[w + 1] - c0;
      if (c < nc) ch = chars[c0 + c];
    }
    char_ids[i] = ch;
    if (c == 0) {
      word_ids[bt] = wid;
      tmask[bt] = wid != 0 ? 1.0f : 0.0f;
    }
  }
}

cudaError_t launch_collate_text(const int64_t* words, const int64_t* woff, const int64_t* chars, const int64_t* coff, int B, int T, int C,
                                int64_t* word_ids, int64_t* char_ids, float* tmask, cudaStream_t st) {
  const long long total = (long long)B * T * C;
  if (total <= 0) return cudaSuccess;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  collate_text_kernel<<<(unsigned)blocks, 256, 0, st>>>(words, woff, chars, coff, B, T, C, word_ids, char_ids, tmask);
  return cudaGetLastError();
}

cudaError_t launch_collate_clips(const float* raw, const int64_t* offs_dev, int B, int vlen, int row_floats, int mode,
                                 float* out, float* vmask, int64_t* vlens, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  const bool vec = (row_floats & 3) == 0 && ((reinterpret_cast<uintptr_t>(raw) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  for (int b0 = 0; b0 < B; b0 += 65535) {   // gridDim.y limit
    const int nb = B - b0 < 65535 ? B - b0 : 65535;
    const dim3 grid(vlen, nb);
    float* o = out + (size_t)b0 * vlen * row_floats;
    float* m = vmask ? vmask + (size_t)b0 * vlen : nullptr;
    int64_t* l = vlens ? vlens + b0 : nullptr;
    if (vec)
      collate_clips_kernel<float4><<<grid, 256, 0, st>>>(reinterpret_cast<const float4*>(raw), offs_dev + b0, vlen, row_floats / 4,
                                                         mode, reinterpret_cast<float4*>(o), m, l);
    else
      collate_clips_kernel<float><<<grid, 256, 0, st>>>(raw, offs_dev + b0, vlen, row_floats, mode, o, m, l);
  }
  return cudaGetLastError();
}

}  // namespace sq
