// Training primitives (SURVEY.md section 8 rows a19 / f4: the training step of models/SeqPAN.py:171-182 + main.py:93-97).
// The backward of SeqPAN is assembled on the host (vmrframe_b200/train.py: a reverse-mode tape over these kernels, one
// vector-Jacobian rule per primitive); all arithmetic runs here, in fp32, on the GPU.  First correct version: generic
// strided kernels (a 64x64 SGEMM tile, a 4-D broadcasting element-wise kernel, strided softmax / LayerNorm / depthwise
// conv rules, row gather / scatter-add, max-pool with indices, fused AdamW and a squared-norm reduction for
// clip_grad_norm_).  The tcgen05 forward kernels are not reused here yet (they keep no activations).
#include <cstdio>

#include "common.cuh"
#include "train_ops.cuh"

namespace {

// ---- strided batched SGEMM: C[b0,b1] = alpha * A.B + beta * C, every operand addressed by (row stride, column stride) ----
constexpr int GT = 64, GK = 16;

// PARTIAL (deterministic split-K): each K-split stores its raw tile to part[ks][M][N]; a template parameter, so that the default
// instantiation is the kernel it was before (its register count, and so its occupancy, is unchanged)
template <bool PARTIAL>
__global__ void __launch_bounds__(256) t_gemm_kernel(const float* __restrict__ A, const float* __restrict__ B, float* __restrict__ C,
                                                     const float* __restrict__ bias, SeqpanGemm g, float* __restrict__ part) {
  __shared__ __align__(16) float As[GK][GT + 4];
  __shared__ __align__(16) float Bs[GK][GT + 4];
  const int split = g.splitk > 1 ? g.splitk : 1;
  const int z = blockIdx.z;
  const int ks = z % split, bz = z / split;
  const int b1 = bz % g.batch1, b0 = bz / g.batch1;
  A += b0 * g.a_b0 + b1 * g.a_b1;
  B += b0 * g.b_b0 + b1 * g.b_b1;
  C += b0 * g.c_b0 + b1 * g.c_b1;
  const long long m0 = (long long)blockIdx.y * GT, n0 = (long long)blockIdx.x * GT;
  const long long kchunk = ((g.K + split - 1) / split + GK - 1) / GK * GK;
  const long long kbeg = ks * kchunk, kend = min((long long)g.K, kbeg + kchunk);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4] = {};
  for (long long k0 = kbeg; k0 < kend; k0 += GK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = threadIdx.x + i * 256;          // 0..1023
      // A tile: element (m = e % 64, k = e / 64) when A is row-strided small (a_cs == 1 -> k fastest is better); pick the
      // mapping that walks the unit-stride dimension with consecutive threads
      int am, ak;
      if (g.a_cs == 1) { ak = e & 15; am = e >> 4; } else { am = e & 63; ak = e >> 6; }
      const long long gm = m0 + am, gk = k0 + ak;
      As[ak][am] = (gm < g.M && gk < kend) ? __ldg(A + gm * g.a_rs + gk * g.a_cs) : 0.f;
      int bn, bk;
      if (g.b_rs == 1) { bk = e & 15; bn = e >> 4; } else { bn = e & 63; bk = e >> 6; }
      const long long gn = n0 + bn, gk2 = k0 + bk;
      Bs[bk][bn] = (gn < g.N && gk2 < kend) ? __ldg(B + gk2 * g.b_rs + gn * g.b_cs) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < GK; ++k) {
      // one 16-byte shared-memory read per operand and k (rows of As / Bs are 272 bytes apart: 16-byte aligned)
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a[4] = {av.x, av.y, av.z, av.w}, b[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long gm = m0 + ty * 4 + i, gn = n0 + tx * 4 + j;
      if (gm >= g.M || gn >= g.N) continue;
      if (PARTIAL) { part[(ks * g.M + gm) * g.N + gn] = acc[i][j]; continue; }
      float* c = C + gm * g.c_rs + gn * g.c_cs;
      const float v = g.alpha * acc[i][j] + ((bias && ks == 0) ? __ldg(bias + gn) : 0.f);     // bias[n]: added once (by K-split 0)
      if (split > 1) atomicAdd(c, v);                                           // C was pre-scaled by beta (0: zeroed) by the launcher
      else *c = v + (g.beta != 0.f ? g.beta * *c : 0.f);
    }
}

// ---- deterministic split-K: C = alpha * (((p0 + p1) + p2) + ...) + bias + beta * C, one thread per element ----
__global__ void __launch_bounds__(256) t_splitk_reduce_kernel(float* __restrict__ C, const float* __restrict__ part,
                                                              const float* __restrict__ bias, SeqpanGemm g, int split) {
  const long long mn = g.M * g.N;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < mn; i += (long long)gridDim.x * blockDim.x) {
    const long long m = i / g.N, n = i % g.N;
    float s = part[i];
    for (int k = 1; k < split; ++k) s += part[k * mn + i];
    float* c = C + m * g.c_rs + n;                                   // split-K: c_cs == 1
    const float v = g.alpha * s + (bias ? __ldg(bias + n) : 0.f);
    *c = g.beta != 0.f ? v + g.beta * *c : v;
  }
}

// ---- out[i] += part[0][i] + part[1][i] + ... in ascending partial order, one thread per element; elements i >= split_at
// go to out1[i - split_at] (LayerNorm: dgamma | dbeta) ----
__global__ void __launch_bounds__(256) t_ordered_sum_kernel(float* __restrict__ out0, float* __restrict__ out1, int split_at,
                                                            const float* __restrict__ part, int parts, int width) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= width) return;
  float s = part[i];
  for (int p = 1; p < parts; ++p) s += part[(long long)p * width + i];
  float* o = i < split_at ? out0 + i : out1 + (i - split_at);
  *o += s;
}

// ---- 4-D broadcasting element-wise kernel ----
__device__ __forceinline__ float ew_apply(int op, float a, float b, float c, float alpha, float beta) {
  switch (op) {
    case SEQPAN_EW_COPY: return a;
    case SEQPAN_EW_AXPBY: return alpha * a + beta * b;
    case SEQPAN_EW_MUL: return alpha * a * b;
    case SEQPAN_EW_RELU: return fmaxf(a, 0.f);
    case SEQPAN_EW_RELU_BWD: return b > 0.f ? a : 0.f;
    case SEQPAN_EW_SIGMOID: return 1.0f / (1.0f + expf(-a));
    case SEQPAN_EW_SIGMOID_BWD: return a * b * (1.0f - b);
    case SEQPAN_EW_MASK_LOGITS: return a + (1.0f - b) * SQ_MASK;
    case SEQPAN_EW_FMA: return a * b + c;
    case SEQPAN_EW_LOG: return logf(a);
    case SEQPAN_EW_EXP: return expf(a);
    case SEQPAN_EW_DIV: return a / b;
    case SEQPAN_EW_SQRT: return sqrtf(a);
    case SEQPAN_EW_AFFINE: return alpha * a + beta;
    case SEQPAN_EW_EQ: return a == alpha ? 1.0f : 0.f;
    case SEQPAN_EW_DIV_SAFE: return b != 0.f ? a / b : 0.f;
    case SEQPAN_EW_DROPOUT: return b >= alpha ? a * beta : 0.f;
    default: return 0.f;
  }
}

__global__ void __launch_bounds__(256) t_ewise_kernel(float* __restrict__ out, const float* __restrict__ a, const float* __restrict__ b,
                                                      const float* __restrict__ c, SeqpanEwise e, long long total) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long r = i;
    const long long i3 = r % e.shape[3]; r /= e.shape[3];
    const long long i2 = r % e.shape[2]; r /= e.shape[2];
    const long long i1 = r % e.shape[1]; r /= e.shape[1];
    const long long i0 = r;
    const float va = a ? a[i0 * e.sa[0] + i1 * e.sa[1] + i2 * e.sa[2] + i3 * e.sa[3]] : 0.f;
    const float vb = b ? b[i0 * e.sb[0] + i1 * e.sb[1] + i2 * e.sb[2] + i3 * e.sb[3]] : 0.f;
    const float vc = c ? c[i0 * e.sc[0] + i1 * e.sc[1] + i2 * e.sc[2] + i3 * e.sc[3]] : 0.f;
    float* o = out + i0 * e.so[0] + i1 * e.so[1] + i2 * e.so[2] + i3 * e.so[3];
    const float v = ew_apply(e.op, va, vb, vc, e.alpha, e.beta);
    *o = e.accumulate ? *o + v : v;
  }
}

// ---- strided softmax over `cols` (one warp per row; row = (r0, r1)) and its vector-Jacobian product ----
__global__ void __launch_bounds__(256) t_softmax_kernel(float* __restrict__ y, const float* __restrict__ x, SeqpanSoftmax s) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= (long long)s.rows0 * s.rows1) return;
  const int lane = threadIdx.x & 31;
  const long long base = (row / s.rows1) * s.r0_stride + (row % s.rows1) * s.r1_stride;
  float mx = -INFINITY;
  for (int c = lane; c < s.cols; c += 32) mx = fmaxf(mx, x[base + c * s.c_stride]);
  mx = sq::warp_max(mx);
  float sum = 0.f;
  for (int c = lane; c < s.cols; c += 32) sum += expf(x[base + c * s.c_stride] - mx);
  sum = sq::warp_sum(sum);
  const float inv = 1.0f / sum;
  for (int c = lane; c < s.cols; c += 32) y[base + c * s.c_stride] = expf(x[base + c * s.c_stride] - mx) * inv;
}
// dx = y * (dy - sum(y * dy))
__global__ void __launch_bounds__(256) t_softmax_bwd_kernel(float* __restrict__ dx, const float* __restrict__ y, const float* __restrict__ dy,
                                                            SeqpanSoftmax s) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= (long long)s.rows0 * s.rows1) return;
  const int lane = threadIdx.x & 31;
  const long long base = (row / s.rows1) * s.r0_stride + (row % s.rows1) * s.r1_stride;
  float dot = 0.f;
  for (int c = lane; c < s.cols; c += 32) dot = fmaf(y[base + c * s.c_stride], dy[base + c * s.c_stride], dot);
  dot = sq::warp_sum(dot);
  for (int c = lane; c < s.cols; c += 32) {
    const long long i = base + c * s.c_stride;
    dx[i] = y[i] * (dy[i] - dot);
  }
}

// ---- LayerNorm backward over 128-wide rows: dx, and dgamma / dbeta accumulated with atomics (or written as per-CTA partials) ----
__global__ void __launch_bounds__(256) t_layernorm_bwd_kernel(float* __restrict__ dx, float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                              const float* __restrict__ x, const float* __restrict__ dy,
                                                              const float* __restrict__ gamma, float eps, long long M,
                                                              float* __restrict__ part) {
  __shared__ float sg[8][128], sb[8][128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float4 g = sq::ldg4(gamma + lane * 4);
  float4 ag = make_float4(0.f, 0.f, 0.f, 0.f), ab = ag;
  for (long long row = (long long)blockIdx.x * 8 + warp; row < M; row += (long long)gridDim.x * 8) {
    const float4 v = sq::ld4(x + row * 128 + lane * 4), d = sq::ld4(dy + row * 128 + lane * 4);
    float mean, rstd;
    sq::row_stats(v, eps, mean, rstd);
    const float4 xh = make_float4((v.x - mean) * rstd, (v.y - mean) * rstd, (v.z - mean) * rstd, (v.w - mean) * rstd);
    const float4 dg = make_float4(d.x * g.x, d.y * g.y, d.z * g.z, d.w * g.w);        // dL/dxhat
    const float s1 = sq::warp_sum(dg.x + dg.y + dg.z + dg.w) * (1.0f / 128.0f);
    const float s2 = sq::warp_sum(dg.x * xh.x + dg.y * xh.y + dg.z * xh.z + dg.w * xh.w) * (1.0f / 128.0f);
    sq::st4(dx + row * 128 + lane * 4, make_float4(rstd * (dg.x - s1 - xh.x * s2), rstd * (dg.y - s1 - xh.y * s2),
                                                   rstd * (dg.z - s1 - xh.z * s2), rstd * (dg.w - s1 - xh.w * s2)));
    ag.x += d.x * xh.x; ag.y += d.y * xh.y; ag.z += d.z * xh.z; ag.w += d.w * xh.w;
    ab.x += d.x; ab.y += d.y; ab.z += d.z; ab.w += d.w;
  }
  sq::st4(&sg[warp][lane * 4], ag);
  sq::st4(&sb[warp][lane * 4], ab);
  __syncthreads();
  if (threadIdx.x < 128) {
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) { a += sg[w][threadIdx.x]; b += sb[w][threadIdx.x]; }
    if (part) {                                   // deterministic: this CTA's [dgamma | dbeta] partial row
      part[blockIdx.x * 256 + threadIdx.x] = a;
      part[blockIdx.x * 256 + 128 + threadIdx.x] = b;
    } else {
      atomicAdd(dgamma + threadIdx.x, a);
      atomicAdd(dbeta + threadIdx.x, b);
    }
  }
}

// ---- depthwise conv k=7 along the rows of equal-length segments; flip = 1 gives the input gradient ----
__global__ void __launch_bounds__(128) t_dwconv_kernel(float* __restrict__ y, const float* __restrict__ x, const float* __restrict__ w,
                                                       long long rows, int len, int flip) {
  const long long r = blockIdx.x;
  const int c = threadIdx.x, l = (int)(r % len);
  float acc = 0.f;
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    const int d = j - 3;
    if (l + d < 0 || l + d >= len) continue;
    acc = fmaf(__ldg(w + c * 7 + (flip ? 6 - j : j)), x[(r + d) * 128 + c], acc);
  }
  y[r * 128 + c] = acc;
}
// dw[c, j] += sum over rows of dy[r, c] * x[r + j - 3, c] (inside the row's segment)
__global__ void __launch_bounds__(128) t_dwconv_bwd_w_kernel(float* __restrict__ dw, const float* __restrict__ x, const float* __restrict__ dy,
                                                             long long rows, int len, float* __restrict__ part) {
  const int c = threadIdx.x;
  float acc[7] = {};
  for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
    const int l = (int)(r % len);
    const float g = dy[r * 128 + c];
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      const int d = j - 3;
      if (l + d >= 0 && l + d < len) acc[j] = fmaf(g, x[(r + d) * 128 + c], acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    if (part) part[blockIdx.x * (128 * 7) + c * 7 + j] = acc[j];   // deterministic: this CTA's [128 x 7] partial
    else atomicAdd(dw + c * 7 + j, acc[j]);
  }
}

// ---- row gather / scatter-add (embeddings) ----
__global__ void __launch_bounds__(128) t_gather_rows_kernel(float* __restrict__ out, const float* __restrict__ table, const int64_t* __restrict__ ids,
                                                            int dim, long long nrows_table) {
  const long long n = blockIdx.x;
  long long id = ids[n];
  id = id < 0 ? 0 : (id >= nrows_table ? nrows_table - 1 : id);
  for (int d = threadIdx.x; d < dim; d += blockDim.x) out[n * dim + d] = table[id * dim + d];
}
__global__ void __launch_bounds__(128) t_scatter_add_rows_kernel(float* __restrict__ dtable, const float* __restrict__ dout,
                                                                 const int64_t* __restrict__ ids, int dim, long long nrows_table) {
  const long long n = blockIdx.x;
  long long id = ids[n];
  id = id < 0 ? 0 : (id >= nrows_table ? nrows_table - 1 : id);
  for (int d = threadIdx.x; d < dim; d += blockDim.x) atomicAdd(dtable + id * dim + d, dout[n * dim + d]);
}

// Deterministic adjoint: CTAs own table rows (grid-stride over rows); a CTA scans all ids 128 at a time and adds the matching
// dout rows in ascending n into registers, then adds the sum once into dtable.  Columns: thread t owns t, t + 128, ...
constexpr int SC_COLS = 4;   // columns per thread per pass: dim <= 512 in one scan of the ids
__global__ void __launch_bounds__(128) t_scatter_add_rows_det_kernel(float* __restrict__ dtable, const float* __restrict__ dout,
                                                                     const int64_t* __restrict__ ids, long long n, int dim,
                                                                     long long nrows_table) {
  __shared__ unsigned hits[4];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (long long row = blockIdx.x; row < nrows_table; row += gridDim.x) {
    for (int d0 = 0; d0 < dim; d0 += 128 * SC_COLS) {
      float acc[SC_COLS] = {};
      bool any = false;
      for (long long n0 = 0; n0 < n; n0 += 128) {
        const long long nn = n0 + threadIdx.x;
        bool hit = false;
        if (nn < n) {
          long long id = __ldg(ids + nn);
          id = id < 0 ? 0 : (id >= nrows_table ? nrows_table - 1 : id);
          hit = id == row;
        }
        const unsigned b = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) hits[warp] = b;
        __syncthreads();
        for (int w = 0; w < 4; ++w) {
          for (unsigned m = hits[w]; m; m &= m - 1) {
            const float* src = dout + (n0 + w * 32 + __ffs(m) - 1) * dim;
            any = true;
#pragma unroll
            for (int k = 0; k < SC_COLS; ++k) {
              const int d = d0 + k * 128 + threadIdx.x;
              if (d < dim) acc[k] += src[d];
            }
          }
        }
        __syncthreads();
      }
      if (!any) continue;                       // no id hits this row: dtable's row is left untouched
#pragma unroll
      for (int k = 0; k < SC_COLS; ++k) {
        const int d = d0 + k * 128 + threadIdx.x;
        if (d < dim) dtable[row * dim + d] += acc[k];
      }
    }
  }
}

// ---- max over the middle dim of [N, P, C] with indices (torch.max(dim): first maximum wins), and its scatter ----
__global__ void __launch_bounds__(128) t_maxpool_kernel(float* __restrict__ out, int32_t* __restrict__ idx, const float* __restrict__ x, int P, int C) {
  const long long n = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float best = x[(n * P) * C + c];
    int bi = 0;
    for (int p = 1; p < P; ++p) {
      const float v = x[(n * P + p) * C + c];
      if (v > best) { best = v; bi = p; }
    }
    out[n * C + c] = best;
    idx[n * C + c] = bi;
  }
}
__global__ void __launch_bounds__(128) t_maxpool_bwd_kernel(float* __restrict__ dx, const float* __restrict__ dout, const int32_t* __restrict__ idx,
                                                            int P, int C) {
  const long long n = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) dx[(n * P + idx[n * C + c]) * C + c] = dout[n * C + c];   // dx pre-zeroed
}

// ---- optimizer: sum of squares (clip_grad_norm_) and fused AdamW (torch.optim.AdamW semantics, utils/utils.py:87-97) ----
__global__ void __launch_bounds__(256) t_sumsq_kernel(const float* __restrict__ x, long long n, double* __restrict__ out,
                                                      double* __restrict__ part) {
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) acc = fmaf(x[i], x[i], acc);
  acc = sq::warp_sum(acc);
  __shared__ float red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < 8; ++i) s += red[i];
    if (part) part[blockIdx.x] = s;               // deterministic: this CTA's partial
    else atomicAdd(out, s);
  }
}
__global__ void t_sumsq_reduce_kernel(double* __restrict__ out, const double* __restrict__ part, int parts) {
  double s = 0.0;
  for (int p = 0; p < parts; ++p) s += part[p];
  *out += s;
}
__global__ void __launch_bounds__(256) t_adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                      float* __restrict__ v, long long n, SeqpanAdamW a, const double* __restrict__ sumsq,
                                                      const float* __restrict__ dyn) {
  if (dyn) { a.lr = dyn[0]; a.bias1 = dyn[1]; a.bias2_sqrt = dyn[2]; }   // per-step scalars of a step replayed as a CUDA graph
  // clip coefficient of clip_grad_norm_(max_norm): min(1, max_norm / (norm + 1e-6)), computed from the device-side sum of squares
  float clip = 1.0f;
  if (sumsq && a.max_grad_norm > 0.f) {
    const float norm = (float)sqrt(*sumsq);
    clip = fminf(1.0f, a.max_grad_norm / (norm + 1e-6f));
  }
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * clip;
    float pi = p[i];
    pi *= 1.0f - a.lr * a.weight_decay;                    // decoupled weight decay
    const float mi = a.beta1 * m[i] + (1.0f - a.beta1) * gi;
    const float vi = a.beta2 * v[i] + (1.0f - a.beta2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / a.bias2_sqrt + a.eps;  // sqrt(v) / sqrt(1 - beta2^t) + eps
    p[i] = pi - (a.lr / a.bias1) * (mi / denom);
  }
}

thread_local char g_terr[256] = "";
unsigned grid_for(long long n, int per_block, long long cap = 148 * 16) {
  long long b = (n + per_block - 1) / per_block;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}
// grids of the reductions: functions of the shape only (the deterministic entry points size their scratch from them)
unsigned ln_bwd_grid(long long M) { return grid_for(M, 8, 148 * 4); }
unsigned dwconv_bwd_w_grid(long long rows) { return grid_for(rows, 64, 148 * 8); }
unsigned sumsq_grid(long long n) { return grid_for(n, 1024, 148 * 4); }

}  // namespace

int tfail(const char* msg) { snprintf(g_terr, sizeof(g_terr), "%s", msg); return SEQPAN_E_INVALID; }
int tcheck() {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { snprintf(g_terr, sizeof(g_terr), "%s", cudaGetErrorString(e)); return SEQPAN_E_CUDA; }
  return SEQPAN_OK;
}

int t_gemm_prepare(const float* A, const float* B, float* C, const SeqpanGemm* gp, cudaStream_t st, int& split, long long& gz,
                   bool zero_c) {
  gz = 0;
  if (!A || !B || !C || !gp) return tfail("gemm: NULL argument");
  const SeqpanGemm& g = *gp;
  if (g.M < 0 || g.N < 0 || g.K < 0 || g.batch0 < 1 || g.batch1 < 1) return tfail("gemm: bad sizes");
  if (g.M == 0 || g.N == 0) return SEQPAN_OK;
  split = g.splitk > 1 ? g.splitk : 1;
  if (split > 1) {
    if (g.beta != 0.f && g.beta != 1.f) return tfail("gemm: split-K needs beta 0 or 1");
    if (g.batch0 * g.batch1 != 1 || g.c_cs != 1) return tfail("gemm: split-K needs one batch and a row-major C");
    if (g.beta == 0.f && zero_c) {
      if (cudaMemset2DAsync(C, (size_t)g.c_rs * sizeof(float), 0, (size_t)g.N * sizeof(float), (size_t)g.M, st) != cudaSuccess) return tcheck();
    }
  }
  const long long z = (long long)g.batch0 * g.batch1 * split;
  if (z > 65535) return tfail("gemm: too many batches");
  gz = z;
  return SEQPAN_OK;
}

size_t t_gemm_det_scratch(const SeqpanGemm& g) {
  return g.splitk > 1 && g.M > 0 && g.N > 0 ? (size_t)g.splitk * g.M * g.N * sizeof(float) : 0;
}
int t_gemm_det_check(const SeqpanGemm& g, const void* scratch, size_t scratch_bytes) {
  if (!scratch || scratch_bytes < t_gemm_det_scratch(g)) {
    snprintf(g_terr, sizeof(g_terr), "gemm: split-K scratch needs %zu bytes", t_gemm_det_scratch(g));
    return SEQPAN_E_WORKSPACE;
  }
  return SEQPAN_OK;
}
int t_gemm_splitk_reduce(float* C, const float* part, const float* bias, const SeqpanGemm& g, int split, cudaStream_t st) {
  t_splitk_reduce_kernel<<<grid_for(g.M * g.N, 256), 256, 0, st>>>(C, part, bias, g, split);
  return tcheck();
}

extern "C" const char* seqpan_t_last_error(void) { return g_terr; }

extern "C" int seqpan_t_gemm(const float* A, const float* B, float* C, const float* bias, const SeqpanGemm* gp, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  int split = 1;
  long long gz = 0;
  const int rc = t_gemm_prepare(A, B, C, gp, st, split, gz);
  if (rc != SEQPAN_OK || gz == 0) return rc;
  const SeqpanGemm g = *gp;
  dim3 grid((unsigned)((g.N + GT - 1) / GT), (unsigned)((g.M + GT - 1) / GT), (unsigned)gz);
  t_gemm_kernel<false><<<grid, 256, 0, st>>>(A, B, C, bias, g, nullptr);
  return tcheck();
}
extern "C" size_t seqpan_t_gemm_det_scratch_bytes(const SeqpanGemm* g) { return g ? t_gemm_det_scratch(*g) : 0; }
extern "C" int seqpan_t_gemm_det(const float* A, const float* B, float* C, const float* bias, const SeqpanGemm* gp, void* scratch,
                                 size_t scratch_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  int split = 1;
  long long gz = 0;
  int rc = t_gemm_prepare(A, B, C, gp, st, split, gz, false);
  if (rc != SEQPAN_OK || gz == 0) return rc;
  const SeqpanGemm g = *gp;
  dim3 grid((unsigned)((g.N + GT - 1) / GT), (unsigned)((g.M + GT - 1) / GT), (unsigned)gz);
  if (split == 1) {                             // no K-split: every element is already written by one thread
    t_gemm_kernel<false><<<grid, 256, 0, st>>>(A, B, C, bias, g, nullptr);
    return tcheck();
  }
  if ((rc = t_gemm_det_check(g, scratch, scratch_bytes)) != SEQPAN_OK) return rc;
  t_gemm_kernel<true><<<grid, 256, 0, st>>>(A, B, C, nullptr, g, (float*)scratch);
  if ((rc = tcheck()) != SEQPAN_OK) return rc;
  return t_gemm_splitk_reduce(C, (const float*)scratch, bias, g, split, st);
}

extern "C" int seqpan_t_ewise(float* out, const float* a, const float* b, const float* c, const SeqpanEwise* ep, void* stream) {
  if (!out || !ep) return tfail("ewise: NULL argument");
  SeqpanEwise e = *ep;
  long long total = 1;
  for (int i = 0; i < 4; ++i) { if (e.shape[i] < 0) return tfail("ewise: negative shape"); total *= e.shape[i]; }
  if (total == 0) return SEQPAN_OK;
  t_ewise_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(out, a, b, c, e, total);
  return tcheck();
}

extern "C" int seqpan_t_softmax(float* y, const float* x, const SeqpanSoftmax* sp, void* stream) {
  if (!y || !x || !sp || sp->cols < 1) return tfail("softmax: bad argument");
  const long long rows = (long long)sp->rows0 * sp->rows1;
  if (rows <= 0) return SEQPAN_OK;
  t_softmax_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(y, x, *sp);
  return tcheck();
}
extern "C" int seqpan_t_softmax_bwd(float* dx, const float* y, const float* dy, const SeqpanSoftmax* sp, void* stream) {
  if (!dx || !y || !dy || !sp || sp->cols < 1) return tfail("softmax_bwd: bad argument");
  const long long rows = (long long)sp->rows0 * sp->rows1;
  if (rows <= 0) return SEQPAN_OK;
  t_softmax_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(dx, y, dy, *sp);
  return tcheck();
}

extern "C" int seqpan_t_layernorm_bwd(float* dx, float* dgamma, float* dbeta, const float* x, const float* dy, const float* gamma,
                                      float eps, int64_t M, void* stream) {
  if (!dx || !dgamma || !dbeta || !x || !dy || !gamma) return tfail("layernorm_bwd: NULL argument");
  if (M <= 0) return SEQPAN_OK;
  t_layernorm_bwd_kernel<<<ln_bwd_grid(M), 256, 0, (cudaStream_t)stream>>>(dx, dgamma, dbeta, x, dy, gamma, eps, M, nullptr);
  return tcheck();
}
extern "C" size_t seqpan_t_layernorm_bwd_det_scratch_bytes(int64_t M) {
  return M > 0 ? (size_t)ln_bwd_grid(M) * 256 * sizeof(float) : 0;
}
extern "C" int seqpan_t_layernorm_bwd_det(float* dx, float* dgamma, float* dbeta, const float* x, const float* dy, const float* gamma,
                                          float eps, int64_t M, void* scratch, size_t scratch_bytes, void* stream) {
  if (!dx || !dgamma || !dbeta || !x || !dy || !gamma) return tfail("layernorm_bwd: NULL argument");
  if (M <= 0) return SEQPAN_OK;
  if (!scratch || scratch_bytes < seqpan_t_layernorm_bwd_det_scratch_bytes(M)) {
    tfail("layernorm_bwd: scratch too small");
    return SEQPAN_E_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned nb = ln_bwd_grid(M);
  t_layernorm_bwd_kernel<<<nb, 256, 0, st>>>(dx, dgamma, dbeta, x, dy, gamma, eps, M, (float*)scratch);
  t_ordered_sum_kernel<<<1, 256, 0, st>>>(dgamma, dbeta, 128, (const float*)scratch, (int)nb, 256);
  return tcheck();
}

extern "C" int seqpan_t_dwconv(float* y, const float* x, const float* w, int64_t rows, int len, int flip, void* stream) {
  if (!y || !x || !w || len < 1 || rows % len) return tfail("dwconv: bad argument");
  if (rows <= 0) return SEQPAN_OK;
  t_dwconv_kernel<<<(unsigned)rows, 128, 0, (cudaStream_t)stream>>>(y, x, w, rows, len, flip);
  return tcheck();
}
extern "C" int seqpan_t_dwconv_bwd_w(float* dw, const float* x, const float* dy, int64_t rows, int len, void* stream) {
  if (!dw || !x || !dy || len < 1 || rows % len) return tfail("dwconv_bwd_w: bad argument");
  if (rows <= 0) return SEQPAN_OK;
  t_dwconv_bwd_w_kernel<<<dwconv_bwd_w_grid(rows), 128, 0, (cudaStream_t)stream>>>(dw, x, dy, rows, len, nullptr);
  return tcheck();
}
extern "C" size_t seqpan_t_dwconv_bwd_w_det_scratch_bytes(int64_t rows) {
  return rows > 0 ? (size_t)dwconv_bwd_w_grid(rows) * 128 * 7 * sizeof(float) : 0;
}
extern "C" int seqpan_t_dwconv_bwd_w_det(float* dw, const float* x, const float* dy, int64_t rows, int len, void* scratch,
                                         size_t scratch_bytes, void* stream) {
  if (!dw || !x || !dy || len < 1 || rows % len) return tfail("dwconv_bwd_w: bad argument");
  if (rows <= 0) return SEQPAN_OK;
  if (!scratch || scratch_bytes < seqpan_t_dwconv_bwd_w_det_scratch_bytes(rows)) {
    tfail("dwconv_bwd_w: scratch too small");
    return SEQPAN_E_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned nb = dwconv_bwd_w_grid(rows);
  t_dwconv_bwd_w_kernel<<<nb, 128, 0, st>>>(dw, x, dy, rows, len, (float*)scratch);
  t_ordered_sum_kernel<<<(128 * 7 + 255) / 256, 256, 0, st>>>(dw, dw, 128 * 7, (const float*)scratch, (int)nb, 128 * 7);
  return tcheck();
}

extern "C" int seqpan_t_gather_rows(float* out, const float* table, const int64_t* ids, int64_t n, int dim, int64_t table_rows, void* stream) {
  if (!out || !table || !ids || dim < 1 || table_rows < 1) return tfail("gather_rows: bad argument");
  if (n <= 0) return SEQPAN_OK;
  t_gather_rows_kernel<<<(unsigned)n, 128, 0, (cudaStream_t)stream>>>(out, table, ids, dim, table_rows);
  return tcheck();
}
extern "C" int seqpan_t_scatter_add_rows(float* dtable, const float* dout, const int64_t* ids, int64_t n, int dim, int64_t table_rows,
                                         void* stream) {
  if (!dtable || !dout || !ids || dim < 1 || table_rows < 1) return tfail("scatter_add_rows: bad argument");
  if (n <= 0) return SEQPAN_OK;
  t_scatter_add_rows_kernel<<<(unsigned)n, 128, 0, (cudaStream_t)stream>>>(dtable, dout, ids, dim, table_rows);
  return tcheck();
}
extern "C" int seqpan_t_scatter_add_rows_det(float* dtable, const float* dout, const int64_t* ids, int64_t n, int dim,
                                             int64_t table_rows, void* stream) {
  if (!dtable || !dout || !ids || dim < 1 || table_rows < 1) return tfail("scatter_add_rows: bad argument");
  if (n <= 0) return SEQPAN_OK;
  t_scatter_add_rows_det_kernel<<<grid_for(table_rows, 1), 128, 0, (cudaStream_t)stream>>>(dtable, dout, ids, n, dim, table_rows);
  return tcheck();
}

extern "C" int seqpan_t_maxpool(float* out, int32_t* idx, const float* x, int64_t N, int P, int C, void* stream) {
  if (!out || !idx || !x || P < 1 || C < 1) return tfail("maxpool: bad argument");
  if (N <= 0) return SEQPAN_OK;
  t_maxpool_kernel<<<(unsigned)N, 128, 0, (cudaStream_t)stream>>>(out, idx, x, P, C);
  return tcheck();
}
extern "C" int seqpan_t_maxpool_bwd(float* dx, const float* dout, const int32_t* idx, int64_t N, int P, int C, void* stream) {
  if (!dx || !dout || !idx || P < 1 || C < 1) return tfail("maxpool_bwd: bad argument");
  if (N <= 0) return SEQPAN_OK;
  if (cudaMemsetAsync(dx, 0, sizeof(float) * (size_t)N * P * C, (cudaStream_t)stream) != cudaSuccess) return tcheck();
  t_maxpool_bwd_kernel<<<(unsigned)N, 128, 0, (cudaStream_t)stream>>>(dx, dout, idx, P, C);
  return tcheck();
}

extern "C" int seqpan_t_sumsq(const float* x, int64_t n, double* out_accum, void* stream) {
  if (!x || !out_accum) return tfail("sumsq: NULL argument");
  if (n <= 0) return SEQPAN_OK;
  t_sumsq_kernel<<<sumsq_grid(n), 256, 0, (cudaStream_t)stream>>>(x, n, out_accum, nullptr);
  return tcheck();
}
extern "C" size_t seqpan_t_sumsq_det_scratch_bytes(int64_t n) { return n > 0 ? (size_t)sumsq_grid(n) * sizeof(double) : 0; }
extern "C" int seqpan_t_sumsq_det(const float* x, int64_t n, double* out_accum, void* scratch, size_t scratch_bytes, void* stream) {
  if (!x || !out_accum) return tfail("sumsq: NULL argument");
  if (n <= 0) return SEQPAN_OK;
  if (!scratch || scratch_bytes < seqpan_t_sumsq_det_scratch_bytes(n) || ((uintptr_t)scratch & 7)) {
    tfail("sumsq: scratch too small or not 8-byte aligned");
    return SEQPAN_E_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned nb = sumsq_grid(n);
  t_sumsq_kernel<<<nb, 256, 0, st>>>(x, n, out_accum, (double*)scratch);
  t_sumsq_reduce_kernel<<<1, 1, 0, st>>>(out_accum, (const double*)scratch, (int)nb);
  return tcheck();
}
extern "C" int seqpan_t_adamw(float* p, const float* g, float* m, float* v, int64_t n, const SeqpanAdamW* a, const double* sumsq,
                              const float* dyn, void* stream) {
  if (!p || !g || !m || !v || !a) return tfail("adamw: NULL argument");
  if (n <= 0) return SEQPAN_OK;
  t_adamw_kernel<<<grid_for(n, 1024, 148 * 4), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, *a, sumsq, dyn);
  return tcheck();
}
