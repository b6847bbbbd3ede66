// Shared device helpers for the SeqPAN sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/seqpan_b200.h"

#define SQ_D 128          // model width (configs.model.dim)
#define SQ_H 4            // heads
#define SQ_HD 32          // head dim
#define SQ_MASK (-1e30f)  // models/layers.py:9 mask_value

// ---- host-side process state shared by the launchers -------------------------------------------------------------------
// SEQPAN_* run-time switches (DESIGN.md section 5).  The environment is read ONCE per seqpan_create (not on the forward
// path): sq_env() is the snapshot the launchers consult, sq_env_refresh() re-reads it.
struct SqEnv {
  bool no_joint_attn = false, no_graph = false, force_graph = false, no_side_stream = false;
  int h2d_threads = 128;
};
const SqEnv& sq_env();
void sq_env_refresh();

// Opt-in to > 48 KB of dynamic shared memory.  The attribute belongs to the (function, device) pair, so a process that
// touches a second GPU must set it there too: one bit per device ordinal, set on first use from that device.
struct SqSmemOptIn {
  unsigned long long done = 0;   // benign race: two threads may both set the attribute, which is idempotent
  cudaError_t ensure(const void* fn, size_t bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const unsigned long long bit = dev < 64 ? (1ull << dev) : 0ull;
    if (bit && (__atomic_load_n(&done, __ATOMIC_ACQUIRE) & bit)) return cudaSuccess;
    e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess && bit) __atomic_fetch_or(&done, bit, __ATOMIC_RELEASE);
    return e;
  }
};

namespace sq {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float dot4(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }

// LayerNorm statistics of one 128-wide row held as one float4 per lane (biased variance, two pass).
__device__ __forceinline__ void row_stats(float4 v, float eps, float& mean, float& rstd) {
  mean = warp_sum(v.x + v.y + v.z + v.w) * (1.0f / SQ_D);
  float dx = v.x - mean, dy = v.y - mean, dz = v.z - mean, dw = v.w - mean;
  float var = warp_sum(dx * dx + dy * dy + dz * dz + dw * dw) * (1.0f / SQ_D);
  rstd = 1.0f / sqrtf(var + eps);
}
__device__ __forceinline__ float4 ln_apply(float4 v, float mean, float rstd, float4 g, float4 b) {
  return make_float4((v.x - mean) * rstd * g.x + b.x, (v.y - mean) * rstd * g.y + b.y,
                     (v.z - mean) * rstd * g.z + b.z, (v.w - mean) * rstd * g.w + b.w);
}

}  // namespace sq
