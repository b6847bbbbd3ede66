// Counter-based Gumbel(0,1) noise of a seeded evaluation sweep (DESIGN.md section 13): gumbel_noise_kernel, and the probe
// kernel tests/test_eval_reproducible.py compiles from this header to read the Philox words and uniforms back.
#pragma once
#include <cuda_runtime.h>
#include <curand_philox4x32_x.h>
#include <stdint.h>

namespace sq {

// Philox4x32-10, key = (seed lo, seed hi), counter = (row, batch_id, 0, 0) with row = b * L + l: the four words are the four
// labels of row (b, l).
__device__ __forceinline__ uint4 gumbel_words(uint64_t seed, uint32_t batch_id, uint32_t row) {
  return curand_Philox4x32_10(make_uint4(row, batch_id, 0u, 0u), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}

// ((x >> 9) + 0.5) * 2^-23: exact in fp32 and strictly inside (0, 1), so both logarithms below are finite.
__device__ __forceinline__ float open_uniform(uint32_t x) { return ((float)(x >> 9) + 0.5f) * 0x1p-23f; }

// IEEE logf (the library is built without fast-math): -log(Exp(1)) with Exp(1) = -log(u).
__device__ __forceinline__ float gumbel_of(uint32_t x) { return -logf(-logf(open_uniform(x))); }

}  // namespace sq
