// Host-side pieces shared by the training GEMM launchers (train_ops.cu: fp32 SIMT, train_tc.cu: bf16 tensor cores).
#pragma once
#include <cuda_runtime.h>

#include "../../include/seqpan_b200.h"

// error path of the seqpan_t_* entry points (read back by seqpan_t_last_error)
int tfail(const char* msg);
int tcheck();

// Argument checks and the split-K pre-pass of seqpan_t_gemm, shared so that both GEMM entry points reject the same inputs
// with the same errors.  On SEQPAN_OK, `gz` = CTAs along grid z (batch0 * batch1 * split), 0 when there is nothing to launch
// (M == 0 or N == 0); with split > 1, beta == 0 and zero_c the C view has been zeroed on `st` (the atomic split-K epilogue adds
// into it; the deterministic entry points overwrite it and pass zero_c = false).
int t_gemm_prepare(const float* A, const float* B, float* C, const SeqpanGemm* gp, cudaStream_t st, int& split, long long& gz,
                   bool zero_c = true);

// Deterministic split-K, shared by seqpan_t_gemm_det and seqpan_t_gemm_bf16_det: the K-splits store their raw partial tiles to
// scratch [split][M][N] (plain stores); t_gemm_splitk_reduce then writes C = alpha * (((p0 + p1) + p2) + ...) + bias + beta * C,
// one thread per element.  t_gemm_det_check: SEQPAN_E_WORKSPACE unless the scratch holds t_gemm_det_scratch(g) bytes.
size_t t_gemm_det_scratch(const SeqpanGemm& g);
int t_gemm_det_check(const SeqpanGemm& g, const void* scratch, size_t scratch_bytes);
int t_gemm_splitk_reduce(float* C, const float* part, const float* bias, const SeqpanGemm& g, int split, cudaStream_t st);
