// Host-side pieces shared by the training GEMM launchers (train_ops.cu: fp32 SIMT, train_tc.cu: bf16 tensor cores).
#pragma once
#include <cuda_runtime.h>

#include "../../include/seqpan_b200.h"

// error path of the seqpan_t_* entry points (read back by seqpan_t_last_error)
int tfail(const char* msg);
int tcheck();

// Argument checks and the split-K pre-pass of seqpan_t_gemm, shared so that both GEMM entry points reject the same inputs
// with the same errors.  On SEQPAN_OK, `gz` = CTAs along grid z (batch0 * batch1 * split), 0 when there is nothing to launch
// (M == 0 or N == 0); with split > 1 and beta == 0 the C view has been zeroed on `st`.
int t_gemm_prepare(const float* A, const float* B, float* C, const SeqpanGemm* gp, cudaStream_t st, int& split, long long& gz);
