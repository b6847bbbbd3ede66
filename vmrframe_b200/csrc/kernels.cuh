// Launchers of the fp32 (CUDA-core) SeqPAN kernels.  All are asynchronous on `st` and return the
// launch status.  Row buffers are row-major fp32 with 128 columns unless a leading dimension is given.
#pragma once
#include "common.cuh"

namespace sq {

// Up to 3 same-shaped problems in one launch (gridDim.z): y = act(x.w^T + bias) (+ residual)
struct LinearArgs {
  const float* x[3];
  const float* w[3];     // [N, K] row-major (nn.Conv1d weight [out, in, 1])
  const float* bias[3];  // [N] or nullptr
  const float* res[3];   // [M, ldr] or nullptr, added after the activation
  float* y[3];
  long long M;
  int N, K, ldx, ldw, ldy, ldr;
  int relu;
  int count;
};
cudaError_t launch_linear_f32(const LinearArgs& a, cudaStream_t st);

// Two groups of equal-length row segments inside one row buffer (video: B segments of L rows starting
// at row 0; text: B segments of T rows starting at row B*L).  Group 1 may be empty.
struct Segs {
  long long row0[2];
  int nseg[2];
  int len[2];
};

cudaError_t launch_layernorm(const float* x, int ldx, long long M, const float* g1, const float* b1, float eps,
                             float* y1, int ldy1, const float* g2, const float* b2, float* y2, int ldy2,
                             const float* copy_src, float* copy_dst, int ldcopy, cudaStream_t st);

// z = depthwise_conv7(LayerNorm(x (+pos))) per segment; if pos != nullptr also writes x0 = x + pos.
cudaError_t launch_ln_dwconv(const float* x, const float* pos, float* x0_out, const float* gamma, const float* beta,
                             float eps, const float* dw, float* z, const Segs& sg, cudaStream_t st);

cudaError_t launch_char_table(const float* const conv_w[4], const float* char_emb, int num_chars, float* table,
                              cudaStream_t st);
cudaError_t launch_embed_text(const int64_t* word_ids, const int64_t* char_ids, long long n_words, int C,
                              const float* pad, const float* unk, const float* glove, const float* table,
                              int num_words, int num_chars, const float* ctab, const float* cbias, float* out,
                              cudaStream_t st);

struct DualAttnArgs {
  const float* qkv;  // [M, 384]: q | f_key | f_value of LN1(x) for every joint row
  const float* tkv;  // [M, 256]: t_key | t_value of LNt(x)
  const float* vmask;
  const float* tmask;
  float* sa;  // [M,128] self-attention values, heads concatenated
  float* xa;  // [M,128] cross-attention values
  int B, L, T;
  void* sa_bf16;  // optional: bf16 [M,128] copies (operands of the fused tcgen05 chain); fp32 outputs skipped if set
  void* xa_bf16;
};
size_t dual_attention_smem(int L, int T);
cudaError_t launch_dual_attention(const DualAttnArgs& a, cudaStream_t st);

cudaError_t launch_gate_combine(const float* sg, const float* x, const float* xg, const float* s, float* out,
                                long long n4, cudaStream_t st);
cudaError_t launch_sigmoid_gate(const float* scva, const float* rowmask, float* y, long long M, cudaStream_t st);

struct CqArgs {
  const float* x;  // joint rows
  const float* vmask;
  const float* tmask;
  const float* w4c[2];
  const float* w4q[2];
  const float* w4mlu[2];
  float* cat[2];  // dir 0: [B*L, 512], dir 1: [B*T, 512]
  int B, L, T;
  int stage_video;  // 1: the video rows are staged in shared memory too (set by the launcher when they fit)
};
size_t cq_attention_smem(int L, int T);
cudaError_t launch_cq_attention(const CqArgs& a, cudaStream_t st);

cudaError_t launch_pool_tile(const float* v2t, const float* tmask, const float* pool_w, float* cat2, int B, int L,
                             int T, cudaStream_t st);
cudaError_t launch_match_head(const float* fuse, const float* wm, const float* bm, const float* gumbel,
                              const float* label_embs, const float* vmask, float* match_score, float* fuse2,
                              long long M, cudaStream_t st);

size_t batch_attention_smem(int B);
// out_bf16 != nullptr: write bf16 [B*L,128] (operand of the fused FEP tail) instead of the fp32 `out`
cudaError_t launch_batch_attention(const float* qkv, const float* vmask, float* out, void* out_bf16, int B, int L,
                                   cudaStream_t st);

cudaError_t launch_rowdot(const float* x, int ldx, const float* w, const float* b, float* out, long long M,
                          cudaStream_t st);
cudaError_t launch_build_rowmask(const float* vmask, long long nv, const float* tmask, long long nt, float* out,
                                 cudaStream_t st);
cudaError_t launch_span_decode(const float* s, const float* e, const float* vmask, int B, int L, int64_t* si,
                               int64_t* ei, float* fracs, cudaStream_t st);
// exact: the IoU sum adds multiples of 2^-28 (order-independent, DESIGN.md section 13)
cudaError_t launch_iou_counters(const float* fracs, const float* gt, int B, double* counters, bool exact, cudaStream_t st);
// rows = B * L rows of 4 labels, out 16-byte aligned
cudaError_t launch_gumbel_noise(uint64_t seed, uint32_t batch_id, uint32_t rows, float* out, cudaStream_t st);
cudaError_t launch_span_topk(const float* s, const float* e, const float* vmask, int B, int L, int k, float thr,
                             int64_t* si, int64_t* ei, float* scores, float* fracs, cudaStream_t st);
cudaError_t launch_topk_counters(const float* fracs, const float* gt, int B, int k, double* counters, cudaStream_t st);
cudaError_t launch_h2d_ragged(float* dst, const float* src_host, const int32_t* valid_dev, int B, int L, int row_floats,
                              int ctas, cudaStream_t st);
cudaError_t launch_zero_tail_rows(float* dst, const int32_t* valid_dev, int B, int L, int row_floats, cudaStream_t st);
cudaError_t launch_collate_clips(const float* raw, const int64_t* offs_dev, int B, int vlen, int row_floats, int mode,
                                 float* out, float* vmask, int64_t* vlens, cudaStream_t st);

cudaError_t launch_collate_text(const int64_t* words, const int64_t* woff, const int64_t* chars, const int64_t* coff, int B, int T, int C,
                                int64_t* word_ids, int64_t* char_ids, float* tmask, cudaStream_t st);

}  // namespace sq
