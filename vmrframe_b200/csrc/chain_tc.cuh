// Fused tcgen05 chain kernels (bf16 mode): interface used by seqpan_api.cu.
#pragma once
#include "linear_tc.cuh"

const char* chain_last_error();
// phase timeline of the instrumented build (-DSEQPAN_TIMELINE): 64 SM-clock stamps; SEQPAN_E_INVALID otherwise
int chain_read_timeline(long long* out64);
int attn_read_timeline(long long* out64);
int tail_read_timeline(long long* out64);
int tc_read_timeline(long long* out64);

// Everything of a DualAttentionBlock after the attention cores, for all joint rows, in one launch
// (models/layers.py:362-381 and 288-297; tail_tc.cu).  hostv = HOST copies of: s_dense, x_dense, s_gate, x_gate,
// guided_dense biases, the packed bilinear bias [256] (2b + bias_value), dense_1, dense_2 biases, LayerNorm2 weight, bias.
// ln1_g / ln1_b are device pointers.  xout may alias xin (a CTA reads its rows before it writes them).
// The gate's row mask is read in place: rows [0, Mv) from vmask, rows [Mv, M) from tmask.
int chain_dab_post(const TcArena& a, int block, const void* sa_bf16, const void* xa_bf16, const float* xin, float* xout,
                   const float* vmask, const float* tmask, long long Mv, long long M, const float* const* hostv,
                   const float* ln1_g, const float* ln1_b, cudaStream_t st);

// out_A = LN_A(x).W_A^T + b_A and (slotB >= 0) out_B = LN_B(x).W_B^T + b_B from one read of x (fp32 outputs).
int chain_proj_ln(const TcArena& a, int slotA, int slotB, const float* x, long long M, float eps, const float* gA,
                  const float* bA, const float* gB, const float* bB, float* outA, const float* biasA, float* outB,
                  const float* biasB, cudaStream_t st, void* const* hb = nullptr, int hbL = 0, int hbB = 0,
                  const float* hb_mask = nullptr, bool out_bf16 = false);
// out_bf16: outA/outB are bf16 row-major [M, n*128] (cast the pointers).
// hb != nullptr: the three A tiles (q,k,v) are written as bf16 head blocks [L][4][B][64|64|32] instead of outA;
// q is pre-scaled by 1/sqrt(32), column 32 of q rows is 1 and column 32 of k rows is hb_mask[row] (additive key mask).

// Batch-axis attention of the predictor (TopSelfAttention2, models/layers.py:567-574) on tensor cores: one CTA per
// (position l, head); q/k/v are the head-blocked bf16 tensors above; out is bf16 [B*L,128].  B <= 256.
int attn_batch_tc(const void* q_hb, const void* k_hb, const void* v_hb, const float* vmask, void* out_bf16, int B, int L,
                  cudaStream_t st);

// Fused row-local tails (tail_tc.cu).
//   chain_fep_head   = FeatureEncoderPredict tail r = out_proj(att) + h; out = dense(LN_1e-5(r)) + r (att bf16 [M,128]),
//                      then the logit head logits = dense(hidden(cat[LN_1e-6(out), x])) in one launch;
//                      slot_hidden = TC_START_HID / TC_END_HID, x_bf16 = bf16 copy of the predictor input [M,128].
//   chain_fuse_match = CQConcatenate's projection (t2v half by tensor core, pooled half as the per-sample bias `pbias`
//                      [B,128]) + the match head; writes fuse, fuse2 (fp32), fuse2_bf16 and match_score.
//   launch_pool_bias = WeightedPool + its half of the concat projection: pbias[b] = Wcat[:, 128:] . pool(v2t[b]).
const char* tail_last_error();
// hostv = HOST copies of the small vectors (they travel as __grid_constant__ kernel parameters: constant-bank operands).
int chain_fep_head(const TcArena& a, int slot_hidden, const void* att_bf16, const void* x_bf16, const float* h, float* out,
                   long long M, const float* const* hostv /*b_o, ln_g, ln_b, b_d, head ln_g, head ln_b, b_h, w_d, b_dense*/,
                   float* logits, cudaStream_t st);
int chain_fuse_match(const TcArena& a, const float* t2v, int ldx, long long M, int L, const float* pbias,
                     const float* const* hostv /*b_cat [128], wm [4][128], label_embs [128][4], bm [4]*/, const float* gumbel,
                     const float* vmask, float* fuse_or_null, float* fuse2, void* fuse2_bf16, float* match_score, cudaStream_t st,
                     bool no_match = false);   // no_match (BackBone): fuse2 = fuse, no match head, match_score / gumbel unused
int launch_pool_bias(const float* v2t, const float* tmask, const float* pool_w, const float* wcat_f32, float* pbias, int B,
                     int T, cudaStream_t st);

// DualMultiAttention cores (models/layers.py:339-367) on tensor cores: one CTA per (sample, direction), all 4 heads.
// qkv_bf16 [M,384] = q|f_key|f_value and tkv_bf16 [M,256] = t_key|t_value (bf16, joint rows); outputs bf16 [M,128].
// Needs L <= 128 and T <= 64.
bool attn_dual_tc_supported(int L, int T);
int attn_dual_tc(const void* qkv_bf16, const void* tkv_bf16, const float* vmask, const float* tmask, void* sa_bf16,
                 void* xa_bf16, int B, int L, int T, cudaStream_t st);

// Whole 4-layer conv block + position add in one launch (group 0: nseg0 x len0 rows starting at row 0, len0 <=
// SEQPAN_MAX_VLEN, segments longer than 128 rows are tiled with halos; group 1: nseg1 x len1 rows right after, len1 <= 128;
// other lengths are SEQPAN_E_INVALID).  slot0 = tensor-core slot of the first pointwise weight.
// Optional tail: the LayerNorm + projections that consume the block's output (same semantics as chain_proj_ln with bf16
// row-major outputs, or head-blocked q/k/v when hb != nullptr), computed from the rows while they are still on the SM.
struct ChainProjTail {
  int slotA, slotB;            // tensor-core slots of the projection weights (slotB < 0: none)
  float eps;
  const float* gA; const float* bA; const float* gB; const float* bB;
  const float* biasA; const float* biasB;
  void* outA; void* outB;      // bf16 [Mtot, N]
  void* const* hb; int hbL, hbB; const float* hb_mask;
};
// `tab` = chain_conv_tab_floats() floats built once per weight set by chain_conv_tables (pointwise biases + depthwise tap
// tables with the LayerNorm affine folded in): every CTA bulk-copies them instead of rebuilding them.
size_t chain_conv_tab_floats();
int chain_conv_tables(const float* const* ln_g, const float* const* ln_b, const float* const* dw, const float* const* bias,
                      float* tab, cudaStream_t st);
int chain_conv_block(const TcArena& a, int slot0, const float* x, const float* pos, float* out, const float* tab, int nseg0,
                     int len0, int nseg1, int len1, cudaStream_t st, const ChainProjTail* tail = nullptr, int nlayers = 4);

// CQAttention both directions + cqa_linear in one launch (models/layers.py:417-437, models/SeqPAN.py:73-74): one CTA per
// (sample, direction); x = joint rows fp32; out_v [B*L, ldo_v] = q2v_attn(video ctx, text query), out_t [B*T, ldo_t] =
// v2q_attn(text ctx, video query).  Index 0 of the weight arrays = q2v_attn, 1 = v2q_attn.  Needs L, T <= 128.
bool cq_tc_supported(int L, int T);
int cq_attention_tc(const TcArena& a, const float* x, const float* vmask, const float* tmask, const float* const* w4c,
                    const float* const* w4q, const float* const* w4mlu, const float* const* bias, float* out_v, int ldo_v,
                    float* out_t, int ldo_t, int B, int L, int T, cudaStream_t st);
