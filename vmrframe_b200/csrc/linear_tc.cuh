// Tensor-core (tcgen05 + TMA + TMEM) linear layers of the bf16 mode: interface used by seqpan_api.cu.
#pragma once
#include "common.cuh"

// One slot per projection weight that a tcgen05 kernel of the bf16 forward reads; the bf16 weight copy and its TMA
// descriptor are built once at pack time and addressed by slot.
enum TcSlot {
  TC_ENC_PW0 = 0, TC_ENC_PW1, TC_ENC_PW2, TC_ENC_PW3,
  TC_TENC_PW0, TC_TENC_PW1, TC_TENC_PW2, TC_TENC_PW3,   // the text's own encoder (BackBone variant)
  TC_DAB0,  // + k * TC_DAB_STRIDE + one of the TC_DAB_* below
  TC_DAB_QKV = 0, TC_DAB_TKV, TC_DAB_SDENSE, TC_DAB_XDENSE, TC_DAB_BIL, TC_DAB_D1, TC_DAB_D2,
  TC_DAB_SGSD, TC_DAB_XGXD, TC_DAB_BILGD,   // folded products s_gate.s_dense, x_gate.x_dense, [bilinear_1|bilinear_2].guided_dense
  TC_DAB_STRIDE,
  TC_Q2V_LIN = TC_DAB0 + 2 * TC_DAB_STRIDE, TC_V2Q_LIN, TC_CAT,
  TC_PRED_PW0, TC_PRED_PW1, TC_PRED_PW2, TC_PRED_PW3, TC_INPROJ, TC_OUTPROJ, TC_PRED_DENSE, TC_START_HID, TC_END_HID,
  TC_NUM_SLOTS
};

struct TcSlotInfo {
  void* w_bf16;  // [N, Kpad] bf16, K-major
  int N, K;
  unsigned char tmap[128] __attribute__((aligned(64)));  // CUtensorMap of the weight
};

struct TcArena {
  TcSlotInfo slot[TC_NUM_SLOTS];
};
struct TcWorkspace {
  void* sa_bf16;      // [M,128] bf16 attention outputs feeding the fused DualAttentionBlock chain
  void* xa_bf16;
  void* qkv_bf16;     // [M,384] / [M,256] bf16 projections feeding the tcgen05 dual attention
  void* tkv_bf16;
  void* hb_q;         // head-blocked bf16 q/k/v of the predictor's in_proj: [L][4][B][64|64|32]
  void* hb_k;
  void* hb_v;
};

void tc_carve_arena(char* base, size_t& off, const SeqpanShapes& s, TcArena& a);
void tc_carve_workspace(char* base, size_t& off, const SeqpanShapes& s, int B, int T, TcWorkspace& w);
// slot_src[i]: fp32 [N,K] weight of slot i (device).  Converts to bf16 and encodes the weight's TMA descriptor.
int tc_pack(const SeqpanShapes& s, const float* const* slot_src, TcArena& a, cudaStream_t st);
// fp32 operands straight from global memory (TMA) on kind::tf32: y = act(x.w^T + bias) (+res).
// ln_g != nullptr (N == ldy == 128, no residual / ReLU): y = LayerNorm(x.w^T + bias) -- the LayerNorm rides in the epilogue.
int tc_linear_tf32(const float* x, int ldx, const float* w, const float* bias, const float* res, float* y, int ldy,
                   long long M, int N, int K, bool relu, cudaStream_t st, const float* ln_g = nullptr,
                   const float* ln_b = nullptr, float ln_eps = 0.f);
const char* tc_last_error();
// TMA descriptor of a bf16 activation matrix [rows, K] (row stride ld elements), box 64 x 128, 128-byte swizzle.
int tc_make_act_tmap(void* map_out /*CUtensorMap*/, const void* ptr, long long rows, int K, int ld, int box_rows = 128);
// TMA descriptor of an fp32 matrix [rows, K] (row stride ld elements), box 32 x box_rows, 128-byte swizzle (loads and stores).
int tc_make_f32_tmap(void* map_out /*CUtensorMap*/, const void* ptr, long long rows, int K, int ld, int box_rows = 128);
// TMA descriptor with a 32-column x box_rows box and 64-byte swizzle (one attention head of a value matrix, MN-major B operand).
int tc_make_head_tmap(void* map_out /*CUtensorMap*/, const void* ptr, long long rows, int K, int ld, int box_rows);
// TMA descriptor of a head-blocked bf16 tensor [L][4][B][stride] as (d, b, head, l) with box (32, 1, 1, 128), 64-byte swizzle.
int tc_make_hb_tmap(void* map_out /*CUtensorMap*/, const void* ptr, int B, int L, int stride, int box_cols = 32);
size_t tc_op_scratch_bytes(long long M, int N, int K);
int tc_op_linear(const float* x, const float* w, const float* bias, const float* res, float* y, long long M, int N,
                 int K, bool relu, void* scratch, size_t scratch_bytes, cudaStream_t st);
