/*
 * seqpan_b200.h -- C ABI of the B200-native SeqPAN inference hot path.
 *
 * The reference (renjie-liang/VMRFrame) is pure Python: it has no plugin/FFI layer, its boundary is
 * the nn.Module `models/SeqPAN.py::SeqPAN` resolved by name (`main.py:21`).  This header is therefore
 * the boundary a maintainer would bind from that module (ctypes/cffi stub in INTEGRATION.md): plain
 * pointers and sizes, no torch types.  Every pointer is a DEVICE pointer unless the name ends in
 * `_host`.  All entry points return 0 on success or a negative SEQPAN_E_* code;
 * `seqpan_last_error()` gives the message.  The library never allocates device memory: the caller
 * owns weights, the packed-weight arena and the workspace (PyTorch's caching allocator in our host
 * module).  A handle is not thread-safe; use one handle per stream/thread.
 *
 * What each entry point replaces in the reference:
 *   seqpan_forward        models/SeqPAN.py:50-95   SeqPAN.forward (text/video embedding, shared
 *                         FeatureEncoder, 2x DualAttentionBlock both directions, 2x CQAttention,
 *                         CQConcatenate, match head with injected Gumbel noise, SeqPANPredictor)
 *   seqpan_span_decode    utils/engine.py:28-44    infer_basic      (vmask != NULL: mask + fractions)
 *                         models/layers.py:549-557 extract_index    (vmask == NULL: plain indices)
 *   seqpan_iou_counters   models/loss.py:83-90,103-109 + utils/utils.py:161-185
 *                         append_ious / calculate_iou / get_i345_mi as 5 summable counters
 *   seqpan_op_*           single blocks of models/layers.py, exposed for per-block parity tests
 */
#ifndef SEQPAN_B200_H_
#define SEQPAN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SEQPAN_ABI_VERSION 2

enum {
  SEQPAN_OK = 0,
  SEQPAN_E_INVALID = -1,   /* bad argument / shape outside the handle's limits */
  SEQPAN_E_CUDA = -2,      /* a CUDA runtime call or launch failed */
  SEQPAN_E_WORKSPACE = -3, /* workspace / arena too small or misaligned */
  SEQPAN_E_NODEVICE = -4   /* no sm_100 device available: there is NO CPU fallback */
};

/* Arithmetic of the dense projections.  LayerNorm/softmax/mask/decode are fp32 in both modes. */
enum {
  SEQPAN_PREC_FP32 = 0, /* fp32 FFMA everywhere: the rtol 1e-4 parity gate                     */
  SEQPAN_PREC_BF16 = 1, /* bf16 operands on tcgen05 tensor cores, fp32 accumulate (rtol 1e-2)   */
  SEQPAN_PREC_TF32 = 2  /* every dense projection on tcgen05 kind::tf32 straight from the fp32 rows (the arithmetic the
                           reference itself uses on a GPU: nn.Conv1d under torch's default cudnn.allow_tf32 = True,
                           SURVEY.md section 0 #16); attention products, softmax, LayerNorm stay fp32             */
};

/* Model constants fixed by every SeqPAN config of the reference (config/{charades,anet,tacos}/SeqPAN.yaml:
 * dim 128, num_heads 4, word_dim 300, char_dim 100) and by the hard-wired char-CNN (models/layers.py:55). */
#define SEQPAN_DIM 128
#define SEQPAN_HEADS 4
#define SEQPAN_HEAD_DIM 32
#define SEQPAN_WORD_DIM 300
#define SEQPAN_CHAR_DIM 100
#define SEQPAN_CHAR_OUT 100
#define SEQPAN_LABELS 4
#define SEQPAN_KSIZE 7
#define SEQPAN_MAX_VLEN 256
#define SEQPAN_MAX_TLEN 128

typedef struct SeqpanShapes {
  int32_t abi_version; /* SEQPAN_ABI_VERSION */
  int32_t max_batch;   /* largest B a forward will be called with                         */
  int32_t vlen;        /* L = configs.model.vlen (position tables have vlen rows)          */
  int32_t max_tlen;    /* largest padded word count T (<= vlen: text shares the video position table) */
  int32_t max_clen;    /* largest padded characters-per-word C (>= 4)                      */
  int32_t vdim;        /* configs.model.vdim                                               */
  int32_t num_words;   /* configs.num_words (rows of cat[pad, unk, glove])                 */
  int32_t num_chars;   /* configs.num_chars                                                */
  int32_t precision;   /* SEQPAN_PREC_*                                                    */
  int32_t pretrained_words; /* 1: pad_vec/unk_vec/glove_vec triplet, 0: single word_emb.weight table */
  int32_t variant;     /* SEQPAN_VARIANT_*: which sibling model of the reference the handle computes */
} SeqpanShapes;

/* Sibling models that reuse SeqPAN's blocks (SURVEY.md section 8 row f3).  The weight table is shared; entries a variant
 * does not use have seqpan_weight_numel() == 0 and may be NULL. */
enum {
  SEQPAN_VARIANT_SEQPAN = 0,   /* models/SeqPAN.py:11-95 */
  SEQPAN_VARIANT_BASEFAST = 1, /* models/BaseFast.py:10-97: 2-layer shared FeatureEncoder, no DualAttentionBlocks */
  SEQPAN_VARIANT_MULTITEACHER = 2, /* models/MultiTeacher.py:12-91 (student forward): 2-layer shared FeatureEncoder, SeqPAN otherwise */
  SEQPAN_VARIANT_STUDENT4 = 4, /* the student of models/OneTeacher.py:18-31,98-112: SeqPAN's blocks on a 4-layer shared encoder WITHOUT the
                                  DualAttentionBlock passes (and without their parameters) */
  SEQPAN_VARIANT_BACKBONE = 3  /* models/BackBone.py:10-75: the text has its own FeatureEncoder (tfeat_encoder), no match head
                                  (no match_conv1d / label_embs / Gumbel noise: the concat output feeds the predictor unmasked);
                                  the match_score and gumbel arguments of seqpan_forward are ignored and may be NULL */
};

typedef struct SeqpanHandle SeqpanHandle;

/* ---- weight table -------------------------------------------------------------------------------
 * The model's parameters are passed as an array of fp32 device pointers indexed like the table
 * returned by seqpan_weight_name(): entry i is the tensor stored under that key in the reference
 * state_dict (SURVEY.md App. A.6), contiguous, in the reference's own layout (Conv1d weights
 * [out,in,1], nn.MultiheadAttention in_proj_weight [384,128], ...).  Dead parameters of the reference
 * (BiLinear.dense_2, DualMultiAttention.layer_norm1/2/out_layer; models/layers.py:257-263,325-327)
 * are not in the table. */
int seqpan_num_weights(void);
const char* seqpan_weight_name(int index);
/* number of fp32 elements expected for weight `index` under `shapes` (for caller-side checks) */
int64_t seqpan_weight_numel(const SeqpanShapes* shapes, int index);

/* ---- lifetime ----------------------------------------------------------------------------------- */
size_t seqpan_arena_bytes(const SeqpanShapes* shapes);     /* packed/derived weights (bf16 copies, fused tables) */
size_t seqpan_workspace_bytes(const SeqpanShapes* shapes); /* activations of one forward at max shapes */

/* Creates a handle and packs the weights into `arena` (device, 256-byte aligned, seqpan_arena_bytes).
 * `weights` is a HOST array of seqpan_num_weights() device pointers.  Packing runs on `stream`.
 * Call seqpan_repack() after the parameters changed in place (e.g. load_state_dict). */
int seqpan_create(const SeqpanShapes* shapes, const float* const* weights_host, void* arena,
                  size_t arena_bytes, void* stream, SeqpanHandle** out);
int seqpan_repack(SeqpanHandle* h, const float* const* weights_host, void* stream);
void seqpan_destroy(SeqpanHandle* h);

/* ---- the hot path ------------------------------------------------------------------------------- */
/* One forward over a batch of B query-video pairs (B <= max_batch, T <= max_tlen, 4 <= C <= max_clen).
 *   word_ids [B,T] int64, char_ids [B,T,C] int64, vfeat [B,vlen,vdim] fp32, vmask [B,vlen] fp32 {0,1},
 *   tmask [B,T] fp32 {0,1}, gumbel [B,vlen,4] fp32 = -log(Exp(1)) noise (models/SeqPAN.py:79).
 * Outputs: slogits, elogits [B,vlen] fp32 (unmasked), match_score [B,vlen,4] fp32.
 * Asynchronous on `stream` (a cudaStream_t); no host synchronisation, no allocation. */
int seqpan_forward(SeqpanHandle* h, const int64_t* word_ids, const int64_t* char_ids, const float* vfeat,
                   const float* vmask, const float* tmask, const float* gumbel, int B, int T, int C,
                   float* slogits, float* elogits, float* match_score, void* workspace,
                   size_t workspace_bytes, void* stream);

/* The same forward when several of the B pairs share a clip (dense-query datasets: TACoS has ~150 queries per video):
 * vfeat_unique [U,vlen,vdim] holds every clip ONCE, video_index [B] int32 (device) names the clip of pair b (0 <= . < U).
 * VisualProjection + the video half of the shared FeatureEncoder (models/SeqPAN.py:57,59) do not depend on the query, so
 * they run on U*vlen rows and only U clips have to cross PCIe; the outputs equal seqpan_forward on the expanded
 * [B,vlen,vdim] tensor.  vmask stays per pair ([B,vlen]).  The reference has no such entry point (it re-encodes the clip
 * for every query); SURVEY.md section 8 row (f1). */
int seqpan_forward_shared_video(SeqpanHandle* h, const int64_t* word_ids, const int64_t* char_ids,
                                const float* vfeat_unique, const int32_t* video_index, int U, const float* vmask,
                                const float* tmask, const float* gumbel, int B, int T, int C, float* slogits,
                                float* elogits, float* match_score, void* workspace, size_t workspace_bytes,
                                void* stream);

/* The query-independent video branch on its own (DESIGN.md section 12): VisualProjection + the video half of the shared
 * FeatureEncoder (2 layers for BaseFast / MultiTeacher, 4 otherwise) of U clips vfeat [U,vlen,vdim] fp32 -> venc
 * [U,vlen,128] fp32, the caller's buffer.  1 <= U <= max_batch (the workspace holds max_batch*vlen rows).  vfeat and venc
 * must be 16-byte aligned (TMA and float4 access; every cudaMalloc'ed or torch tensor start is).  A clip's rows do
 * not depend on the other clips of the call.  The encodings stay valid for this handle's weights and precision. */
int seqpan_encode_videos(SeqpanHandle* h, const float* vfeat, int U, float* venc, void* workspace, size_t workspace_bytes,
                         void* stream);

/* seqpan_forward_shared_video on stored encodings: venc [U,vlen,128] from seqpan_encode_videos, video_index [B] int32
 * (device) names the clip of pair b; out-of-range indices are clamped.  venc must be 16-byte aligned (float4 reads).  U is the size of the caller's encoding library and
 * is not bounded by B; video_index == NULL pairs b with row block b (requires U >= B).  The outputs are bit-identical to
 * seqpan_forward_shared_video on the raw clips.  Debug tap "video_affine" does not exist on this path. */
int seqpan_forward_encoded(SeqpanHandle* h, const int64_t* word_ids, const int64_t* char_ids, const float* venc,
                           const int32_t* video_index, int U, const float* vmask, const float* tmask, const float* gumbel,
                           int B, int T, int C, float* slogits, float* elogits, float* match_score, void* workspace,
                           size_t workspace_bytes, void* stream);

/* Span decode.  vmask != NULL: infer_basic (mask_logits, softmax, triu outer-product argmax, indices
 * divided by vmask.sum(1)) -> fracs [B,2] fp32.  vmask == NULL: extract_index.  start_idx/end_idx
 * [B] int64 and fracs may each be NULL.  Ties resolve to the lowest index (torch CPU behaviour). */
int seqpan_span_decode(const float* slogits, const float* elogits, const float* vmask, int B, int L,
                       int64_t* start_idx, int64_t* end_idx, float* fracs, void* stream);

/* counters[0..4] (fp64, device) += {n, sum IoU, #IoU>=0.3, #IoU>=0.5, #IoU>=0.7} of fracs vs gt [B,2]. */
int seqpan_iou_counters(const float* fracs, const float* gt_fracs, int B, double* counters, void* stream);

/* Reproducible evaluation sweeps (DESIGN.md section 13).
 * seqpan_gumbel_noise: out [B,L,4] fp32 (16-byte aligned) = Gumbel(0,1) noise of batch `batch_id` of a sweep seeded with `seed`,
 * a function of (seed, batch_id, B, L) alone.  Philox4x32-10 with key = (seed & 0xffffffff, seed >> 32) and counter =
 * (b * L + l, batch_id, 0, 0); its four output words x are the labels c = 0..3 of row (b, l).  u = ((x >> 9) + 0.5f) * 2^-23
 * (exact in fp32, never 0 or 1) and out = -logf(-logf(u)) with IEEE logf.  0 <= B, B * L < 2^32, 1 <= L <= SEQPAN_MAX_VLEN.
 * seqpan_iou_counters_exact: seqpan_iou_counters with each sample's fp64 IoU rounded to rint(iou * 2^28) * 2^-28 before it is
 * added to the sum (the thresholds test the unrounded IoU).  Every partial sum is then an integer multiple of 2^-28, so the
 * adds, and any later sum of such buffers, are exact in any order while the sample count stays <= 2^25; the mean IoU moves by
 * less than 2^-29 per sample.  Both: no allocation, no host synchronisation, shape-only work split (graph-capturable). */
int seqpan_gumbel_noise(uint64_t seed, uint32_t batch_id, int B, int L, float* out, void* stream);
int seqpan_iou_counters_exact(const float* fracs, const float* gt_fracs, int B, double* counters, void* stream);

/* Top-k spans per sample with greedy temporal NMS (infer_basic's probabilities; DESIGN.md section 11).  Candidates are the
 * spans i <= j with score sp[i]*ep[j] > 0, best first, exact ties to the lower i, then the lower j.  Each of k rounds keeps
 * the best candidate not yet kept and not suppressed: a kept (a,b) suppresses (i,j) when union > 0 and
 * (float)inter >= nms_thresh * (float)union on the integer indices (nms_thresh = 1: plain top-k).
 * Outputs in selection order: start_idx/end_idx [B,k] int64, scores [B,k] fp32, fracs [B,k,2] fp32 (nullable; indices
 * divided by vmask.sum(1), or by L when vmask is NULL).  Slots beyond the last surviving candidate are -1, -1, 0, -1.
 * 1 <= k <= SEQPAN_TOPK_MAX, 0 < nms_thresh <= 1, 1 <= L <= SEQPAN_MAX_VLEN.  No allocation, no host synchronisation. */
#define SEQPAN_TOPK_MAX 32
int seqpan_span_topk(const float* slogits, const float* elogits, const float* vmask, int B, int L, int k, float nms_thresh,
                     int64_t* start_idx, int64_t* end_idx, float* scores, float* fracs, void* stream);

/* counters[0..3] (fp64, device) += {n, #>=0.3, #>=0.5, #>=0.7} of the best IoU over each sample's filled top-k slots
 * (fracs [B,k,2] from seqpan_span_topk, empty slots -1) against gt [B,2]: R@k as counters that add exactly across shards. */
int seqpan_topk_counters(const float* fracs, const float* gt_fracs, int B, int k, double* counters, void* stream);

/* Host -> device copy of BaseCollate's zero-padded clip features [B,L,row_floats] (utils/BaseDataset.py:201-234 pads
 * every clip to vlen rows) that moves only the first valid_rows[b] rows of each sample over PCIe and writes the
 * padding rows as zeros on the device.  src_host must be PINNED host memory (cudaHostAlloc / torch pin_memory).
 * mode 0: one cudaMemcpyAsync per sample + a zero-fill kernel; mode N >= 1: ONE kernel of N CTAs that reads the pinned
 * buffer directly (UVA zero-copy, coalesced 16-byte loads).  valid_rows_host (pinned, B int32) must stay alive until the
 * stream has consumed it; valid_rows_dev is B int32 of device scratch.  Rows of src_host beyond valid_rows[b] are never
 * read: they are zeros by the collate contract. */
int seqpan_h2d_ragged(float* dst, const float* src_host, const int32_t* valid_rows_host, int32_t* valid_rows_dev,
                      int B, int L, int row_floats, int mode, void* stream);

/* Clip resampling + padding + mask on the device, for clips that are already resident in HBM: the feature half of
 * sample_vfeat_linear / interpolate_avrage (utils/data_utils.py:161-199; BaseDataset.__getitem__, utils/BaseDataset.py:40),
 * pad_video_seq (utils/data_utils.py:70-84) and convert_length_to_mask as BaseCollate applies them
 * (utils/BaseDataset.py:209-213), for a whole batch in one launch.
 * raw [row_offsets[B], row_floats] fp32 (device): the clips' rows back to back; clip b = rows [row_offsets[b], row_offsets[b+1]).
 * row_offsets_host: B+1 ascending int64 on the HOST (validated there; if PINNED it must stay alive until the stream has
 * consumed it, pageable memory is staged by cudaMemcpyAsync before the call returns);
 * row_offsets_dev: B+1 int64 of device scratch.  mode = configs.dataprocess.sample_type (enum below).
 * vfeats [B,vlen,row_floats] fp32, vmask [B,vlen] fp32 {0,1} (may be NULL), vlens [B] int64 (may be NULL), all device.
 * row_floats = 1 resamples the 1-D frame labels the same way (interpolate_avrage(label, max_vlen)).
 * Errors like the reference: "original" with a clip longer than vlen (torch.stack would fail), "samelen" on an empty clip. */
enum { SEQPAN_SAMPLE_ORIGINAL = 0, SEQPAN_SAMPLE_TRUNCATION = 1, SEQPAN_SAMPLE_SAMELEN = 2 };
int seqpan_collate_clips(const float* raw, const int64_t* row_offsets_host, int64_t* row_offsets_dev, int B, int vlen,
                         int row_floats, int mode, float* vfeats, float* vmask, int64_t* vlens, void* stream);

/* Text half of BaseCollate.__call__ (utils/BaseDataset.py:201-207) on the device: pad_seq (utils/data_utils.py:42-52) of the word
 * ids to the batch maximum T, pad_char_seq (:55-68) of the character ids to [B,T,C] (C = longest word of the batch), and
 * tmask = (word_ids != 0).  words [W] int64 = the word ids of all samples back to back, word_offsets [B+1] (sample b owns words
 * word_offsets[b] .. word_offsets[b+1]); chars [N] int64 = the characters of all words back to back, char_offsets [W+1].  All
 * device pointers.  The caller passes T = max words per sample and C = max characters per word (what pad_seq / pad_char_seq
 * compute with max_length=None); shorter limits truncate like the reference's seq[:max_length]. */
int seqpan_collate_text(const int64_t* words, const int64_t* word_offsets, const int64_t* chars, const int64_t* char_offsets,
                        int B, int T, int C, int64_t* word_ids, int64_t* char_ids, float* tmask, void* stream);

/* Copies a named intermediate of the LAST forward out of the workspace (per-block parity tests):
 * "text_emb","video_affine","venc","tenc","dab1_v","dab1_t","dab2_v","dab2_t","t2v","v2t","fuse",
 * "fuse2","fep_s","fep_e".  `out` receives rows*128 fp32; returns the row count or a negative error. */
int64_t seqpan_debug_tap(SeqpanHandle* h, const char* name, const void* workspace, float* out,
                         int64_t out_capacity_floats, void* stream);

/* Debug taps on/off (off by default: taps cost one device copy each). */
int seqpan_set_debug(SeqpanHandle* h, int on);
/* Per-launch CUDA-event timing on the launching stream.  After seqpan_set_profile(h,1) every kernel launch of
 * seqpan_forward is bracketed by two events; seqpan_profile_summary synchronises and writes one
 * "tag count total_ms" line per kernel tag into buf.  Used by bench.py for the roofline of the dominant kernel. */
int seqpan_set_profile(SeqpanHandle* h, int on);
int seqpan_profile_summary(SeqpanHandle* h, char* buf, size_t cap);

/* The text branch of a forward (embedding + query projection: two 50-CTA kernels) runs on a side stream of the handle,
 * concurrently with the video affine (+2.5 % device-resident).  A caller that keeps the PCIe bus busy with its own copy KERNEL
 * next to the forwards (vmrframe_b200.evaluate) turns it off: the extra concurrency takes issue slots from that kernel and the
 * sweep is bound by it (measured: 157 k -> 143 k queries/s end to end).  Default on; SEQPAN_NO_SIDE_STREAM=1 never creates it. */
int seqpan_set_side_stream(SeqpanHandle* h, int on);

/* number of kernel launches issued by the last seqpan_forward on this handle */
int seqpan_last_launch_count(const SeqpanHandle* h);

/* ---- training primitives (SURVEY.md section 8 rows a19 / f4) -------------------------------------------------
 * The training step of the reference (train_engine_SeqPAN, models/SeqPAN.py:171-182; lossfun_loc / lossfun_match,
 * models/loss.py:24-54; zero_grad / backward / clip_grad_norm_(1.0) / AdamW step, main.py:93-97, utils/utils.py:87-97) is
 * torch autograd over ~430 ATen operators.  Here the host module (vmrframe_b200/train.py) runs a reverse-mode tape whose
 * every node is one of the fp32 kernels below (forward rule and vector-Jacobian rule); no arithmetic happens on the host.
 * All pointers are device pointers; every call is asynchronous on `stream`. */
typedef struct SeqpanGemm {       /* C[b0,b1] = alpha * A . B + beta * C;  X(i,j) = X[i * x_rs + j * x_cs] (+ batch offsets) */
  int64_t M, N, K;
  int64_t a_rs, a_cs, b_rs, b_cs, c_rs, c_cs;   /* A is M x K, B is K x N, C is M x N: transposes are stride swaps */
  int64_t a_b0, a_b1, b_b0, b_b1, c_b0, c_b1;   /* batch strides (0 broadcasts an operand over a batch dim)            */
  int32_t batch0, batch1;                       /* two batch dims (>= 1): e.g. (sample, head)                          */
  float alpha, beta;
  int32_t splitk;                               /* > 1: K split over CTAs, partial sums added atomically (beta 0 or 1, one batch) */
} SeqpanGemm;
/* bias (may be NULL): a [N] vector added to every row of the product (the bias of a Conv1D / nn.Linear) */
int seqpan_t_gemm(const float* A, const float* B, float* C, const float* bias, const SeqpanGemm* g, void* stream);
/* The same product on the tensor cores (bf16 mixed precision): every element of A and B is rounded to bf16
 * (round-to-nearest-even) before the product, products accumulate in fp32; C, bias, alpha and beta stay fp32.  Every other
 * field of SeqpanGemm means what it means for seqpan_t_gemm, and the same bad arguments give the same errors.  Operands need
 * no alignment; elements of C outside the (M, N, c_rs, c_cs) view are never touched. */
int seqpan_t_gemm_bf16(const float* A, const float* B, float* C, const float* bias, const SeqpanGemm* g, void* stream);

enum {   /* out = f(a, b, c) element-wise over a 4-D index space with per-operand strides (0 = broadcast) */
  SEQPAN_EW_COPY = 0,        /* a                                    */
  SEQPAN_EW_AXPBY = 1,       /* alpha * a + beta * b                 */
  SEQPAN_EW_MUL = 2,         /* alpha * a * b                        */
  SEQPAN_EW_RELU = 3,        /* max(a, 0)                            */
  SEQPAN_EW_RELU_BWD = 4,    /* b > 0 ? a : 0   (a = grad, b = output) */
  SEQPAN_EW_SIGMOID = 5,
  SEQPAN_EW_SIGMOID_BWD = 6, /* a * b * (1 - b) (b = sigmoid output) */
  SEQPAN_EW_MASK_LOGITS = 7, /* a + (1 - b) * -1e30   (models/layers.py:9-12) */
  SEQPAN_EW_FMA = 8,         /* a * b + c                            */
  SEQPAN_EW_LOG = 9, SEQPAN_EW_EXP = 10, SEQPAN_EW_DIV = 11, SEQPAN_EW_SQRT = 12,
  SEQPAN_EW_AFFINE = 13,     /* alpha * a + beta                     */
  SEQPAN_EW_EQ = 14,         /* a == alpha ? 1 : 0                   */
  SEQPAN_EW_DIV_SAFE = 15,   /* b != 0 ? a / b : 0  (adjoint of a 2-norm at the origin, like torch.norm) */
  SEQPAN_EW_DROPOUT = 16     /* b >= alpha ? a * beta : 0  (b = the uniform draw or a 0/1 keep-mask, alpha = p, beta = 1/(1-p)):
                                nn.Dropout's forward and, applied to the gradient with the same b, its adjoint */
};
typedef struct SeqpanEwise {
  int32_t op, accumulate;    /* accumulate != 0: out += f(...)       */
  int64_t shape[4];
  int64_t so[4], sa[4], sb[4], sc[4];
  float alpha, beta;
} SeqpanEwise;
int seqpan_t_ewise(float* out, const float* a, const float* b, const float* c, const SeqpanEwise* e, void* stream);

typedef struct SeqpanSoftmax {   /* softmax over `cols` elements c_stride apart, for rows (r0, r1) at r0 * r0_stride + r1 * r1_stride */
  int64_t rows0, rows1, r0_stride, r1_stride;
  int32_t cols; int64_t c_stride;
} SeqpanSoftmax;
int seqpan_t_softmax(float* y, const float* x, const SeqpanSoftmax* s, void* stream);
int seqpan_t_softmax_bwd(float* dx, const float* y, const float* dy, const SeqpanSoftmax* s, void* stream);   /* dx = y (dy - sum(y dy)) */

/* LayerNorm over 128-wide rows (forward: seqpan_op_layernorm): dx written, dgamma / dbeta ACCUMULATED (atomics). */
int seqpan_t_layernorm_bwd(float* dx, float* dgamma, float* dbeta, const float* x, const float* dy, const float* gamma,
                           float eps, int64_t M, void* stream);
/* Depthwise conv k = 7, pad 3, no bias, along the rows of equal-length segments of a [rows,128] matrix, w [128,1,7]
 * (models/layers.py:131).  flip = 1 applies the reversed taps = the input gradient.  dw is ACCUMULATED. */
int seqpan_t_dwconv(float* y, const float* x, const float* w, int64_t rows, int len, int flip, void* stream);
int seqpan_t_dwconv_bwd_w(float* dw, const float* x, const float* dy, int64_t rows, int len, void* stream);
/* out[n,:] = table[ids[n],:] and its adjoint dtable[ids[n],:] += dout[n,:] (ids clamped to the table). */
int seqpan_t_gather_rows(float* out, const float* table, const int64_t* ids, int64_t n, int dim, int64_t table_rows, void* stream);
int seqpan_t_scatter_add_rows(float* dtable, const float* dout, const int64_t* ids, int64_t n, int dim, int64_t table_rows, void* stream);
/* max over the middle dim of x [N,P,C] with the index of the first maximum (torch.max(dim)); bwd scatters dout into a zeroed dx. */
int seqpan_t_maxpool(float* out, int32_t* idx, const float* x, int64_t N, int P, int C, void* stream);
int seqpan_t_maxpool_bwd(float* dx, const float* dout, const int32_t* idx, int64_t N, int P, int C, void* stream);
/* *out_accum (fp64, device) += sum(x^2): the squared gradient norm clip_grad_norm_ needs (main.py:95). */
int seqpan_t_sumsq(const float* x, int64_t n, double* out_accum, void* stream);
typedef struct SeqpanAdamW {     /* torch.optim.AdamW (utils/utils.py:94): decoupled decay, bias-corrected moments */
  float lr, beta1, beta2, eps, weight_decay;
  float bias1, bias2_sqrt;       /* 1 - beta1^t, sqrt(1 - beta2^t) */
  float max_grad_norm;           /* > 0 and sumsq != NULL: gradients are scaled by min(1, max_norm / (sqrt(*sumsq) + 1e-6)) */
} SeqpanAdamW;
/* dyn != NULL: device float[3] = {lr, 1 - beta1^t, sqrt(1 - beta2^t)} overrides the struct's per-step scalars, so that a whole
 * optimisation step captured as a CUDA graph can be replayed with the scalars of step t written before each launch. */
int seqpan_t_adamw(float* p, const float* g, float* m, float* v, int64_t n, const SeqpanAdamW* a, const double* sumsq,
                   const float* dyn, void* stream);
const char* seqpan_t_last_error(void);

/* ---- deterministic training mode --------------------------------------------------------------------------------------------
 * The entry points above combine partial sums with float atomics (split-K GEMM, LayerNorm dgamma / dbeta, depthwise-conv dw,
 * embedding scatter-add, the clipping norm), so their last bits depend on CTA scheduling.  The entry points below compute the
 * same quantities with every output element written by one thread, or combined from partials in a fixed order; the work split
 * depends only on the shapes.  Run twice on the same inputs they give bit-identical results.  Arguments, errors and the
 * ACCUMULATE contracts are those of the atomic entry points.  The library still never allocates: where partials are needed the
 * caller passes device scratch of at least the bytes the matching *_scratch_bytes query returns (SEQPAN_E_WORKSPACE when it
 * is NULL or smaller).  The scratch is only written before it is read: it needs no initialisation.
 *
 * seqpan_t_gemm_det / seqpan_t_gemm_bf16_det: split-K > 1 stores the raw product of each K-split (K ranges as in
 *   seqpan_t_gemm) to scratch [split][M][N], then C = alpha * (((p0 + p1) + p2) + ...) + bias + beta * C, one thread per
 *   element, splits in ascending order.  Without split-K they equal seqpan_t_gemm / _bf16 (and need no scratch). */
size_t seqpan_t_gemm_det_scratch_bytes(const SeqpanGemm* g);     /* splitk * M * N * 4 for splitk > 1, else 0 */
int seqpan_t_gemm_det(const float* A, const float* B, float* C, const float* bias, const SeqpanGemm* g, void* scratch,
                      size_t scratch_bytes, void* stream);
int seqpan_t_gemm_bf16_det(const float* A, const float* B, float* C, const float* bias, const SeqpanGemm* g, void* scratch,
                           size_t scratch_bytes, void* stream);
/* Each CTA of a grid fixed by M (resp. rows) writes its partial dgamma | dbeta rows (resp. its [128 x 7] dw) to scratch; one
 * ordered pass adds the partials in ascending CTA order and adds the result once into dgamma / dbeta (resp. dw). */
size_t seqpan_t_layernorm_bwd_det_scratch_bytes(int64_t M);
int seqpan_t_layernorm_bwd_det(float* dx, float* dgamma, float* dbeta, const float* x, const float* dy, const float* gamma,
                               float eps, int64_t M, void* scratch, size_t scratch_bytes, void* stream);
size_t seqpan_t_dwconv_bwd_w_det_scratch_bytes(int64_t rows);
int seqpan_t_dwconv_bwd_w_det(float* dw, const float* x, const float* dy, int64_t rows, int len, void* scratch,
                              size_t scratch_bytes, void* stream);
/* dtable[r,:] += s_r with s_r = (((0 + dout[n0,:]) + dout[n1,:]) + ...) over the positions n0 < n1 < ... whose clamped id is r,
 * in ascending n, in fp32; a row that no id hits is left untouched.  One CTA owns each table row: no scratch. */
int seqpan_t_scatter_add_rows_det(float* dtable, const float* dout, const int64_t* ids, int64_t n, int dim, int64_t table_rows,
                                  void* stream);
/* fp64 partial sums of a grid fixed by n (8-byte aligned scratch), added in ascending order by one thread, once into *out_accum. */
size_t seqpan_t_sumsq_det_scratch_bytes(int64_t n);
int seqpan_t_sumsq_det(const float* x, int64_t n, double* out_accum, void* scratch, size_t scratch_bytes, void* stream);

/* ---- single-block entry points (tests / micro-benchmarks) --------------------------------------- */
/* y[M,N] (+)= x[M,K] . w[N,K]^T + bias ; flags: bit0 ReLU, bit1 add `residual` [M,N] after activation.
 * precision SEQPAN_PREC_FP32: fp32 FFMA kernel.  SEQPAN_PREC_BF16: x and w are rounded to bf16 and the
 * product runs on tcgen05 (TMA-fed, TMEM accumulators); `scratch` must then hold
 * seqpan_op_linear_scratch_bytes(M,N,K) bytes.  precision 2: fp32 operands on tcgen05 kind::tf32 (no scratch). */
size_t seqpan_op_linear_scratch_bytes(int64_t M, int N, int K);
int seqpan_op_linear(const float* x, const float* w, const float* bias, const float* residual, float* y,
                     int64_t M, int N, int K, int flags, int precision, void* scratch, size_t scratch_bytes,
                     void* stream);
/* y = LayerNorm(x) over the last dim (128), affine, biased variance. */
int seqpan_op_layernorm(const float* x, const float* gamma, const float* beta, float eps, float* y,
                        int64_t M, void* stream);

const char* seqpan_last_error(void);
/* 1 if a CUDA device with compute capability 10.x is present, else 0 (never falls back to CPU). */
int seqpan_device_ok(void);

#ifdef __cplusplus
}
#endif
#endif /* SEQPAN_B200_H_ */
