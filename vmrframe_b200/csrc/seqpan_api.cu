// C ABI of the SeqPAN hot path (include/seqpan_b200.h): handle, weight packing, the forward schedule and the
// single-block test entry points.  The schedule follows models/SeqPAN.py:50-95 step by step; video rows and
// text rows of a batch live in ONE joint row buffer ([B*L video rows | B*T text rows] x 128) because the
// shared FeatureEncoder and both directions of each DualAttentionBlock apply the same weights to both
// (models/SeqPAN.py:59-60, 64-70), so every such projection is a single launch.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>
#include <map>

#include "kernels.cuh"
#include "linear_tc.cuh"
#include "chain_tc.cuh"

using namespace sq;

// ---- weight table ---------------------------------------------------------------------------------
enum WeightId {
#define W(id, key, numel) W_##id,
#include "weights.def"
#undef W
  W_COUNT
};
static const char* const kWeightNames[W_COUNT] = {
#define W(id, key, numel) key,
#include "weights.def"
#undef W
};

static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

extern "C" const char* seqpan_last_error(void) { return g_err; }

static SqEnv g_env;
const SqEnv& sq_env() { return g_env; }
void sq_env_refresh() {
  auto on = [](const char* name) { const char* v = getenv(name); return v && v[0] == '1'; };
  auto num = [](const char* name, int dflt) { const char* v = getenv(name); return v ? atoi(v) : dflt; };
  SqEnv e;
  e.no_joint_attn = on("SEQPAN_NO_JOINT_ATTN"); e.no_graph = on("SEQPAN_NO_GRAPH"); e.force_graph = on("SEQPAN_GRAPH");
  e.no_side_stream = on("SEQPAN_NO_SIDE_STREAM");
  e.h2d_threads = num("SEQPAN_H2D_THREADS", 128);
  if (e.h2d_threads < 32 || e.h2d_threads > 1024 || (e.h2d_threads & 31)) e.h2d_threads = 128;
  g_env = e;
}
extern "C" int seqpan_num_weights(void) { return W_COUNT; }
extern "C" const char* seqpan_weight_name(int i) { return (i >= 0 && i < W_COUNT) ? kWeightNames[i] : nullptr; }
extern "C" int64_t seqpan_weight_numel(const SeqpanShapes* s, int index) {
  if (!s) return -1;
  switch (index) {
#define W(id, key, numel) \
  case W_##id:            \
    return (int64_t)(numel);
#include "weights.def"
#undef W
    default:
      return -1;
  }
}

extern "C" int seqpan_device_ok(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return 0;
  }
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10 ? 1 : 0;
}

// ---- layouts ----------------------------------------------------------------------------------------
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Carver {  // carves 256-byte aligned slices out of one allocation (or just measures when base == 0)
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base((char*)b) {}
  template <class T>
  T* take(size_t n) {
    off = align_up(off, 256);
    T* p = base ? (T*)(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
};

struct DabPacked {
  float *qkv_w, *qkv_b;  // [384,128] query|f_key|f_value, [384]
  float *tkv_w, *tkv_b;  // [256,128] t_key|t_value, [256]
  float *bil_w, *bil_b;  // [256,128] bilinear_1.dense_1|bilinear_2.dense_1, [256] = 2*b + bias_value
  // Folded products of the fused chain (two MMA round trips fewer, see dab_post_kernel):
  //   s_gate(s_dense(a)) = (Wsg.Wsd) a + (Wsg.b_sd + b_sg);  x_gate(x_dense(a)) likewise;
  //   bilinear(o + guided_dense(zin)) = Wbil.o + (Wbil.Wgd) zin + (Wbil.b_gd + bil_b)
  float *sgsd_w, *xgxd_w, *bilgd_w;   // [128,128], [128,128], [256,128]
  float *fold_b;                      // [512]: folded gate biases (128 + 128) | folded bilinear bias (256)
};

struct Arena {
  float* ctab;   // [300*num_chars] char-CNN tables
  float* cbias;  // [100]
  DabPacked dab[2];
  float* conv_tab[3];   // tap/bias tables of the whole-block conv kernel: [0] vfeat_encoder, [1] predictor's encoder, [2] tfeat_encoder (BackBone)
  TcArena tc;    // bf16 copies for the tensor-core path
};

static void carve_arena(Carver& c, const SeqpanShapes& s, Arena& a) {
  a.ctab = c.take<float>((size_t)300 * s.num_chars);
  a.cbias = c.take<float>(100);
  for (int k = 0; k < 2; ++k) {
    a.dab[k].qkv_w = c.take<float>(384 * 128); a.dab[k].qkv_b = c.take<float>(384);
    a.dab[k].tkv_w = c.take<float>(256 * 128); a.dab[k].tkv_b = c.take<float>(256);
    a.dab[k].bil_w = c.take<float>(256 * 128); a.dab[k].bil_b = c.take<float>(256);
    a.dab[k].sgsd_w = c.take<float>(128 * 128); a.dab[k].xgxd_w = c.take<float>(128 * 128);
    a.dab[k].bilgd_w = c.take<float>(256 * 128); a.dab[k].fold_b = c.take<float>(512);
  }
  for (int k = 0; k < 3; ++k) a.conv_tab[k] = c.take<float>(chain_conv_tab_floats());
  tc_carve_arena(c.base, c.off, s, a.tc);
}

#define NUM_TAPS 14
static const char* const kTapNames[NUM_TAPS] = {"text_emb", "video_affine", "venc", "tenc", "dab1_v", "dab1_t", "dab2_v",
                                                "dab2_t", "t2v", "v2t", "fuse", "fuse2", "fep_s", "fep_e"};
static const bool kTapIsText[NUM_TAPS] = {true, false, false, true, false, true, false, true, false, true, false, false, false, false};

struct Workspace {
  float *rowmask, *et, *x, *xb, *z, *o, *u, *qkv, *tkv, *sa, *xa, *s, *xx, *sg, *xg, *zin, *oz, *scva, *y, *lnr;
  float *catv, *catt, *cat2, *v2t, *fuse, *fuse2, *ph, *pa, *pqkv, *patt, *ps, *pe, *cat3, *hid;
  float* pbias;        // [B,128] per-sample bias of the concat projection (pooled half of CQConcatenate)
  float* fuse2_bf16;   // [Mv,128] bf16 copy of fuse2: x operand of the logit heads
  float* taps[NUM_TAPS];
  TcWorkspace tc;
};

static void carve_workspace(Carver& c, const SeqpanShapes& s, int B, int T, Workspace& w) {
  const size_t Mv = (size_t)B * s.vlen, Mt = (size_t)B * T, M = Mv + Mt, D = SQ_D;
  w.rowmask = c.take<float>(M);
  w.et = c.take<float>(Mt * 400);
  w.x = c.take<float>(M * D); w.xb = c.take<float>(M * D); w.z = c.take<float>(M * D);
  w.o = c.take<float>(M * D); w.u = c.take<float>(M * D);
  w.qkv = c.take<float>(M * 384); w.tkv = c.take<float>(M * 256);
  w.sa = c.take<float>(M * D); w.xa = c.take<float>(M * D); w.s = c.take<float>(M * D); w.xx = c.take<float>(M * D);
  w.sg = c.take<float>(M * D); w.xg = c.take<float>(M * D); w.zin = c.take<float>(M * D); w.oz = c.take<float>(M * D);
  w.scva = c.take<float>(M * 256); w.y = c.take<float>(M * D); w.lnr = c.take<float>(M * D);
  w.catv = c.take<float>(Mv * 512); w.catt = c.take<float>(Mt * 512); w.cat2 = c.take<float>(Mv * 256);
  w.v2t = c.take<float>(Mt * D); w.fuse = c.take<float>(Mv * D); w.fuse2 = c.take<float>(Mv * D);
  w.ph = c.take<float>(Mv * D); w.pa = c.take<float>(Mv * D); w.pqkv = c.take<float>(Mv * 384);
  w.patt = c.take<float>(Mv * D); w.ps = c.take<float>(Mv * D); w.pe = c.take<float>(Mv * D);
  w.cat3 = c.take<float>(Mv * 256); w.hid = c.take<float>(Mv * D);
  w.pbias = c.take<float>((size_t)B * D); w.fuse2_bf16 = c.take<float>((Mv + 128) * D / 2);
  for (int i = 0; i < NUM_TAPS; ++i) w.taps[i] = c.take<float>((kTapIsText[i] ? Mt : Mv) * D);
  tc_carve_workspace(c.base, c.off, s, B, T, w.tc);
}

// One captured forward: every argument that is baked into the kernel nodes (pointers, shapes) is part of the key.
struct GraphKey {
  const void* p[11];
  int B, T, C, U, side, mode;   // mode: FWD_RAW / FWD_SHARED / FWD_ENCODED (the same pointers may serve two of them)
  bool operator<(const GraphKey& o) const { return memcmp(this, &o, sizeof(GraphKey)) < 0; }
};
struct GraphEntry { cudaGraphExec_t exec; int launches; unsigned long long last_use; };

struct SeqpanHandle {
  SeqpanShapes s;
  const float* w[W_COUNT];
  Arena arena;
  int launches = 0;
  int debug = 0;
  // host mirror of the small parameter vectors (<= 1024 floats): they reach the fused tail kernels as __grid_constant__
  // kernel parameters.  Refreshed by pack_weights (seqpan_create / seqpan_repack).
  std::vector<float> hostw[W_COUNT];
  float dab_fold_host[2][512];        // host mirror of DabPacked::fold_b
  int lastB = 0, lastT = 0;
  bool last_encoded = false;          // the last forward read stored encodings (no "video_affine" tap)
  // CUDA graphs: a forward whose arguments (pointers + shapes) were seen before is replayed as ONE graph launch instead of
  // 18+ kernel launches and ~40 tensor-map encodes (static ring buffers of the eval sweep, bench.py's resident batches, and
  // in practice torch's caching allocator hand the same pointers back).  Captured on the handle's own stream (the caller's
  // may be the legacy default stream, which cannot be captured), launched on the caller's.
  // Measured on B200 (profiles/README.md, round 2): replay wins where the forward is launch-bound -- Charades shape +2.5 %
  // device-resident, +26 % end to end; ANet shape on ONE stream +5.5 % -- but two streams of replayed graphs overlap worse
  // than two streams of plain launches (ANet, 2 streams: 455 k vs 516 k queries/s), so the default is "small shapes only":
  // use_graph = 2 (auto: B * vlen <= 8192 rows), 1 = always (SEQPAN_GRAPH=1), 0 = never (SEQPAN_NO_GRAPH=1).
  int use_graph = 2;
  cudaStream_t cap_stream = nullptr;
  // The text branch (embedding + query projection: 50-CTA kernels, ~35 us) and the video affine do not depend on each other
  // (models/SeqPAN.py:56-57): the text branch runs on this side stream, forked from and joined back into the caller's stream.
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int use_side = 1;   // seqpan_set_side_stream: a pipelined sweep that runs its own host->device copy kernel turns it off
  std::map<GraphKey, GraphEntry> graphs;
  std::map<GraphKey, int> seen;
  unsigned long long tick = 0;
  void drop_graphs() {
    for (auto& kv : graphs) cudaGraphExecDestroy(kv.second.exec);
    graphs.clear();
    seen.clear();
  }
  // optional per-launch CUDA-event timing (seqpan_set_profile): tag -> events on the launching stream
  int profile = 0;
  struct Rec { char tag[48]; cudaEvent_t a, b; };
  std::vector<Rec> recs;
  std::vector<cudaEvent_t> pool;
  size_t pool_used = 0;
  cudaEvent_t ev() {
    if (pool_used == pool.size()) { cudaEvent_t e; cudaEventCreate(&e); pool.push_back(e); }
    return pool[pool_used++];
  }
  void begin(const char* tag, cudaStream_t st) {
    if (!profile) return;
    Rec r; snprintf(r.tag, sizeof(r.tag), "%.47s", tag);   // LAUNCH passes the call text: cut at 47 characters, then at "("
    const char* paren = strchr(tag, '(');
    if (paren && (size_t)(paren - tag) < sizeof(r.tag)) r.tag[paren - tag] = 0;
    r.a = ev(); r.b = ev();
    cudaEventRecord(r.a, st);
    recs.push_back(r);
  }
  void end(cudaStream_t st) { if (profile) cudaEventRecord(recs.back().b, st); }
};

static int check_shapes(const SeqpanShapes* s) {
  if (!s) return fail(SEQPAN_E_INVALID, "shapes is NULL");
  if (s->abi_version != SEQPAN_ABI_VERSION) return fail(SEQPAN_E_INVALID, "ABI version %d != %d", s->abi_version, SEQPAN_ABI_VERSION);
  if (s->variant < SEQPAN_VARIANT_SEQPAN || s->variant > SEQPAN_VARIANT_STUDENT4) return fail(SEQPAN_E_INVALID, "unknown model variant %d", s->variant);
  if (s->max_batch < 1 || s->max_batch > 768) return fail(SEQPAN_E_INVALID, "max_batch %d outside [1,768]", s->max_batch);
  if (s->vlen < 4 || s->vlen > SEQPAN_MAX_VLEN) return fail(SEQPAN_E_INVALID, "vlen %d outside [4,%d]", s->vlen, SEQPAN_MAX_VLEN);
  if (s->max_tlen < 1 || s->max_tlen > SEQPAN_MAX_TLEN || s->max_tlen > s->vlen)
    return fail(SEQPAN_E_INVALID, "max_tlen %d outside [1,min(%d,vlen)] (text shares the video position table)", s->max_tlen, SEQPAN_MAX_TLEN);
  if (s->max_clen < 4 || s->max_clen > 64) return fail(SEQPAN_E_INVALID, "max_clen %d outside [4,64]", s->max_clen);
  if (s->vdim < 4 || s->vdim % 4) return fail(SEQPAN_E_INVALID, "vdim %d must be a positive multiple of 4", s->vdim);
  if (s->num_words < 2 || s->num_chars < 1) return fail(SEQPAN_E_INVALID, "bad vocabulary sizes");
  if (s->precision != SEQPAN_PREC_FP32 && s->precision != SEQPAN_PREC_BF16 && s->precision != SEQPAN_PREC_TF32)
    return fail(SEQPAN_E_INVALID, "bad precision");
  return SEQPAN_OK;
}

extern "C" size_t seqpan_arena_bytes(const SeqpanShapes* s) {
  if (check_shapes(s) != SEQPAN_OK) return 0;
  Carver c(nullptr);
  Arena a;
  carve_arena(c, *s, a);
  return align_up(c.off, 256);
}
extern "C" size_t seqpan_workspace_bytes(const SeqpanShapes* s) {
  if (check_shapes(s) != SEQPAN_OK) return 0;
  Carver c(nullptr);
  Workspace w;
  carve_workspace(c, *s, s->max_batch, s->max_tlen, w);
  return align_up(c.off, 256);
}

#define CK(expr)                                                                                         \
  do {                                                                                                   \
    cudaError_t _e = (expr);                                                                             \
    if (_e != cudaSuccess) return fail(SEQPAN_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)
#define CHAIN(h, tag, expr)                                                          \
  do {                                                                               \
    (h)->begin(tag, st);                                                             \
    int _rc = (expr);                                                                \
    (h)->end(st);                                                                    \
    ++(h)->launches;                                                                 \
    if (_rc != SEQPAN_OK) return fail(_rc, "%s failed: %s%s", tag, chain_last_error(), tail_last_error()); \
  } while (0)
#define LAUNCH(h, expr)        \
  do {                         \
    (h)->begin(#expr, st);     \
    CK(expr);                  \
    (h)->end(st);              \
    ++(h)->launches;           \
  } while (0)

__global__ void bil_bias_kernel(const float* __restrict__ b1, const float* __restrict__ bv1, const float* __restrict__ b2,
                                const float* __restrict__ bv2, float* __restrict__ out) {
  const int i = threadIdx.x;  // 256 threads
  // BiLinear.forward applies dense_1 (with its bias) to both inputs, then adds bias_value (models/layers.py:257-263)
  out[i] = i < 128 ? 2.0f * b1[i] + bv1[i] : 2.0f * b2[i - 128] + bv2[i - 128];
}

// dst[b*L + l][:] = src[index[b]*L + l][:] -- expands the encoded rows of U unique clips to the B pairs that share them
// (SURVEY.md section 8 (f1): VisualProjection + FeatureEncoder(video) do not depend on the query, models/SeqPAN.py:57,59).
// index == nullptr: pair b reads clip b (the caller guarantees B <= U).
__global__ void __launch_bounds__(256) gather_clips_kernel(const float* __restrict__ src, const int32_t* __restrict__ index,
                                                           float* __restrict__ dst, int L, int U, long long rows) {
  const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int b = (int)(r / L), l = (int)(r % L);
  const int u = min(max(index ? __ldg(index + b) : b, 0), U - 1);
  const int lane = threadIdx.x & 31;
  reinterpret_cast<float4*>(dst + r * SQ_D)[lane] = __ldg(reinterpret_cast<const float4*>(src + ((long long)u * L + l) * SQ_D) + lane);
}

// C[i,:] = A[i,:] . B (B is [128,128] row-major), bC[i] = A[i,:] . bB + bA[i]: composition of two 128-wide projections
// y = A (B x + bB) + bA = C x + bC, evaluated once per weight set in fp32
__global__ void __launch_bounds__(128) fold_linear_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                                          const float* __restrict__ bA, const float* __restrict__ bB,
                                                          float* __restrict__ Cm, float* __restrict__ bC) {
  __shared__ float a[128];
  __shared__ float red[4];
  const int i = blockIdx.x, j = threadIdx.x;
  a[j] = A[(long long)i * 128 + j];
  __syncthreads();
  float acc = 0.f;
  for (int k = 0; k < 128; ++k) acc = fmaf(a[k], B[k * 128 + j], acc);
  Cm[(long long)i * 128 + j] = acc;
  float v = a[j] * bB[j];
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((j & 31) == 0) red[j >> 5] = v;
  __syncthreads();
  if (j == 0) bC[i] = (red[0] + red[1]) + (red[2] + red[3]) + bA[i];
}

static int pack_weights(SeqpanHandle* h, cudaStream_t st) {
  h->drop_graphs();   // captured forwards carry the old weight pointers and host-mirrored constants
  const float* const* w = h->w;
  Arena& a = h->arena;
  const float* cw[4] = {w[W_CHAR_CONV0_W], w[W_CHAR_CONV1_W], w[W_CHAR_CONV2_W], w[W_CHAR_CONV3_W]};
  CK(launch_char_table(cw, w[W_CHAR_EMB], h->s.num_chars, a.ctab, st));
  const int cb[4] = {W_CHAR_CONV0_B, W_CHAR_CONV1_B, W_CHAR_CONV2_B, W_CHAR_CONV3_B};
  const int coff[4] = {0, 10, 30, 60};
  for (int k = 0; k < 4; ++k)
    CK(cudaMemcpyAsync(a.cbias + coff[k], w[cb[k]], sizeof(float) * 10 * (k + 1), cudaMemcpyDeviceToDevice, st));
  const int base[2] = {W_DAB1_LN1_W, W_DAB2_LN1_W};
  const bool has_dab = h->s.variant != SEQPAN_VARIANT_BASEFAST && h->s.variant != SEQPAN_VARIANT_STUDENT4;   // BaseFast never calls its DualAttentionBlocks
  const int enc_layers = (h->s.variant == SEQPAN_VARIANT_BASEFAST || h->s.variant == SEQPAN_VARIANT_MULTITEACHER) ? 2 : 4;   // layers of vfeat_encoder
  const bool has_tenc = h->s.variant == SEQPAN_VARIANT_BACKBONE;      // the text's own FeatureEncoder
  for (int k = 0; k < (has_dab ? 2 : 0); ++k) {
    const int d = base[k] - W_DAB1_LN1_W;
    auto cp = [&](float* dst, int id, size_t n) {
      return cudaMemcpyAsync(dst, w[id + d], sizeof(float) * n, cudaMemcpyDeviceToDevice, st);
    };
    const size_t DD = 128 * 128;
    CK(cp(a.dab[k].qkv_w, W_DAB1_QUERY_W, DD)); CK(cp(a.dab[k].qkv_w + DD, W_DAB1_FKEY_W, DD));
    CK(cp(a.dab[k].qkv_w + 2 * DD, W_DAB1_FVALUE_W, DD));
    CK(cp(a.dab[k].qkv_b, W_DAB1_QUERY_B, 128)); CK(cp(a.dab[k].qkv_b + 128, W_DAB1_FKEY_B, 128));
    CK(cp(a.dab[k].qkv_b + 256, W_DAB1_FVALUE_B, 128));
    CK(cp(a.dab[k].tkv_w, W_DAB1_TKEY_W, DD)); CK(cp(a.dab[k].tkv_w + DD, W_DAB1_TVALUE_W, DD));
    CK(cp(a.dab[k].tkv_b, W_DAB1_TKEY_B, 128)); CK(cp(a.dab[k].tkv_b + 128, W_DAB1_TVALUE_B, 128));
    CK(cp(a.dab[k].bil_w, W_DAB1_BIL1_W, DD)); CK(cp(a.dab[k].bil_w + DD, W_DAB1_BIL2_W, DD));
    bil_bias_kernel<<<1, 256, 0, st>>>(w[W_DAB1_BIL1_B + d], w[W_DAB1_BIL1_BV + d], w[W_DAB1_BIL2_B + d],
                                       w[W_DAB1_BIL2_BV + d], a.dab[k].bil_b);
    CK(cudaGetLastError());
    fold_linear_kernel<<<128, 128, 0, st>>>(w[W_DAB1_SGATE_W + d], w[W_DAB1_SDENSE_W + d], w[W_DAB1_SGATE_B + d],
                                            w[W_DAB1_SDENSE_B + d], a.dab[k].sgsd_w, a.dab[k].fold_b);
    fold_linear_kernel<<<128, 128, 0, st>>>(w[W_DAB1_XGATE_W + d], w[W_DAB1_XDENSE_W + d], w[W_DAB1_XGATE_B + d],
                                            w[W_DAB1_XDENSE_B + d], a.dab[k].xgxd_w, a.dab[k].fold_b + 128);
    fold_linear_kernel<<<256, 128, 0, st>>>(a.dab[k].bil_w, w[W_DAB1_GUIDED_W + d], a.dab[k].bil_b, w[W_DAB1_GUIDED_B + d],
                                            a.dab[k].bilgd_w, a.dab[k].fold_b + 256);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->dab_fold_host[k], a.dab[k].fold_b, sizeof(float) * 512, cudaMemcpyDeviceToHost, st));
  }
  for (int i = 0; i < W_COUNT; ++i) {
    const int64_t n = seqpan_weight_numel(&h->s, i);
    h->hostw[i].clear();
    if (n > 0 && n <= 1024) {
      h->hostw[i].resize((size_t)n);
      CK(cudaMemcpyAsync(h->hostw[i].data(), w[i], sizeof(float) * n, cudaMemcpyDeviceToHost, st));
    }
  }
  CK(cudaStreamSynchronize(st));
  if (h->s.precision == SEQPAN_PREC_BF16) {
    const int encs[3] = {W_ENC_POS, W_PRED_POS, W_TENC_POS};
    for (int e = 0; e < (has_tenc ? 3 : 2); ++e) {
      const float *g4[4], *b4[4], *d4[4], *bias4[4];
      for (int i = 0; i < 4; ++i) {
        const int li = (e == 0 && i >= enc_layers) ? 0 : i;   // absent layers: any valid pointers (their table rows are never read)
        const int dwid = encs[e] + 1 + 5 * li;   // DWi, PWi_W, PWi_B, LNi_W, LNi_B
        d4[i] = w[dwid]; bias4[i] = w[dwid + 2]; g4[i] = w[dwid + 3]; b4[i] = w[dwid + 4];
      }
      int rc = chain_conv_tables(g4, b4, d4, bias4, a.conv_tab[e], st);
      if (rc != SEQPAN_OK) return fail(rc, "conv block table packing failed: %s", chain_last_error());
    }
    const float* src[TC_NUM_SLOTS] = {};
    for (int i = 0; i < 4; ++i) {
      src[TC_ENC_PW0 + i] = i < enc_layers ? w[W_ENC_PW0_W + 5 * i] : nullptr;   // nullptr: slot not used by this variant
      src[TC_PRED_PW0 + i] = w[W_PRED_PW0_W + 5 * i];
      src[TC_TENC_PW0 + i] = has_tenc ? w[W_TENC_PW0_W + 5 * i] : nullptr;
    }
    for (int k = 0; k < (has_dab ? 2 : 0); ++k) {
      const int d = base[k] - W_DAB1_LN1_W, ts = TC_DAB0 + k * TC_DAB_STRIDE;
      src[ts + TC_DAB_QKV] = a.dab[k].qkv_w; src[ts + TC_DAB_TKV] = a.dab[k].tkv_w; src[ts + TC_DAB_BIL] = a.dab[k].bil_w;
      src[ts + TC_DAB_SDENSE] = w[W_DAB1_SDENSE_W + d]; src[ts + TC_DAB_XDENSE] = w[W_DAB1_XDENSE_W + d];
      src[ts + TC_DAB_D1] = w[W_DAB1_D1_W + d]; src[ts + TC_DAB_D2] = w[W_DAB1_D2_W + d];
      src[ts + TC_DAB_SGSD] = a.dab[k].sgsd_w; src[ts + TC_DAB_XGXD] = a.dab[k].xgxd_w; src[ts + TC_DAB_BILGD] = a.dab[k].bilgd_w;
    }
    src[TC_Q2V_LIN] = w[W_Q2V_LIN_W]; src[TC_V2Q_LIN] = w[W_V2Q_LIN_W]; src[TC_CAT] = w[W_CAT_W];
    src[TC_INPROJ] = w[W_INPROJ_W]; src[TC_OUTPROJ] = w[W_OUTPROJ_W]; src[TC_PRED_DENSE] = w[W_PRED_DENSE_W];
    src[TC_START_HID] = w[W_START_HID_W]; src[TC_END_HID] = w[W_END_HID_W];
    int rc = tc_pack(h->s, src, a.tc, st);
    if (rc != SEQPAN_OK) return fail(rc, "tensor-core weight packing failed: %s", tc_last_error());
  }
  return SEQPAN_OK;
}

static int bind_weights(SeqpanHandle* h, const float* const* weights_host) {
  if (!weights_host) return fail(SEQPAN_E_INVALID, "weights_host is NULL");
  for (int i = 0; i < W_COUNT; ++i) {
    const int64_t n = seqpan_weight_numel(&h->s, i);
    if (n > 0 && !weights_host[i]) return fail(SEQPAN_E_INVALID, "weight '%s' is NULL", kWeightNames[i]);
    h->w[i] = weights_host[i];
  }
  return SEQPAN_OK;
}

extern "C" int seqpan_create(const SeqpanShapes* shapes, const float* const* weights_host, void* arena,
                             size_t arena_bytes, void* stream, SeqpanHandle** out) {
  if (!out) return fail(SEQPAN_E_INVALID, "out is NULL");
  *out = nullptr;
  int rc = check_shapes(shapes);
  if (rc != SEQPAN_OK) return rc;
  if (!seqpan_device_ok()) return fail(SEQPAN_E_NODEVICE, "no sm_100 CUDA device: this library has no CPU fallback");
  if (!arena || ((uintptr_t)arena & 255)) return fail(SEQPAN_E_WORKSPACE, "arena must be a 256-byte aligned device pointer");
  if (arena_bytes < seqpan_arena_bytes(shapes)) return fail(SEQPAN_E_WORKSPACE, "arena too small: %zu < %zu", arena_bytes, seqpan_arena_bytes(shapes));
  SeqpanHandle* h = new (std::nothrow) SeqpanHandle();
  if (!h) return fail(SEQPAN_E_INVALID, "out of host memory");
  h->s = *shapes;
  sq_env_refresh();   // the only place the SEQPAN_* switches are read: once per handle, never on the forward path
  h->use_graph = sq_env().no_graph ? 0 : (sq_env().force_graph ? 1 : 2);
  if (!sq_env().no_side_stream && cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking) == cudaSuccess) {
    if (cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess) {
      cudaStreamDestroy(h->side);
      h->side = nullptr;
    }
  }
  cudaGetLastError();
  Carver c(arena);
  carve_arena(c, h->s, h->arena);
  rc = bind_weights(h, weights_host);
  if (rc == SEQPAN_OK) rc = pack_weights(h, (cudaStream_t)stream);
  if (rc != SEQPAN_OK) {
    delete h;
    return rc;
  }
  *out = h;
  return SEQPAN_OK;
}

extern "C" int seqpan_repack(SeqpanHandle* h, const float* const* weights_host, void* stream) {
  if (!h) return fail(SEQPAN_E_INVALID, "handle is NULL");
  int rc = bind_weights(h, weights_host);
  if (rc != SEQPAN_OK) return rc;
  return pack_weights(h, (cudaStream_t)stream);
}

extern "C" void seqpan_destroy(SeqpanHandle* h) {
  if (!h) return;
  h->drop_graphs();
  if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
  if (h->side) { cudaStreamDestroy(h->side); cudaEventDestroy(h->ev_fork); cudaEventDestroy(h->ev_join); }
  for (cudaEvent_t e : h->pool) cudaEventDestroy(e);
  delete h;
}
extern "C" int seqpan_last_launch_count(const SeqpanHandle* h) { return h ? h->launches : 0; }
extern "C" int seqpan_set_debug(SeqpanHandle* h, int on) {
  if (!h) return fail(SEQPAN_E_INVALID, "handle is NULL");
  h->debug = on;
  return SEQPAN_OK;
}

extern "C" int seqpan_set_side_stream(SeqpanHandle* h, int on) {
  if (!h) return fail(SEQPAN_E_INVALID, "handle is NULL");
  h->use_side = on ? 1 : 0;                              // part of the capture key: both variants of a forward can be cached
  return SEQPAN_OK;
}

extern "C" int seqpan_set_profile(SeqpanHandle* h, int on) {
  if (!h) return fail(SEQPAN_E_INVALID, "handle is NULL");
  h->profile = on;
  h->recs.clear();
  h->pool_used = 0;
  return SEQPAN_OK;
}

// Writes "tag count total_ms\n" lines for every launch tag recorded since seqpan_set_profile(h, 1); synchronises.
extern "C" int seqpan_profile_summary(SeqpanHandle* h, char* buf, size_t cap) {
  if (!h || !buf || cap == 0) return fail(SEQPAN_E_INVALID, "bad argument");
  CK(cudaDeviceSynchronize());
  std::map<std::string, std::pair<int, double>> agg;
  for (auto& r : h->recs) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) continue;
    auto& e = agg[r.tag];
    e.first += 1;
    e.second += ms;
  }
  size_t off = 0;
  buf[0] = 0;
  for (auto& kv : agg) {
    int n = snprintf(buf + off, cap - off, "%s %d %.6f\n", kv.first.c_str(), kv.second.first, kv.second.second);
    if (n < 0 || (size_t)n >= cap - off) break;
    off += n;
  }
  h->recs.clear();
  h->pool_used = 0;
  return SEQPAN_OK;
}

// ---- forward -----------------------------------------------------------------------------------------
enum { FWD_RAW = 0, FWD_SHARED = 1, FWD_ENCODED = 2 };   // what `vfeat` of forward_impl holds: [B,L,V], [U,L,V] or [U,L,128]

namespace {

struct Fwd {
  SeqpanHandle* h;
  Workspace ws;
  cudaStream_t st;
  int B, L, T, C;
  long long Mv, Mt, M;
  bool tc;             // SEQPAN_PREC_BF16: the fused tcgen05 chain kernels
  bool tf32 = false;   // SEQPAN_PREC_TF32: the fp32 schedule with every projection on tcgen05 kind::tf32

  // y = act(x.w^T + b) (+res).  tf32 mode: kind::tf32 wherever the shape allows it.  bf16 mode reaches this only from the
  // CUDA-core CQAttention path (L > 128): its two K = 512 cqa_linear projections read the fp32 concat once by TMA on
  // kind::tf32, with no fp32 -> bf16 staging pass.
  int linear(const float* x, int ldx, const float* w, const float* b, const float* res, float* y, int ldy, long long M_,
             int N, int K, bool relu) {
    if (tc || (tf32 && N % 128 == 0 && !(K & 3) && !(ldx & 3))) {
      char tag[48];
      if (tc) snprintf(tag, sizeof(tag), "tc_linear_tf32_cqa");
      else snprintf(tag, sizeof(tag), "tc_linear_tf32_N%d_K%d", N, K);
      h->begin(tag, st);
      int rc = tc_linear_tf32(x, ldx, w, b, res, y, ldy, M_, N, K, relu, st);
      h->end(st);
      if (rc != SEQPAN_OK) return fail(rc, "tc_linear_tf32 failed: %s", tc_last_error());
      ++h->launches;
      return SEQPAN_OK;
    }
    LinearArgs a{};
    a.x[0] = x; a.w[0] = w; a.bias[0] = b; a.res[0] = res; a.y[0] = y;
    a.M = M_; a.N = N; a.K = K; a.ldx = ldx; a.ldw = K; a.ldy = ldy; a.ldr = ldy; a.relu = relu; a.count = 1;
    char tag[48];
    snprintf(tag, sizeof(tag), "linear_f32_N%d_K%d", N, K);
    h->begin(tag, st);
    CK(launch_linear_f32(a, st));
    h->end(st);
    ++h->launches;
    return SEQPAN_OK;
  }
  // VisualProjection (models/layers.py:118-123): Conv1D(vdim -> 128) + LayerNorm(1e-6).  bf16 / tf32 mode: one launch, the
  // fp32 features are read once by TMA (kind::tf32) and the LayerNorm rides in the epilogue; `tmp` is the pre-LN buffer in fp32 mode.
  int video_affine(const float* x, long long rows, float* tmp, float* y) {
    const float* const* w = h->w;
    const SeqpanShapes& s = h->s;
    if (tf32 || tc) {
      h->begin("tc_linear_tf32_video+ln", st);
      int rc = tc_linear_tf32(x, s.vdim, w[W_VIDEO_W], w[W_VIDEO_B], nullptr, y, SQ_D, rows, SQ_D, s.vdim, false, st, w[W_VLN_W],
                              w[W_VLN_B], 1e-6f);
      h->end(st);
      if (rc != SEQPAN_OK) return fail(rc, "tc_linear_tf32 (+LayerNorm) failed: %s", tc_last_error());
      ++h->launches;
      return SEQPAN_OK;
    }
    int rc = linear(x, s.vdim, w[W_VIDEO_W], w[W_VIDEO_B], nullptr, tmp, SQ_D, rows, SQ_D, s.vdim, false);
    return rc ? rc : ln(tmp, rows, W_VLN_W, 1e-6f, y);
  }
  int linear2(const float* x0, const float* w0, const float* b0, float* y0, const float* x1, const float* w1,
              const float* b1, float* y1, long long M_) {
    if (tf32) {
      int rc = linear(x0, SQ_D, w0, b0, nullptr, y0, SQ_D, M_, SQ_D, SQ_D, false);
      if (rc != SEQPAN_OK) return rc;
      return linear(x1, SQ_D, w1, b1, nullptr, y1, SQ_D, M_, SQ_D, SQ_D, false);
    }
    LinearArgs a{};
    a.x[0] = x0; a.w[0] = w0; a.bias[0] = b0; a.y[0] = y0;
    a.x[1] = x1; a.w[1] = w1; a.bias[1] = b1; a.y[1] = y1;
    a.M = M_; a.N = SQ_D; a.K = SQ_D; a.ldx = SQ_D; a.ldw = SQ_D; a.ldy = SQ_D; a.ldr = SQ_D; a.relu = 0; a.count = 2;
    LAUNCH(h, launch_linear_f32(a, st));
    return SEQPAN_OK;
  }
  int ln(const float* x, long long M_, int wid, float eps, float* y, int ldy = SQ_D, const float* copy_src = nullptr,
         float* copy_dst = nullptr) {
    LAUNCH(h, launch_layernorm(x, SQ_D, M_, h->w[wid], h->w[wid + 1], eps, y, ldy, nullptr, nullptr, nullptr, 0, copy_src,
                               copy_dst, 256, st));
    return SEQPAN_OK;
  }
  int tap(int idx, const float* src, int ld) {
    if (!h->debug) return SEQPAN_OK;
    const long long rows = kTapIsText[idx] ? Mt : Mv;
    CK(cudaMemcpy2DAsync(ws.taps[idx], SQ_D * sizeof(float), src, (size_t)ld * sizeof(float), SQ_D * sizeof(float),
                         (size_t)rows, cudaMemcpyDeviceToDevice, st));
    return SEQPAN_OK;
  }

  // FeatureEncoder conv block (models/layers.py:139-148, 396-399): x0 = in + pos; 4x { x += ReLU(PW(DW(LN(x)))) }.
  // `enc` is the first weight id of the ENCODER() group; the result is left in `xout` (must differ from `in`).
  // `tail` (optional, bf16 mode): LayerNorm + projections of the block's consumer, fused behind the last layer.
  int conv_block(const float* in, float* xout, int enc, const Segs& sg, long long rows, int tc_slot0,
                 const ChainProjTail* tail = nullptr) {
    // the shared FeatureEncoder of BaseFast has 2 layers (models/BaseFast.py:27); every other conv block has 4
    const int nl = (enc == W_ENC_POS && (h->s.variant == SEQPAN_VARIANT_BASEFAST || h->s.variant == SEQPAN_VARIANT_MULTITEACHER)) ? 2 : 4;
    float* tab = h->arena.conv_tab[enc == W_ENC_POS ? 0 : (enc == W_PRED_POS ? 1 : 2)];
    if (tc) {
      CHAIN(h, tail ? "chain_conv_block+proj" : "chain_conv_block",
            chain_conv_block(h->arena.tc, tc_slot0, in, h->w[enc], xout, tab, sg.nseg[0],
                             sg.len[0], sg.nseg[1], sg.nseg[1] > 0 ? sg.len[1] : 0, st, tail, nl));
      return SEQPAN_OK;
    }
    for (int i = 0; i < nl; ++i) {
      const int dwid = enc + 1 + 5 * i;  // DWi, PWi_W, PWi_B, LNi_W, LNi_B
      LAUNCH(h, launch_ln_dwconv(i == 0 ? in : xout, i == 0 ? h->w[enc] : nullptr, i == 0 ? xout : nullptr,
                                 h->w[dwid + 3], h->w[dwid + 4], 1e-6f, h->w[dwid], ws.z, sg, st));
      int rc = linear(ws.z, SQ_D, h->w[dwid + 1], h->w[dwid + 2], xout, xout, SQ_D, rows, SQ_D, SQ_D, true);
      if (rc != SEQPAN_OK) return rc;
    }
    return SEQPAN_OK;
  }

  // DualAttentionBlock on the joint rows, both directions at once (models/layers.py:281-297, 336-381)
  int dual_block(int k, float* cur, bool proj_done = false) {
    const int d = k == 0 ? 0 : (W_DAB2_LN1_W - W_DAB1_LN1_W);
    const DabPacked& p = h->arena.dab[k];
    const float* const* w = h->w;
    const int ts = TC_DAB0 + k * TC_DAB_STRIDE;
    int rc;
    const bool tc_att = tc && attn_dual_tc_supported(L, T);
    if (tc_att) {
      if (!proj_done)
        CHAIN(h, "chain_proj_ln", chain_proj_ln(h->arena.tc, ts + TC_DAB_QKV, ts + TC_DAB_TKV, cur, M, 1e-6f, w[W_DAB1_LN1_W + d],
                                                w[W_DAB1_LN1_B + d], w[W_DAB1_LNT_W + d], w[W_DAB1_LNT_B + d],
                                                (float*)ws.tc.qkv_bf16, p.qkv_b, (float*)ws.tc.tkv_bf16, p.tkv_b, st, nullptr, 0,
                                                0, nullptr, true));
      CHAIN(h, "attn_dual_tc", attn_dual_tc(ws.tc.qkv_bf16, ws.tc.tkv_bf16, vmask, tmask, ws.tc.sa_bf16, ws.tc.xa_bf16, B, L, T, st));
    } else if (tc) {
      CHAIN(h, "chain_proj_ln", chain_proj_ln(h->arena.tc, ts + TC_DAB_QKV, ts + TC_DAB_TKV, cur, M, 1e-6f, w[W_DAB1_LN1_W + d],
                                              w[W_DAB1_LN1_B + d], w[W_DAB1_LNT_W + d], w[W_DAB1_LNT_B + d], ws.qkv, p.qkv_b,
                                              ws.tkv, p.tkv_b, st));
    } else {
      LAUNCH(h, launch_layernorm(cur, SQ_D, M, w[W_DAB1_LN1_W + d], w[W_DAB1_LN1_B + d], 1e-6f, ws.o, SQ_D,
                                 w[W_DAB1_LNT_W + d], w[W_DAB1_LNT_B + d], ws.u, SQ_D, nullptr, nullptr, 0, st));
      if ((rc = linear(ws.o, SQ_D, p.qkv_w, p.qkv_b, nullptr, ws.qkv, 384, M, 384, SQ_D, false))) return rc;
      if ((rc = linear(ws.u, SQ_D, p.tkv_w, p.tkv_b, nullptr, ws.tkv, 256, M, 256, SQ_D, false))) return rc;
    }
    if (!tc_att) {
      DualAttnArgs aa{ws.qkv, ws.tkv, vmask, tmask, ws.sa, ws.xa, B, L, T, tc ? ws.tc.sa_bf16 : nullptr,
                      tc ? ws.tc.xa_bf16 : nullptr};
      LAUNCH(h, launch_dual_attention(aa, st));
    }
    if (tc) {
      auto hv = [&](int id) { return h->hostw[id + d].data(); };
      // gate / bilinear biases with the folded projections' contributions (DabPacked::fold_b, mirrored at pack time)
      const float* fb = h->dab_fold_host[k];
      const float* hostv[10] = {hv(W_DAB1_SDENSE_B), hv(W_DAB1_XDENSE_B), fb, fb + 128, hv(W_DAB1_GUIDED_B),
                                fb + 256, hv(W_DAB1_D1_B), hv(W_DAB1_D2_B), hv(W_DAB1_LN2_W), hv(W_DAB1_LN2_B)};
      h->begin("chain_dab_post", st);
      rc = chain_dab_post(h->arena.tc, k, ws.tc.sa_bf16, ws.tc.xa_bf16, cur, cur, vmask, tmask, Mv, M, hostv, w[W_DAB1_LN1_W + d],
                          w[W_DAB1_LN1_B + d], st);
      h->end(st);
      ++h->launches;
      if (rc != SEQPAN_OK) return fail(rc, "chain_dab_post failed: %s", tail_last_error());
      return SEQPAN_OK;
    }
    if ((rc = linear2(ws.sa, w[W_DAB1_SDENSE_W + d], w[W_DAB1_SDENSE_B + d], ws.s, ws.xa, w[W_DAB1_XDENSE_W + d],
                      w[W_DAB1_XDENSE_B + d], ws.xx, M))) return rc;
    if ((rc = linear2(ws.s, w[W_DAB1_SGATE_W + d], w[W_DAB1_SGATE_B + d], ws.sg, ws.xx, w[W_DAB1_XGATE_W + d],
                      w[W_DAB1_XGATE_B + d], ws.xg, M))) return rc;
    LAUNCH(h, launch_gate_combine(ws.sg, ws.xx, ws.xg, ws.s, ws.zin, M * SQ_D / 4, st));
    // W1.o + W1.z = W1.(o + z): the guided_dense epilogue adds o, one 256-wide GEMM yields scores|values
    if ((rc = linear(ws.zin, SQ_D, w[W_DAB1_GUIDED_W + d], w[W_DAB1_GUIDED_B + d], ws.o, ws.oz, SQ_D, M, SQ_D, SQ_D, false))) return rc;
    if ((rc = linear(ws.oz, SQ_D, p.bil_w, p.bil_b, nullptr, ws.scva, 256, M, 256, SQ_D, false))) return rc;
    LAUNCH(h, launch_sigmoid_gate(ws.scva, ws.rowmask, ws.y, M, st));
    if ((rc = linear(ws.y, SQ_D, w[W_DAB1_D1_W + d], w[W_DAB1_D1_B + d], cur, cur, SQ_D, M, SQ_D, SQ_D, false))) return rc;
    if ((rc = ln(cur, M, W_DAB1_LN2_W + d, 1e-6f, ws.lnr))) return rc;
    return linear(ws.lnr, SQ_D, w[W_DAB1_D2_W + d], w[W_DAB1_D2_B + d], cur, cur, SQ_D, M, SQ_D, SQ_D, false);
  }

  // FeatureEncoderPredict (models/layers.py:626-639); result in `out`
  // bf16 mode: the start/end logit head `head` rides behind the FEP tail (chain_fep_head); fp32 / tf32 mode ignore it
  struct HeadArgs { int slot; int ln_w, ln_b, hid_b, dense_w, dense_b; float* logits; };
  int fep(const float* in, float* out, const HeadArgs* head = nullptr) {
    const float* const* w = h->w;
    Segs sg{{0, 0}, {B, 0}, {L, 0}};
    int rc;
    void* hb[3] = {ws.tc.hb_q, ws.tc.hb_k, ws.tc.hb_v};
    const bool tc_batt = tc && B <= 256;   // in_proj rides behind the conv block as head-blocked q/k/v for attn_batch_tc
    ChainProjTail tl{};
    tl.slotA = TC_INPROJ; tl.slotB = -1; tl.eps = 1e-5f; tl.gA = w[W_PRED_LNA_W]; tl.bA = w[W_PRED_LNA_B];
    tl.biasA = w[W_INPROJ_B]; tl.hb = hb; tl.hbL = L; tl.hbB = B; tl.hb_mask = vmask;
    if ((rc = conv_block(in, ws.ph, W_PRED_POS, sg, Mv, TC_PRED_PW0, tc_batt ? &tl : nullptr))) return rc;
    if (tc) {
      if (tc_batt) {
        CHAIN(h, "attn_batch_tc", attn_batch_tc(ws.tc.hb_q, ws.tc.hb_k, ws.tc.hb_v, vmask, ws.tc.sa_bf16, B, L, st));
      } else {
        CHAIN(h, "chain_proj_ln", chain_proj_ln(h->arena.tc, TC_INPROJ, -1, ws.ph, Mv, 1e-5f, w[W_PRED_LNA_W], w[W_PRED_LNA_B],
                                                nullptr, nullptr, ws.pqkv, w[W_INPROJ_B], nullptr, nullptr, st));
        LAUNCH(h, launch_batch_attention(ws.pqkv, vmask, nullptr, ws.tc.sa_bf16, B, L, st));
      }
      auto hv = [&](int id) { return h->hostw[id].data(); };
      const float* hostv[9] = {hv(W_OUTPROJ_B), hv(W_PRED_LNB_W), hv(W_PRED_LNB_B), hv(W_PRED_DENSE_B), hv(head->ln_w),
                               hv(head->ln_b), hv(head->hid_b), hv(head->dense_w), hv(head->dense_b)};
      CHAIN(h, "chain_fep_head", chain_fep_head(h->arena.tc, head->slot, ws.tc.sa_bf16, ws.fuse2_bf16, ws.ph, out, Mv, hostv,
                                                head->logits, st));
      return SEQPAN_OK;
    }
    if ((rc = ln(ws.ph, Mv, W_PRED_LNA_W, 1e-5f, ws.pa))) return rc;
    if ((rc = linear(ws.pa, SQ_D, w[W_INPROJ_W], w[W_INPROJ_B], nullptr, ws.pqkv, 384, Mv, 384, SQ_D, false))) return rc;
    LAUNCH(h, launch_batch_attention(ws.pqkv, vmask, ws.patt, nullptr, B, L, st));
    if ((rc = linear(ws.patt, SQ_D, w[W_OUTPROJ_W], w[W_OUTPROJ_B], ws.ph, ws.ph, SQ_D, Mv, SQ_D, SQ_D, false))) return rc;
    if ((rc = ln(ws.ph, Mv, W_PRED_LNB_W, 1e-5f, ws.pa))) return rc;
    return linear(ws.pa, SQ_D, w[W_PRED_DENSE_W], w[W_PRED_DENSE_B], ws.ph, out, SQ_D, Mv, SQ_D, SQ_D, false);
  }

  const int64_t* word_ids; const int64_t* char_ids; const float* vfeat; const float* vmask; const float* tmask;
  const float* gumbel; float* slogits; float* elogits; float* match_score;
  const int32_t* video_index = nullptr;   // != nullptr: vfeat (or venc) holds U unique clips, video_index[b] = clip of pair b
  const float* venc = nullptr;            // != nullptr: stored encodings [U,L,128] of seqpan_encode_videos instead of vfeat
  int U = 0;

  int run() {
    const float* const* w = h->w;
    const SeqpanShapes& s = h->s;
    int rc;
    if (!tc)   // the fused DualAttentionBlock chain reads vmask / tmask in place
      LAUNCH(h, launch_build_rowmask(vmask, Mv, tmask, Mt, ws.rowmask, st));
    // text embedding (models/layers.py:87-93) -> rows [Mv, M) of x; on the side stream, concurrently with the video affine
    cudaStream_t main_st = st;
    const bool fork = h->side && h->use_side && !h->profile && !h->debug && !video_index && !venc;
    if (fork) {
      CK(cudaEventRecord(h->ev_fork, main_st));
      CK(cudaStreamWaitEvent(h->side, h->ev_fork, 0));
      st = h->side;
    }
    LAUNCH(h, launch_embed_text(word_ids, char_ids, Mt, C, w[W_WORD_PAD], w[W_WORD_UNK], w[W_WORD_GLOVE],
                                s.pretrained_words ? nullptr : w[W_WORD_TABLE], s.num_words, s.num_chars, h->arena.ctab,
                                h->arena.cbias, ws.et, st));
    float* xt = ws.x + Mv * SQ_D;
    float* zt = ws.z + Mv * SQ_D;
    if (tf32 || tc) {   // Conv1D(400 -> 128) on kind::tf32 straight from the fp32 concat + fused LayerNorm
      h->begin("tc_linear_tf32_query+ln", st);
      rc = tc_linear_tf32(ws.et, 400, w[W_QUERY_W], w[W_QUERY_B], nullptr, xt, SQ_D, Mt, SQ_D, 400, false, st, w[W_QLN_W], w[W_QLN_B], 1e-6f);
      h->end(st);
      if (rc != SEQPAN_OK) return fail(rc, "tc_linear_tf32 (query + LayerNorm) failed: %s", tc_last_error());
      ++h->launches;
    } else {
      if ((rc = linear(ws.et, 400, w[W_QUERY_W], w[W_QUERY_B], nullptr, zt, SQ_D, Mt, SQ_D, 400, false))) return rc;
      if ((rc = ln(zt, Mt, W_QLN_W, 1e-6f, xt))) return rc;
    }
    if (fork) {
      CK(cudaEventRecord(h->ev_join, h->side));
      st = main_st;
    }
    if ((rc = tap(0, xt, SQ_D))) return rc;
    if (venc) return run_encoded(venc, xt);
    if (video_index) return run_shared_video(xt);
    // video affine (models/layers.py:118-123) -> rows [0, Mv)
    if ((rc = video_affine(vfeat, Mv, ws.z, ws.x))) return rc;
    if (fork) CK(cudaStreamWaitEvent(st, h->ev_join, 0));
    if ((rc = tap(1, ws.x, SQ_D))) return rc;
    // shared FeatureEncoder on video and text (models/SeqPAN.py:59-60)
    Segs joint{{0, Mv}, {B, B}, {L, T}};
    // the first DualAttentionBlock's LN1 -> q|fk|fv and LNt -> tk|tv projections ride behind the encoder's last layer
    const bool has_dab = s.variant != SEQPAN_VARIANT_BASEFAST && s.variant != SEQPAN_VARIANT_STUDENT4;
    const bool tc_att0 = has_dab && tc && attn_dual_tc_supported(L, T);
    ChainProjTail dt{};
    dt.slotA = TC_DAB0 + TC_DAB_QKV; dt.slotB = TC_DAB0 + TC_DAB_TKV; dt.eps = 1e-6f;
    dt.gA = w[W_DAB1_LN1_W]; dt.bA = w[W_DAB1_LN1_B]; dt.gB = w[W_DAB1_LNT_W]; dt.bB = w[W_DAB1_LNT_B];
    dt.biasA = h->arena.dab[0].qkv_b; dt.biasB = h->arena.dab[0].tkv_b; dt.outA = ws.tc.qkv_bf16; dt.outB = ws.tc.tkv_bf16;
    if (s.variant == SEQPAN_VARIANT_BACKBONE) {
      // models/BackBone.py:48-49: vfeat_encoder on the video rows, the text's own tfeat_encoder on the text rows; the fused
      // LN + projection tail indexes its outputs by the rows of the call, so the text call gets offset output pointers
      Segs vs{{0, 0}, {B, 0}, {L, 0}}, ts{{0, 0}, {B, 0}, {T, 0}};
      ChainProjTail dtt = dt;
      dtt.outA = reinterpret_cast<char*>(dt.outA) + Mv * 384 * 2;
      dtt.outB = reinterpret_cast<char*>(dt.outB) + Mv * 256 * 2;
      if ((rc = conv_block(ws.x, ws.xb, W_ENC_POS, vs, Mv, TC_ENC_PW0, tc_att0 ? &dt : nullptr))) return rc;
      if ((rc = conv_block(xt, ws.xb + Mv * SQ_D, W_TENC_POS, ts, Mt, TC_TENC_PW0, tc_att0 ? &dtt : nullptr))) return rc;
      return run_after_encoder(tc_att0);
    }
    if ((rc = conv_block(ws.x, ws.xb, W_ENC_POS, joint, M, TC_ENC_PW0, tc_att0 ? &dt : nullptr))) return rc;
    return run_after_encoder(tc_att0);
  }

  // The query-independent video branch of `nclips` clips (models/SeqPAN.py:57,59): VisualProjection -> `aff`, then the video
  // half of the shared FeatureEncoder -> `out` (`tmp`: pre-LayerNorm rows of the fp32 mode).  One segment per clip and
  // row-local arithmetic: a clip's rows do not depend on the other clips of the call (seqpan_encode_videos relies on it).
  int encode_clips(const float* vf, int nclips, float* tmp, float* aff, float* out) {
    const long long Mu = (long long)nclips * L;
    int rc;
    if ((rc = video_affine(vf, Mu, tmp, aff))) return rc;
    Segs clips{{0, 0}, {nclips, 0}, {L, 0}};
    return conv_block(aff, out, W_ENC_POS, clips, Mu, TC_ENC_PW0);
  }
  int gather(const float* src, float* dst) {
    h->begin("gather_clips", st);
    gather_clips_kernel<<<(unsigned)((Mv + 7) / 8), 256, 0, st>>>(src, video_index, dst, L, U, Mv);
    h->end(st);
    ++h->launches;
    CK(cudaGetLastError());
    return SEQPAN_OK;
  }

  // Query-independent video branch once per UNIQUE clip (SURVEY.md section 8 (f1)): the U clips are encoded into the
  // workspace, then the query half runs as on stored encodings.  Same kernels, same per-row arithmetic as the plain path.
  int run_shared_video(float* xt) {
    int rc;
    if ((rc = encode_clips(vfeat, U, ws.o, ws.u, ws.s))) return rc;
    if (h->debug) {
      if ((rc = gather(ws.u, ws.x)) || (rc = tap(1, ws.x, SQ_D))) return rc;
    }
    return run_encoded(ws.s, xt);
  }

  // The query half on encoded clip rows `enc` [U,L,128]: expand them to the B pairs, run the text half of the encoder
  // (BackBone: its own tfeat_encoder), then everything behind the encoder.
  int run_encoded(const float* enc, float* xt) {
    int rc;
    if ((rc = gather(enc, ws.xb))) return rc;
    Segs text{{0, 0}, {B, 0}, {T, 0}};
    const bool own_text = h->s.variant == SEQPAN_VARIANT_BACKBONE;
    if ((rc = conv_block(xt, ws.xb + Mv * SQ_D, own_text ? W_TENC_POS : W_ENC_POS, text, Mt, own_text ? TC_TENC_PW0 : TC_ENC_PW0))) return rc;
    return run_after_encoder(false);
  }

  int run_after_encoder(bool dab0_proj_done) {
    const float* const* w = h->w;
    int rc;
    float* cur = ws.xb;
    if ((rc = tap(2, cur, SQ_D)) || (rc = tap(3, cur + Mv * SQ_D, SQ_D))) return rc;
    for (int k = 0; k < ((h->s.variant != SEQPAN_VARIANT_BASEFAST && h->s.variant != SEQPAN_VARIANT_STUDENT4) ? 2 : 0); ++k) {  // models/SeqPAN.py:64-70 (BaseFast: none, models/BaseFast.py:62-68)
      if ((rc = dual_block(k, cur, k == 0 && dab0_proj_done))) return rc;
      if ((rc = tap(4 + 2 * k, cur, SQ_D)) || (rc = tap(5 + 2 * k, cur + Mv * SQ_D, SQ_D))) return rc;
    }
    // CQAttention both ways + CQConcatenate (models/SeqPAN.py:73-75)
    if (tc && cq_tc_supported(L, T)) {
      const float* w4c[2] = {w[W_Q2V_W4C], w[W_V2Q_W4C]};
      const float* w4q[2] = {w[W_Q2V_W4Q], w[W_V2Q_W4Q]};
      const float* w4m[2] = {w[W_Q2V_W4MLU], w[W_V2Q_W4MLU]};
      const float* lb[2] = {w[W_Q2V_LIN_B], w[W_V2Q_LIN_B]};
      h->begin("cq_attention_tc", st);
      rc = cq_attention_tc(h->arena.tc, cur, vmask, tmask, w4c, w4q, w4m, lb, ws.cat2, 256, ws.v2t, SQ_D, B, L, T, st);
      h->end(st);
      ++h->launches;
      if (rc != SEQPAN_OK) return fail(rc, "cq_attention_tc failed");
    } else {
      CqArgs ca{cur, vmask, tmask, {w[W_Q2V_W4C], w[W_V2Q_W4C]}, {w[W_Q2V_W4Q], w[W_V2Q_W4Q]},
                {w[W_Q2V_W4MLU], w[W_V2Q_W4MLU]}, {ws.catv, ws.catt}, B, L, T};
      LAUNCH(h, launch_cq_attention(ca, st));
      if ((rc = linear(ws.catv, 512, w[W_Q2V_LIN_W], w[W_Q2V_LIN_B], nullptr, ws.cat2, 256, Mv, SQ_D, 512, false))) return rc;
      if ((rc = linear(ws.catt, 512, w[W_V2Q_LIN_W], w[W_V2Q_LIN_B], nullptr, ws.v2t, SQ_D, Mt, SQ_D, 512, false))) return rc;
    }
    if ((rc = tap(8, ws.cat2, 256)) || (rc = tap(9, ws.v2t, SQ_D))) return rc;
    if (tc) {
      // CQConcatenate + match head in two launches: the pooled half of the concat is a per-sample bias
      CHAIN(h, "pool_bias", launch_pool_bias(ws.v2t, tmask, w[W_POOL_W], w[W_CAT_W], ws.pbias, B, T, st));
      const bool no_match = h->s.variant == SEQPAN_VARIANT_BACKBONE;
      const float* mhv[4] = {h->hostw[W_CAT_B].data(), h->hostw[W_MATCH_W].data(), h->hostw[W_LABEL_EMBS].data(),
                             h->hostw[W_MATCH_B].data()};
      CHAIN(h, "chain_fuse_match", chain_fuse_match(h->arena.tc, ws.cat2, 256, Mv, L, ws.pbias, mhv, gumbel, vmask,
                                                    h->debug ? ws.fuse : nullptr, ws.fuse2, ws.fuse2_bf16, match_score, st, no_match));
      if ((rc = tap(10, ws.fuse, SQ_D)) || (rc = tap(11, ws.fuse2, SQ_D))) return rc;
      const HeadArgs hs{TC_START_HID, W_START_LN_W, W_START_LN_B, W_START_HID_B, W_START_DENSE_W, W_START_DENSE_B, slogits};
      const HeadArgs he{TC_END_HID, W_END_LN_W, W_END_LN_B, W_END_HID_B, W_END_DENSE_W, W_END_DENSE_B, elogits};
      if ((rc = fep(ws.fuse2, ws.ps, &hs))) return rc;
      if ((rc = fep(ws.ps, ws.pe, &he))) return rc;
      return (rc = tap(12, ws.ps, SQ_D)) ? rc : tap(13, ws.pe, SQ_D);
    }
    LAUNCH(h, launch_pool_tile(ws.v2t, tmask, w[W_POOL_W], ws.cat2, B, L, T, st));
    if ((rc = linear(ws.cat2, 256, w[W_CAT_W], w[W_CAT_B], nullptr, ws.fuse, SQ_D, Mv, SQ_D, 256, false))) return rc;
    if ((rc = tap(10, ws.fuse, SQ_D))) return rc;
    // match head (models/SeqPAN.py:78-82); BackBone has none: the concat output feeds the predictor (models/BackBone.py:62-63)
    if (h->s.variant == SEQPAN_VARIANT_BACKBONE) {
      CK(cudaMemcpyAsync(ws.fuse2, ws.fuse, sizeof(float) * Mv * SQ_D, cudaMemcpyDeviceToDevice, st));
    } else {
      LAUNCH(h, launch_match_head(ws.fuse, w[W_MATCH_W], w[W_MATCH_B], gumbel, w[W_LABEL_EMBS], vmask, match_score, ws.fuse2,
                                  Mv, st));
    }
    if ((rc = tap(11, ws.fuse2, SQ_D))) return rc;
    // SeqPANPredictor (models/layers.py:659-671)
    if ((rc = fep(ws.fuse2, ws.ps))) return rc;
    if ((rc = fep(ws.ps, ws.pe))) return rc;
    if ((rc = tap(12, ws.ps, SQ_D)) || (rc = tap(13, ws.pe, SQ_D))) return rc;
    if ((rc = ln(ws.ps, Mv, W_START_LN_W, 1e-6f, ws.cat3, 256, ws.fuse2, ws.cat3 + SQ_D))) return rc;
    if ((rc = linear(ws.cat3, 256, w[W_START_HID_W], w[W_START_HID_B], nullptr, ws.hid, SQ_D, Mv, SQ_D, 256, false))) return rc;
    LAUNCH(h, launch_rowdot(ws.hid, SQ_D, w[W_START_DENSE_W], w[W_START_DENSE_B], slogits, Mv, st));
    if ((rc = ln(ws.pe, Mv, W_END_LN_W, 1e-6f, ws.cat3, 256, ws.fuse2, ws.cat3 + SQ_D))) return rc;
    if ((rc = linear(ws.cat3, 256, w[W_END_HID_W], w[W_END_HID_B], nullptr, ws.hid, SQ_D, Mv, SQ_D, 256, false))) return rc;
    LAUNCH(h, launch_rowdot(ws.hid, SQ_D, w[W_END_DENSE_W], w[W_END_DENSE_B], elogits, Mv, st));
    return SEQPAN_OK;
  }
};

}  // namespace

static int forward_impl(SeqpanHandle* h, int mode, const int64_t* word_ids, const int64_t* char_ids, const float* vfeat,
                        const int32_t* video_index, int U, const float* vmask, const float* tmask, const float* gumbel, int B,
                        int T, int C, float* slogits, float* elogits, float* match_score, void* workspace,
                        size_t workspace_bytes, void* stream) {
  if (!h) return fail(SEQPAN_E_INVALID, "handle is NULL");
  const SeqpanShapes& s = h->s;
  if (B < 1 || B > s.max_batch) return fail(SEQPAN_E_INVALID, "B=%d outside [1,%d]", B, s.max_batch);
  if (T < 1 || T > s.max_tlen) return fail(SEQPAN_E_INVALID, "T=%d outside [1,%d]", T, s.max_tlen);
  if (C < 4 || C > s.max_clen) return fail(SEQPAN_E_INVALID, "C=%d outside [4,%d] (the k=4 char conv needs 4 characters)", C, s.max_clen);
  const bool has_match = s.variant != SEQPAN_VARIANT_BACKBONE;     // BackBone: no match head, gumbel / match_score unused
  if (!word_ids || !char_ids || !vfeat || !vmask || !tmask || !slogits || !elogits || (has_match && (!gumbel || !match_score)))
    return fail(SEQPAN_E_INVALID, "NULL tensor argument");
  if (!workspace || ((uintptr_t)workspace & 255)) return fail(SEQPAN_E_WORKSPACE, "workspace must be a 256-byte aligned device pointer");
  Fwd f{};
  f.h = h; f.st = (cudaStream_t)stream; f.B = B; f.L = s.vlen; f.T = T; f.C = C;
  f.Mv = (long long)B * s.vlen; f.Mt = (long long)B * T; f.M = f.Mv + f.Mt;
  f.tc = s.precision == SEQPAN_PREC_BF16;
  f.tf32 = s.precision == SEQPAN_PREC_TF32;
  Carver c(workspace);
  carve_workspace(c, s, B, T, f.ws);
  if (c.off > workspace_bytes) return fail(SEQPAN_E_WORKSPACE, "workspace too small: need %zu, have %zu", c.off, workspace_bytes);
  if (cq_attention_smem(s.vlen, T) > 227 * 1024)
    return fail(SEQPAN_E_INVALID, "L=%d, T=%d: CQAttention score tiles (%zu B) exceed 227 KB of shared memory", s.vlen, T, cq_attention_smem(s.vlen, T));
  if (dual_attention_smem(s.vlen, T) > 227 * 1024 || batch_attention_smem(B) > 227 * 1024)
    return fail(SEQPAN_E_INVALID, "attention tiles exceed 227 KB of shared memory (B=%d, L=%d, T=%d)", B, s.vlen, T);
  f.word_ids = word_ids; f.char_ids = char_ids; f.vmask = vmask; f.tmask = tmask; f.gumbel = gumbel;
  (mode == FWD_ENCODED ? f.venc : f.vfeat) = vfeat;
  f.slogits = slogits; f.elogits = elogits; f.match_score = match_score;
  f.video_index = video_index; f.U = U;
  h->launches = 0;
  h->lastB = B; h->lastT = T; h->last_encoded = mode == FWD_ENCODED;
  if (h->profile && h->recs.size() > 200000) { h->recs.clear(); h->pool_used = 0; }
  if (!h->use_graph || h->debug || h->profile || (h->use_graph == 2 && f.Mv > 8192)) return f.run();
  GraphKey key;
  memset(&key, 0, sizeof(key));
  const void* ptrs[11] = {word_ids, char_ids, vfeat, video_index, vmask, tmask, gumbel, slogits, elogits, match_score, workspace};
  memcpy(key.p, ptrs, sizeof(ptrs));
  key.B = B; key.T = T; key.C = C; key.U = U; key.side = h->use_side; key.mode = mode;
  ++h->tick;
  auto it = h->graphs.find(key);
  if (it != h->graphs.end()) {
    it->second.last_use = h->tick;
    CK(cudaGraphLaunch(it->second.exec, f.st));
    h->launches = it->second.launches;
    return SEQPAN_OK;
  }
  if (h->seen.size() > 4096) h->seen.clear();
  if (++h->seen[key] < 2) return f.run();      // first sighting: plain launches; a repeated argument set is worth a capture
  if (!h->cap_stream) CK(cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
  cudaStream_t user = f.st;
  CK(cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal));
  f.st = h->cap_stream;
  const int rc = f.run();
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(h->cap_stream, &graph);
  if (rc != SEQPAN_OK) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    return rc;
  }
  cudaGraphExec_t exec = nullptr;
  if (ce != cudaSuccess || !graph || cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) {
    // capture is an optimisation: if the runtime refuses it, run this and every later forward as plain launches
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    h->use_graph = 0;
    f.st = user;
    h->launches = 0;
    return f.run();
  }
  cudaGraphDestroy(graph);
  if (h->graphs.size() >= 64) {                 // bounded cache: evict the least recently used capture
    auto lru = h->graphs.begin();
    for (auto i = h->graphs.begin(); i != h->graphs.end(); ++i)
      if (i->second.last_use < lru->second.last_use) lru = i;
    cudaGraphExecDestroy(lru->second.exec);
    h->graphs.erase(lru);
  }
  h->graphs[key] = GraphEntry{exec, h->launches, h->tick};
  CK(cudaGraphLaunch(exec, user));
  return SEQPAN_OK;
}

extern "C" int seqpan_forward(SeqpanHandle* h, const int64_t* word_ids, const int64_t* char_ids, const float* vfeat,
                              const float* vmask, const float* tmask, const float* gumbel, int B, int T, int C,
                              float* slogits, float* elogits, float* match_score, void* workspace,
                              size_t workspace_bytes, void* stream) {
  return forward_impl(h, FWD_RAW, word_ids, char_ids, vfeat, nullptr, 0, vmask, tmask, gumbel, B, T, C, slogits, elogits, match_score,
                      workspace, workspace_bytes, stream);
}

extern "C" int seqpan_forward_shared_video(SeqpanHandle* h, const int64_t* word_ids, const int64_t* char_ids,
                                           const float* vfeat_unique, const int32_t* video_index, int U, const float* vmask,
                                           const float* tmask, const float* gumbel, int B, int T, int C, float* slogits,
                                           float* elogits, float* match_score, void* workspace, size_t workspace_bytes,
                                           void* stream) {
  if (!video_index) return fail(SEQPAN_E_INVALID, "video_index is NULL");
  if (U < 1 || U > B) return fail(SEQPAN_E_INVALID, "U=%d outside [1,B=%d]", U, B);
  return forward_impl(h, FWD_SHARED, word_ids, char_ids, vfeat_unique, video_index, U, vmask, tmask, gumbel, B, T, C, slogits,
                      elogits, match_score, workspace, workspace_bytes, stream);
}

// The argument checks that need no handle come first, so they answer the same with or without a device.
extern "C" int seqpan_encode_videos(SeqpanHandle* h, const float* vfeat, int U, float* venc, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  if (!vfeat || !venc) return fail(SEQPAN_E_INVALID, "NULL tensor argument");
  if (((uintptr_t)vfeat | (uintptr_t)venc) & 15) return fail(SEQPAN_E_INVALID, "vfeat and venc must be 16-byte aligned (vector and TMA access)");
  if (U < 1) return fail(SEQPAN_E_INVALID, "U=%d < 1", U);
  if (!h) return fail(SEQPAN_E_INVALID, "handle is NULL");
  const SeqpanShapes& s = h->s;
  if (U > s.max_batch) return fail(SEQPAN_E_INVALID, "U=%d > max_batch=%d (the workspace holds max_batch*vlen rows)", U, s.max_batch);
  if (!workspace || ((uintptr_t)workspace & 255)) return fail(SEQPAN_E_WORKSPACE, "workspace must be a 256-byte aligned device pointer");
  Fwd f{};
  f.h = h; f.st = (cudaStream_t)stream; f.B = U; f.L = s.vlen; f.T = 1; f.C = 4;
  f.Mv = (long long)U * s.vlen; f.Mt = U; f.M = f.Mv + f.Mt;
  f.tc = s.precision == SEQPAN_PREC_BF16;
  f.tf32 = s.precision == SEQPAN_PREC_TF32;
  Carver c(workspace);
  carve_workspace(c, s, U, 1, f.ws);
  if (c.off > workspace_bytes) return fail(SEQPAN_E_WORKSPACE, "workspace too small: need %zu, have %zu", c.off, workspace_bytes);
  h->launches = 0;
  h->lastB = 0;   // the workspace no longer holds a forward's taps
  if (h->profile && h->recs.size() > 200000) { h->recs.clear(); h->pool_used = 0; }
  return f.encode_clips(vfeat, U, f.ws.o, f.ws.u, venc);
}

extern "C" int seqpan_forward_encoded(SeqpanHandle* h, const int64_t* word_ids, const int64_t* char_ids, const float* venc,
                                      const int32_t* video_index, int U, const float* vmask, const float* tmask,
                                      const float* gumbel, int B, int T, int C, float* slogits, float* elogits,
                                      float* match_score, void* workspace, size_t workspace_bytes, void* stream) {
  if (!venc) return fail(SEQPAN_E_INVALID, "venc is NULL");
  if ((uintptr_t)venc & 15) return fail(SEQPAN_E_INVALID, "venc must be 16-byte aligned (the clip gather reads float4)");
  if (U < 1) return fail(SEQPAN_E_INVALID, "U=%d < 1", U);
  if (!video_index && U < B) return fail(SEQPAN_E_INVALID, "video_index is NULL and U=%d < B=%d: pair b needs clip b", U, B);
  return forward_impl(h, FWD_ENCODED, word_ids, char_ids, venc, video_index, U, vmask, tmask, gumbel, B, T, C, slogits, elogits,
                      match_score, workspace, workspace_bytes, stream);
}

extern "C" int64_t seqpan_debug_tap(SeqpanHandle* h, const char* name, const void* workspace, float* out,
                                    int64_t out_capacity_floats, void* stream) {
  if (!h || !name || !workspace || !out) return fail(SEQPAN_E_INVALID, "NULL argument");
  if (!h->debug || h->lastB == 0) return fail(SEQPAN_E_INVALID, "taps are recorded only after seqpan_set_debug(h,1) and a forward");
  Carver c((void*)workspace);
  Workspace ws;
  carve_workspace(c, h->s, h->lastB, h->lastT, ws);
  for (int i = 0; i < NUM_TAPS; ++i) {
    if (strcmp(name, kTapNames[i]) != 0) continue;
    if (i == 1 && h->last_encoded) return fail(SEQPAN_E_INVALID, "tap 'video_affine' does not exist on a forward from stored encodings");
    const int64_t rows = kTapIsText[i] ? (int64_t)h->lastB * h->lastT : (int64_t)h->lastB * h->s.vlen;
    if (rows * SQ_D > out_capacity_floats) return fail(SEQPAN_E_WORKSPACE, "tap '%s' needs %lld floats", name, (long long)rows * SQ_D);
    CK(cudaMemcpyAsync(out, ws.taps[i], sizeof(float) * rows * SQ_D, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return rows;
  }
  return fail(SEQPAN_E_INVALID, "unknown tap '%s'", name);
}

// ---- decode / metrics / single blocks ----------------------------------------------------------------
extern "C" int seqpan_span_decode(const float* slogits, const float* elogits, const float* vmask, int B, int L,
                                  int64_t* start_idx, int64_t* end_idx, float* fracs, void* stream) {
  if (!slogits || !elogits) return fail(SEQPAN_E_INVALID, "NULL logits");
  if (B < 0 || L < 1 || L > SEQPAN_MAX_VLEN) return fail(SEQPAN_E_INVALID, "L=%d outside [1,%d]", L, SEQPAN_MAX_VLEN);
  CK(launch_span_decode(slogits, elogits, vmask, B, L, start_idx, end_idx, fracs, (cudaStream_t)stream));
  return SEQPAN_OK;
}

extern "C" int seqpan_iou_counters(const float* fracs, const float* gt_fracs, int B, double* counters, void* stream) {
  if (!fracs || !gt_fracs || !counters) return fail(SEQPAN_E_INVALID, "NULL argument");
  CK(launch_iou_counters(fracs, gt_fracs, B, counters, false, (cudaStream_t)stream));
  return SEQPAN_OK;
}

extern "C" int seqpan_iou_counters_exact(const float* fracs, const float* gt_fracs, int B, double* counters, void* stream) {
  if (!fracs) return fail(SEQPAN_E_INVALID, "fracs is NULL");
  if (!gt_fracs) return fail(SEQPAN_E_INVALID, "gt_fracs is NULL");
  if (!counters) return fail(SEQPAN_E_INVALID, "counters is NULL");
  if (B < 0) return fail(SEQPAN_E_INVALID, "B=%d < 0", B);
  CK(launch_iou_counters(fracs, gt_fracs, B, counters, true, (cudaStream_t)stream));
  return SEQPAN_OK;
}

extern "C" int seqpan_gumbel_noise(uint64_t seed, uint32_t batch_id, int B, int L, float* out, void* stream) {
  if (!out) return fail(SEQPAN_E_INVALID, "out is NULL");
  if ((uintptr_t)out & 15) return fail(SEQPAN_E_INVALID, "out must be 16-byte aligned (one float4 per row)");
  if (B < 0) return fail(SEQPAN_E_INVALID, "B=%d < 0", B);
  if (L < 1 || L > SEQPAN_MAX_VLEN) return fail(SEQPAN_E_INVALID, "L=%d outside [1,%d]", L, SEQPAN_MAX_VLEN);
  if ((int64_t)B * L > (int64_t)UINT32_MAX) return fail(SEQPAN_E_INVALID, "B=%d: B*L rows exceed the 32-bit counter word", B);
  CK(launch_gumbel_noise(seed, batch_id, (uint32_t)((int64_t)B * L), out, (cudaStream_t)stream));
  return SEQPAN_OK;
}

extern "C" int seqpan_span_topk(const float* slogits, const float* elogits, const float* vmask, int B, int L, int k,
                                float nms_thresh, int64_t* start_idx, int64_t* end_idx, float* scores, float* fracs,
                                void* stream) {
  if (!slogits || !elogits) return fail(SEQPAN_E_INVALID, "NULL logits");
  if (!start_idx || !end_idx || !scores) return fail(SEQPAN_E_INVALID, "NULL output");
  if (B < 0) return fail(SEQPAN_E_INVALID, "B=%d < 0", B);
  if (L < 1 || L > SEQPAN_MAX_VLEN) return fail(SEQPAN_E_INVALID, "L=%d outside [1,%d]", L, SEQPAN_MAX_VLEN);
  if (k < 1 || k > SEQPAN_TOPK_MAX) return fail(SEQPAN_E_INVALID, "k=%d outside [1,%d]", k, SEQPAN_TOPK_MAX);
  if (!(nms_thresh > 0.f && nms_thresh <= 1.f)) return fail(SEQPAN_E_INVALID, "nms_thresh=%g outside (0,1]", nms_thresh);
  CK(launch_span_topk(slogits, elogits, vmask, B, L, k, nms_thresh, start_idx, end_idx, scores, fracs, (cudaStream_t)stream));
  return SEQPAN_OK;
}

extern "C" int seqpan_topk_counters(const float* fracs, const float* gt_fracs, int B, int k, double* counters, void* stream) {
  if (!fracs || !gt_fracs || !counters) return fail(SEQPAN_E_INVALID, "NULL argument");
  if (B < 0) return fail(SEQPAN_E_INVALID, "B=%d < 0", B);
  if (k < 1 || k > SEQPAN_TOPK_MAX) return fail(SEQPAN_E_INVALID, "k=%d outside [1,%d]", k, SEQPAN_TOPK_MAX);
  CK(launch_topk_counters(fracs, gt_fracs, B, k, counters, (cudaStream_t)stream));
  return SEQPAN_OK;
}

// Host -> device copy of zero-padded clip features that only moves the valid prefix of every sample and writes the
// padding rows as zeros on the device.  mode 0: one cudaMemcpyAsync per sample (copy engine) + a zero-fill kernel;
// mode >= 1: one kernel that reads the pinned host buffer directly (zero-copy over PCIe) with `mode` CTAs.
extern "C" int seqpan_h2d_ragged(float* dst, const float* src_host, const int32_t* valid_rows_host, int32_t* valid_rows_dev,
                                 int B, int L, int row_floats, int mode, void* stream) {
  if (!dst || !src_host || !valid_rows_host || !valid_rows_dev) return fail(SEQPAN_E_INVALID, "NULL argument");
  if (B < 0 || L < 1 || row_floats < 4 || (row_floats & 3)) return fail(SEQPAN_E_INVALID, "bad ragged copy shape");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t row_bytes = (size_t)row_floats * sizeof(float);
  for (int b = 0; b < B; ++b)
    if (valid_rows_host[b] < 0 || valid_rows_host[b] > L)
      return fail(SEQPAN_E_INVALID, "valid_rows[%d]=%d outside [0,%d]", b, valid_rows_host[b], L);
  CK(cudaMemcpyAsync(valid_rows_dev, valid_rows_host, sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
  if (mode >= 1) {
    CK(launch_h2d_ragged(dst, src_host, valid_rows_dev, B, L, row_floats, mode, st));
    return SEQPAN_OK;
  }
  for (int b = 0; b < B; ++b) {
    const int n = valid_rows_host[b];
    if (n > 0)
      CK(cudaMemcpyAsync(dst + (size_t)b * L * row_floats, src_host + (size_t)b * L * row_floats, n * row_bytes,
                         cudaMemcpyHostToDevice, st));
  }
  CK(launch_zero_tail_rows(dst, valid_rows_dev, B, L, row_floats, st));
  return SEQPAN_OK;
}

// sample_vfeat_linear (feature half) + pad_video_seq + convert_length_to_mask for a batch of ragged clips resident in HBM.
extern "C" int seqpan_collate_clips(const float* raw, const int64_t* row_offsets_host, int64_t* row_offsets_dev, int B,
                                    int vlen, int row_floats, int mode, float* vfeats, float* vmask, int64_t* vlens,
                                    void* stream) {
  if (!row_offsets_host || !row_offsets_dev || !vfeats) return fail(SEQPAN_E_INVALID, "NULL argument");
  if (B < 0 || vlen < 1 || vlen > 65535 || row_floats < 1) return fail(SEQPAN_E_INVALID, "bad collate shape");
  if (mode < SEQPAN_SAMPLE_ORIGINAL || mode > SEQPAN_SAMPLE_SAMELEN) return fail(SEQPAN_E_INVALID, "unknown sample mode %d", mode);
  for (int b = 0; b < B; ++b) {
    const int64_t n = row_offsets_host[b + 1] - row_offsets_host[b];
    if (n < 0 || n > INT32_MAX || row_offsets_host[b] < 0) return fail(SEQPAN_E_INVALID, "row_offsets not ascending at clip %d", b);
    // "original" keeps the clip as it is: the reference's torch.stack fails when one is longer than max_vlen
    if (mode == SEQPAN_SAMPLE_ORIGINAL && n > vlen)
      return fail(SEQPAN_E_INVALID, "clip %d has %lld rows > vlen=%d with sample mode \"original\"", b, (long long)n, vlen);
    // interpolate_avrage indexes x[round(i/size*(n-1))]: an empty clip has no row to take
    if (n == 0 && (mode == SEQPAN_SAMPLE_SAMELEN)) return fail(SEQPAN_E_INVALID, "clip %d is empty", b);
  }
  if (B > 0 && !raw && row_offsets_host[B] > 0) return fail(SEQPAN_E_INVALID, "NULL raw features");
  cudaStream_t st = (cudaStream_t)stream;
  if (B == 0) return SEQPAN_OK;
  CK(cudaMemcpyAsync(row_offsets_dev, row_offsets_host, sizeof(int64_t) * (B + 1), cudaMemcpyHostToDevice, st));
  CK(launch_collate_clips(raw, row_offsets_dev, B, vlen, row_floats, mode, vfeats, vmask, vlens, st));
  return SEQPAN_OK;
}

// pad_seq + pad_char_seq + tmask for a batch of ragged id lists resident in HBM (text half of BaseCollate).
extern "C" int seqpan_collate_text(const int64_t* words, const int64_t* word_offsets, const int64_t* chars, const int64_t* char_offsets,
                                   int B, int T, int C, int64_t* word_ids, int64_t* char_ids, float* tmask, void* stream) {
  if (B < 0 || T < 1 || C < 1) return fail(SEQPAN_E_INVALID, "bad text collate shape");
  if (B == 0) return SEQPAN_OK;
  if (!words || !word_offsets || !chars || !char_offsets || !word_ids || !char_ids || !tmask) return fail(SEQPAN_E_INVALID, "NULL argument");
  CK(launch_collate_text(words, word_offsets, chars, char_offsets, B, T, C, word_ids, char_ids, tmask, (cudaStream_t)stream));
  return SEQPAN_OK;
}

#ifdef SEQPAN_TIMELINE   // instrumented builds only (include/seqpan_b200_diag.h)
extern "C" int seqpan_debug_timeline(int which, long long* out_host64) {
  if (!out_host64) return fail(SEQPAN_E_INVALID, "NULL argument");
  CK(cudaDeviceSynchronize());
  int rc = which == 0 ? chain_read_timeline(out_host64)
                      : (which == 2 ? tail_read_timeline(out_host64) : (which == 3 ? tc_read_timeline(out_host64) : attn_read_timeline(out_host64)));
  if (rc != SEQPAN_OK) return fail(rc, "timeline not compiled in (build with SEQPAN_TIMELINE=1)");
  return SEQPAN_OK;
}
#endif

extern "C" size_t seqpan_op_linear_scratch_bytes(int64_t M, int N, int K) { return tc_op_scratch_bytes(M, N, K); }

extern "C" int seqpan_op_linear(const float* x, const float* w, const float* bias, const float* residual, float* y,
                                int64_t M, int N, int K, int flags, int precision, void* scratch, size_t scratch_bytes,
                                void* stream) {
  if (!x || !w || !y || M < 0 || N < 1 || K < 4 || (K & 3)) return fail(SEQPAN_E_INVALID, "bad linear arguments");
  if ((flags & 2) && !residual) return fail(SEQPAN_E_INVALID, "residual flag without residual pointer");
  if (precision == 2) {  // fp32 operands on kind::tf32 (the video-affine path), no scratch needed
    int rc = tc_linear_tf32(x, K, w, bias, (flags & 2) ? residual : nullptr, y, N, M, N, K, flags & 1, (cudaStream_t)stream);
    if (rc != SEQPAN_OK) return fail(rc, "%s", tc_last_error());
    return SEQPAN_OK;
  }
  if (precision == SEQPAN_PREC_BF16) {
    int rc = tc_op_linear(x, w, bias, (flags & 2) ? residual : nullptr, y, M, N, K, flags & 1, scratch, scratch_bytes,
                          (cudaStream_t)stream);
    if (rc != SEQPAN_OK) return fail(rc, "%s", tc_last_error());
    return SEQPAN_OK;
  }
  LinearArgs a{};
  a.x[0] = x; a.w[0] = w; a.bias[0] = bias; a.res[0] = (flags & 2) ? residual : nullptr; a.y[0] = y;
  a.M = M; a.N = N; a.K = K; a.ldx = K; a.ldw = K; a.ldy = N; a.ldr = N; a.relu = flags & 1; a.count = 1;
  CK(launch_linear_f32(a, (cudaStream_t)stream));
  return SEQPAN_OK;
}

extern "C" int seqpan_op_layernorm(const float* x, const float* gamma, const float* beta, float eps, float* y, int64_t M,
                                   void* stream) {
  if (!x || !gamma || !beta || !y) return fail(SEQPAN_E_INVALID, "NULL argument");
  CK(launch_layernorm(x, SQ_D, M, gamma, beta, eps, y, SQ_D, nullptr, nullptr, nullptr, 0, nullptr, nullptr, 0,
                      (cudaStream_t)stream));
  return SEQPAN_OK;
}
