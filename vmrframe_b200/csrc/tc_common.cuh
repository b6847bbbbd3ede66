// PTX wrappers shared by the tcgen05 kernels: mbarrier, TMA, TMEM, UMMA descriptors (sm_100a).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace tcx {

// ---- PTX wrappers ----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug becomes a trap (launch failure) instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) __trap();
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptor: K-major operand tile [rows][64 bf16], 128-byte swizzle, 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);  // start address, 16-byte units
  d |= (uint64_t)1 << 16;                    // leading byte offset: unused for swizzled K-major (canonical value 1)
  d |= (uint64_t)(1024u >> 4) << 32;         // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;                    // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                    // SWIZZLE_128B
  return d;
}
// The same descriptor `byte_off` bytes further on (start-address field, 16-byte units; operands never leave the 256 KB
// shared window, so the add cannot carry out of the field).  The MMA-issuing thread is a single serial instruction
// stream: building every descriptor from scratch costs ~22 SASS instructions per tcgen05.mma, more than the MMA takes.
__device__ __forceinline__ uint64_t desc_add(uint64_t d, uint32_t byte_off) {
  return (d & 0xFFFFFFFF00000000ull) | (uint64_t)((uint32_t)d + (byte_off >> 4));
}
// MN-major B operand: a row-major [k rows][n cols] bf16 matrix exactly as a K-major tile of it would be stored
// (k-blocks of [rows][64 elements], 128-byte swizzle) -- no transposition.  8-row groups are 1024 B apart (SBO), the
// 64-element n-blocks `nblock_bytes` apart (LBO).  Needs bit 16 (b_major) of the instruction descriptor.  Advancing K by
// 16 rows = +2048 bytes on the start address.  Conventions pinned by tests/test_gpu_parity.py::test_umma_descriptor_conventions.
__device__ __forceinline__ uint64_t make_mn_sw128_desc(uint32_t saddr, uint32_t nblock_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((nblock_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)(1024u >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// MN-major B operand of 32 columns: [k rows][32 elements] rows of 64 bytes, 64-byte swizzle, 8-row groups 512 B apart.
__device__ __forceinline__ uint64_t make_mn_sw64_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512u >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;
  return d;
}
constexpr uint32_t IDESC_B_MN_MAJOR = 1u << 16;
// Instruction descriptor, kind::f16: D fp32, A/B bf16, both K-major, M=128, N=BN.
__device__ __forceinline__ uint32_t make_idesc(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// kind::tf32: A/B are fp32 in shared memory (the tensor core reads the top 19 bits), UMMA_K = 8 elements = 32 bytes
__device__ __forceinline__ uint32_t make_idesc_tf32(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}


__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// generic-proxy writes to shared memory (st.shared) -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }


// tcgen05.wait::ld that also names the destination registers of the pending load as read-write operands, so the
// compiler cannot schedule a consumer of those registers above the wait (the load itself is asynchronous).
__device__ __forceinline__ void tmem_wait16(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

// Software-pipelined sweep over NCH 16-column chunks of NSRC accumulators (column bases col[0..NSRC)) of this
// thread's TMEM lane: the tcgen05.ld of chunk c+1 is in flight while f(c, regs) processes chunk c.
template <int NCH, int NSRC, bool PIPE = true, class F>
__device__ __forceinline__ void tmem_pipe16(uint32_t lane_base, const uint32_t (&col)[NSRC], F&& f) {
  if constexpr (!PIPE) {  // plain sweep: fewer live registers (measured faster in the register-heavy chain kernels)
#pragma unroll 1
    for (int c = 0; c < NCH; ++c) {
      uint32_t buf[NSRC][16];
#pragma unroll
      for (int s = 0; s < NSRC; ++s) tmem_ld16(lane_base + col[s] + c * 16, buf[s]);
#pragma unroll
      for (int s = 0; s < NSRC; ++s) tmem_wait16(buf[s]);
      f(c, buf);
    }
  } else {
    uint32_t buf[2][NSRC][16];
#pragma unroll
    for (int s = 0; s < NSRC; ++s) tmem_ld16(lane_base + col[s], buf[0][s]);
#pragma unroll
    for (int s = 0; s < NSRC; ++s) tmem_wait16(buf[0][s]);
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      if (c + 1 < NCH) {
#pragma unroll
        for (int s = 0; s < NSRC; ++s) tmem_ld16(lane_base + col[s] + (c + 1) * 16, buf[(c + 1) & 1][s]);
      }
      f(c, buf[c & 1]);
      if (c + 1 < NCH) {
#pragma unroll
        for (int s = 0; s < NSRC; ++s) tmem_wait16(buf[(c + 1) & 1][s]);
      }
    }
  }
}

// Runtime-length variant for one accumulator: f(c, regs) for c in [0, nch).
template <class F>
__device__ __forceinline__ void tmem_pipe16_rt(uint32_t taddr, int nch, F&& f) {
  uint32_t a[16], b[16];
  tmem_ld16(taddr, a);
  tmem_wait16(a);
#pragma unroll 1
  for (int c = 0; c < nch; c += 2) {
    if (c + 1 < nch) tmem_ld16(taddr + (c + 1) * 16, b);
    f(c, a);
    if (c + 1 < nch) {
      tmem_wait16(b);
      if (c + 2 < nch) tmem_ld16(taddr + (c + 2) * 16, a);
      f(c + 1, b);
      if (c + 2 < nch) tmem_wait16(a);
    }
  }
}

// Byte offset of element (row, col) inside a K-major bf16 operand tile stored as consecutive k-blocks of
// [rows_per_tile][64] with the 128-byte swizzle TMA/UMMA use (16-byte chunk index XOR row-in-group).
// `col` must be a multiple of 8 (one 16-byte chunk).  KB_BYTES = bytes of one k-block (rows * 128).
template <int KB_BYTES>
__device__ __forceinline__ uint32_t sw128_chunk_offset(int row, int col) {
  const int kb = col >> 6, ch = (col & 63) >> 3;
  return (uint32_t)(kb * KB_BYTES + (row >> 3) * 1024 + (row & 7) * 128 + ((ch ^ (row & 7)) << 4));
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// Variants without the "memory" clobber: still ordered among the other volatile asm statements (fences, barriers,
// other stores) but ordinary C++ loads may be scheduled across them -- for operand-building loops whose loads and
// stores touch disjoint shared-memory regions.
__device__ __forceinline__ void st_shared_v2_nc(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b));
}
__device__ __forceinline__ void st_shared_v4_nc(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d));
}
// Packed fp32x2 arithmetic (Blackwell FFMA2 / FADD2 / FMUL2): two independent fp32 operations per instruction on a
// 64-bit register pair -- exact fp32 results at half the issue slots of the scalar forms.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void st_shared_v2(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}

// ---- helpers of the 128 x 128 "chain" tiles: operand tile = 2 k-blocks of [128 rows][64 bf16] (16 KB each) ----
constexpr int CH_KBB = 16384;
constexpr int CH_TILE = 2 * CH_KBB;
// D[128,128] (+)= A-tile . W-tile^T, both K-major bf16, K = 128 (8 UMMAs of K = 16)
__device__ __forceinline__ void ch_mma_tile(uint32_t tmem_d, uint32_t abuf, uint32_t wbuf, uint32_t idesc, bool accumulate) {
  const uint64_t ad = make_sw128_desc(abuf), wd = make_sw128_desc(wbuf);
#pragma unroll
  for (int kb = 0; kb < 2; ++kb)
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma_bf16(tmem_d, desc_add(ad, kb * CH_KBB + k * 32), desc_add(wd, kb * CH_KBB + k * 32), idesc,
                (accumulate || kb || k) ? 1u : 0u);
}
// 16 fp32 values of one row -> bf16 -> operand tile (two 16-byte chunks), swizzled
__device__ __forceinline__ void ch_store_a16(uint32_t abuf, int row, int col, const float (&v)[16]) {
  st_shared_v4(abuf + sw128_chunk_offset<CH_KBB>(row, col), pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]),
               pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
  st_shared_v4(abuf + sw128_chunk_offset<CH_KBB>(row, col + 8), pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]),
               pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
}
// one 128-row weight tile (both k-blocks) by TMA; `col0` = first K column of the tile inside the weight matrix
__device__ __forceinline__ void ch_load_w(uint32_t dst, const CUtensorMap* map, uint32_t bar, int col0, int row0) {
  mbar_expect_tx(bar, CH_TILE);
  tma_load_2d(dst, map, bar, col0, row0);
  tma_load_2d(dst + CH_KBB, map, bar, col0 + 64, row0);
}

// ---- fp32 row tiles moved by TMA: [128 rows][128 floats] = 4 boxes of [128 rows][32 floats] (16 KB each), 128-byte swizzle ----
// A thread that owns a row reads/writes its 16-byte chunks conflict-free (the 8 lanes of a quarter warp hit 8 different
// swizzled chunks); the boxes go to / come from global memory as whole 128-byte row segments.
constexpr int F32_BOX_B = 16384;
constexpr int F32_TILE_B = 4 * F32_BOX_B;
__device__ __forceinline__ uint32_t f32_tile_off(int row, int col) {      // col: multiple of 4
  return (uint32_t)((col >> 5) * F32_BOX_B + row * 128 + ((((col & 31) >> 2) ^ (row & 7)) << 4));
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ float4 ld_shared_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void st_shared_f4(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

}  // namespace tcx

// Optional phase timeline (build with -DSEQPAN_TIMELINE): SM clock stamps written by the thread `threadIdx.x == 32` of
// CTA 1 (slots 0..31) and by any thread of that CTA through TLC (slots 32..63); one buffer per translation unit, read
// back with seqpan_debug_timeline().  Compiled out by default.
#ifdef SEQPAN_TIMELINE
static __device__ long long tl_buf[64];
#define TL(i) do { if (blockIdx.x == 1 && blockIdx.y == 0 && threadIdx.x == 32) tl_buf[(i)] = clock64(); } while (0)
#define TLC(i) do { if (blockIdx.x == 1 && blockIdx.y == 0) tl_buf[32 + (i)] = clock64(); } while (0)
static inline int tl_read(long long* out64) {
  return cudaMemcpyFromSymbol(out64, tl_buf, sizeof(long long) * 64) == cudaSuccess ? 0 : -2;
}
#else
#define TL(i) do {} while (0)
#define TLC(i) do {} while (0)
static inline int tl_read(long long*) { return -1; }
#endif
