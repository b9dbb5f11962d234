// umma.cuh -- thin inline-PTX layer over the sm_100a tensor-core path used by field_tc.cu:
// mbarrier, 1-D bulk TMA copies (cp.async.bulk), TMEM allocation, tcgen05.mma (SS and TS
// operand forms), tcgen05.commit, tcgen05.ld/st.  Bit layouts of the shared-memory and
// instruction descriptors follow the PTX ISA "tcgen05" chapter (same fields as
// cute/arch/mma_sm100_desc.hpp, which was read as documentation only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace snb {
namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One lane of a converged warp (elect.sync).  tcgen05.mma / commit / bulk copies execute on the
// uniform datapath: issuing them under a plain `lane == 0` branch makes the compiler wrap each
// one in a per-active-thread loop; under elect.sync it emits the instruction once.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ------------------------------------------------------------------ bulk copy (TMA engine, 1-D)
// global -> this CTA's shared memory; completion is signalled on `bar` as transaction bytes.
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// make generic-proxy smem writes visible to the async proxy (tcgen05.mma / TMA reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ------------------------------------------------------------------ TMEM
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {  // one full warp
  static_assert(kCols >= 32 && kCols <= 512 && (kCols & (kCols - 1)) == 0, "TMEM columns: power of two in [32,512]");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {  // the allocating warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// TMEM address: lane in bits [31:16], column in [15:0].  A warp may only touch lanes
// 32*(warp_id % 4) .. +31; with the 32x32b shape thread i of the warp owns lane base+i.
__device__ __forceinline__ uint32_t tmem_addr(uint32_t base, uint32_t lane, uint32_t col) {
  return base + (lane << 16) + col;
}

#define SNB_R8(v, o) "=r"(v[o + 0]), "=r"(v[o + 1]), "=r"(v[o + 2]), "=r"(v[o + 3]), "=r"(v[o + 4]), "=r"(v[o + 5]), "=r"(v[o + 6]), "=r"(v[o + 7])
#define SNB_W8(v, o) "r"(v[o + 0]), "r"(v[o + 1]), "r"(v[o + 2]), "r"(v[o + 3]), "r"(v[o + 4]), "r"(v[o + 5]), "r"(v[o + 6]), "r"(v[o + 7])

// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : SNB_R8(v, 0), SNB_R8(v, 8), SNB_R8(v, 16), SNB_R8(v, 24)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : SNB_R8(v, 0)
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%32], "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31};" ::SNB_W8(v, 0),
      SNB_W8(v, 8), SNB_W8(v, 16), SNB_W8(v, 24), "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%16], "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15};" ::SNB_W8(v, 0),
      SNB_W8(v, 8), "r"(taddr)
      : "memory");
}

// ------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor, K-major operand, SWIZZLE_NONE ("interleaved") canonical
// layout: 8-row x 16-byte core matrices, each one contiguous 128 B.
//   lbo_bytes: distance between core matrices adjacent in K
//   sbo_bytes: distance between core matrices adjacent in M/N (next 8 rows)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);        // start address       bits [0,14)
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;    // leading byte offset bits [16,30)
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;    // stride byte offset  bits [32,46)
  d |= (uint64_t)1 << 46;                               // descriptor version 1 (sm_100)
  return d;                                             // base_offset 0, lbo_mode 0, layout SWIZZLE_NONE (0)
}

enum : uint32_t { kFmtF16 = 0, kFmtBF16 = 1 };
// Instruction descriptor for kind::f16, fp32 accumulate, A and B K-major, dense.
__host__ __device__ constexpr uint32_t make_idesc(uint32_t fmt, uint32_t M, uint32_t N) {
  return (1u << 4)             // c_format = F32
         | (fmt << 7)          // a_format
         | (fmt << 10)         // b_format
         | (0u << 15) | (0u << 16)   // a_major = K, b_major = K
         | ((N >> 3) << 17)    // n_dim
         | ((M >> 4) << 24);   // m_dim
}

// D[tmem] (+)= A[smem] * B[smem]^T     (single thread issues)
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                       uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                       uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all MMAs issued so far by this thread arrive on `bar` when they complete
// (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ------------------------------------------------------------------ CTA-pair (cta_group::2) forms
// One MMA spans two SMs: M = 256 (rows 0-127 in the even CTA's TMEM, 128-255 in the odd CTA's),
// each CTA supplies half of B's rows from its own shared memory at the same offset.  Issued by
// the even ("leader") CTA only.  Validated on hardware by probes/umma2_probe.cu.
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_result) {  // same warp index in both CTAs
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(smem_result))
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(taddr) : "memory");
}
__device__ __forceinline__ void mma2_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma2_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Variants that take the smem descriptors as (lo, hi) 32-bit halves: between the MMAs of a chunk
// only the 14-bit start-address field (low word) changes, so the issuing thread does 32-bit adds.
__device__ __forceinline__ void mma2_ts_lohi(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo32, uint32_t b_hi32,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 bd;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 bd, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], bd, %4, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "r"(b_lo32), "r"(b_hi32), "r"(idesc), "r"(accumulate));
}
__device__ __forceinline__ void mma2_ss_lohi(uint32_t d_tmem, uint32_t a_lo32, uint32_t a_hi32, uint32_t b_lo32,
                                             uint32_t b_hi32, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 ad, bd;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 ad, {%1, %2};\n\t"
      "mov.b64 bd, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], ad, bd, %5, p;\n\t}" ::"r"(d_tmem),
      "r"(a_lo32), "r"(a_hi32), "r"(b_lo32), "r"(b_hi32), "r"(idesc), "r"(accumulate));
}
// completion of all prior MMAs arrives on the barrier at this smem offset in both CTAs of the pair
__device__ __forceinline__ void mma2_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}
// arrive on the barrier at this smem offset in CTA `cta` of the cluster.  Default semantics
// (.release at CTA scope): the data hand-offs it orders are tcgen05 / async-proxy operations that
// carry their own fences (tcgen05.fence::before/after_thread_sync, fence.proxy.async); explicit
// cluster-scope release/acquire would add an L1 invalidate + membar per arrive/wait.
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
// wait that also acquires writes released by threads of the peer CTA
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}

}  // namespace umma
}  // namespace snb
