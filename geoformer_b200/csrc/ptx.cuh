// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM).
// Written for this project; syntax cross-checked against the PTX ISA as exercised by CUTLASS 4.x headers.
#pragma once
#include <stdint.h>
#include <cuda.h>

namespace gf { namespace ptx {

__device__ __forceinline__ uint32_t smem_addr(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------- mbarrier ----------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "DONE:\n\t}"
      ::"r"(smem_addr(bar)), "r"(parity) : "memory");
}

// ---------------- TMA ----------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 3-D tiled load: coordinates (c0 = innermost element index, c1 = row, c2 = batch)
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_addr(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_addr(bar)),
        "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_addr(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_addr(bar)),
        "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// multicast variant: the box lands at the same shared-memory offset in every CTA of `cta_mask` and signals the
// mbarrier at the same offset in each of them
__device__ __forceinline__ void tma_load_3d_mcast(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                                  int c0, int c1, int c2, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%3, %4, %5}], [%2], %6;"
      ::"r"(smem_addr(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_addr(bar)),
        "r"(c0), "r"(c1), "r"(c2), "h"(cta_mask)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// 3-D tiled store smem -> global (bulk async-group completion); OOB parts of the box are clipped
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
      ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_addr(smem_src)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }

// ---------------- tcgen05 / TMEM ----------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(smem_slot)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {      // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after()  { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::tf32 or kind::f16 selected at compile time
template <int KIND>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (KIND == 0) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
  }
}
// Lean issue path: shared-memory descriptors as (low word, shared high word).  Only the low word (start address >> 4)
// changes between the MMAs of a tile, so the per-MMA arithmetic is one 32-bit add that stays in a uniform register.
// Call from a CONVERGED warp under `if (elect_one())` (see conv_tc.cu for why).
constexpr uint32_t kDescHiSw128 = (1024u >> 4) | (1u << 14) | (2u << 29);     // SBO 1024 B, version 1, SWIZZLE_128B
constexpr uint32_t kDescHiSw64 = (512u >> 4) | (1u << 14) | (4u << 29);       // SBO 512 B, version 1, SWIZZLE_64B
constexpr uint32_t kDescHiSw32 = (256u >> 4) | (1u << 14) | (6u << 29);       // SBO 256 B, version 1, SWIZZLE_32B
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t smem_byte_addr) {
  return ((smem_byte_addr >> 4) & 0x3FFFu) | (1u << 16);
}
template <int KIND>
__device__ __forceinline__ void umma_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc,
                                        uint32_t accumulate) {
  if constexpr (KIND == 0) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 da, {%1, %4};\n\tmov.b64 db, {%2, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(desc_hi), "r"(accumulate) : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 da, {%1, %4};\n\tmov.b64 db, {%2, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(desc_hi), "r"(accumulate) : "memory");
  }
}
// A operand in tensor memory, B descriptor as (low word, high word)
__device__ __forceinline__ void umma_ts_f16_lo(uint32_t tmem_d, uint32_t tmem_a, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\tsetp.ne.b32 p, %5, 0;\n\tmov.b64 db, {%2, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "r"(b_lo), "r"(idesc), "r"(desc_hi), "r"(accumulate) : "memory");
}

// same with the A operand in tensor memory (".ts" form, kind::f16): A = this CTA's 128 lanes x (K / 2) 32-bit columns at
// `tmem_a` holding two consecutive K elements per column (low half first); B from shared memory
__device__ __forceinline__ void umma_ts_f16(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_addr(bar)) : "memory");
}

// variants taking the barrier's shared-memory address (lets the caller keep it in a uniform register)
__device__ __forceinline__ void umma_commit_addr(uint32_t bar_smem_addr) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_smem_addr) : "memory");
}
__device__ __forceinline__ void umma_commit_mcast_addr(uint32_t bar_smem_addr, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar_smem_addr), "h"(cta_mask) : "memory");
}

// same, arriving on the barrier at this offset in every CTA of `cta_mask` (slot release for multicast operands)
__device__ __forceinline__ void umma_commit_mcast(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_addr(bar)), "h"(cta_mask) : "memory");
}

// ---------------- CTA pairs (cta_group::2): one MMA spans two SMs ----------------
// D rows 0..127 live in CTA 0's tensor memory, rows 128..255 in CTA 1's; each CTA supplies its own 128 rows of A and HALF
// of the N rows of B from its own shared memory (same offsets in both CTAs), so every weight byte is written to and read
// from shared memory once per 256 output rows instead of once per 128.  Only the leader CTA (rank 0) issues.
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_slot, uint32_t ncols) {   // one whole warp in EACH CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(smem_slot)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;     // shared::cluster address of the same offset in the pair's leader CTA
// TMA loads of a CTA pair: the box lands in the ISSUING CTA's shared memory, the bytes are counted on the LEADER's mbarrier
__device__ __forceinline__ void tma_load_3d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_addr(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_addr(bar) & kPeerBitMask),
        "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_addr(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_addr(bar) & kPeerBitMask),
        "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// kind::f16 MMA over the CTA pair (M = 256); descriptors as (low word, shared high word) like umma_lo
__device__ __forceinline__ void umma2_f16_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 da, {%1, %4};\n\tmov.b64 db, {%2, %4};\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(desc_hi), "r"(accumulate) : "memory");
}
// arrive (once all earlier MMAs of this thread retired) on the barrier at this offset in the CTAs of `cta_mask`
__device__ __forceinline__ void umma2_commit_mcast_addr(uint32_t bar_smem_addr, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar_smem_addr), "h"(cta_mask) : "memory");
}
// arrive on the barrier at the same offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(smem_addr(bar)), "r"(rank) : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive 32-bit columns (thread t <- lane t)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// same for 16 consecutive columns
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
// registers -> TMEM: this warp's 32 lanes x 32 (16) consecutive 32-bit columns (lane t <- thread t)
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const float* v) {
  const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const float* v) {
  const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// UMMA shared-memory matrix descriptor, K-major operand tile stored as rows of 128 bytes with the
// 128-byte swizzle (what a TMA box {128B, rows} with CU_TENSOR_MAP_SWIZZLE_128B produces):
// 8-row x 128B swizzle atoms stacked every 1024 bytes (SBO); LBO unused for swizzled K-major.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_byte_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_byte_addr >> 4) & 0x3FFF);   // start address, bits [0,14)
  d |= static_cast<uint64_t>(1) << 16;                          // LBO (ignored), bits [16,30)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;                  // SBO = 1024 B, bits [32,46)
  d |= static_cast<uint64_t>(1) << 46;                          // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;                          // layout: SWIZZLE_128B
  return d;
}

// Same for a K-major tile that is only 32 bytes wide (one K = 16 step of 16-bit elements): rows of 32 bytes with the
// 32-byte swizzle (TMA box {32 B, rows} with CU_TENSOR_MAP_SWIZZLE_32B); 8-row atoms every 256 bytes.
__device__ __forceinline__ uint64_t umma_desc_sw32(uint32_t smem_byte_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_byte_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>(1) << 16;                          // LBO (ignored)
  d |= static_cast<uint64_t>(256 >> 4) << 32;                   // SBO = 256 B
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(6) << 61;                          // layout: SWIZZLE_32B
  return d;
}

// Instruction descriptor for kind::tf32 / kind::f16, fp32 accumulate, both operands K-major.
// fmt: 0 = f16, 1 = bf16, 2 = tf32.
__host__ __device__ constexpr uint32_t umma_idesc(int fmt, int m, int n) {
  return (1u << 4) | (uint32_t(fmt) << 7) | (uint32_t(fmt) << 10) | (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}

}}  // namespace gf::ptx
