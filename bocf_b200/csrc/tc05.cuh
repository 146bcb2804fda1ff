// tc05.cuh -- inline-PTX wrappers for the Blackwell (sm_100a) async machinery used by split_gemm.cu:
// mbarrier, bulk async copies (TMA engine, SASS UBLKCP), tensor memory (TMEM) allocation / loads (LDTM) and
// the 5th-generation tensor-core instruction tcgen05.mma (SASS UTCIMMA for kind::i8).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bocf {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ---- mbarrier ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded spin: a protocol error traps (kernel fails with an error the host sees) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 28)) __trap();
  }
}

// Pure polling variant (mbarrier.test_wait never suspends the thread): lowest wake-up latency, used on the
// latency-critical cross-CTA handshakes of the CTA-pair kernel.
__device__ __forceinline__ void mbar_wait_spin(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0, ok = 0;
  const uint32_t a = smem_u32(bar);
  while (true) {
    asm volatile("{\n .reg .pred p;\n mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok)
                 : "r"(a), "r"(parity)
                 : "memory");
    if (ok) break;
    if (++spins > (1u << 30)) __trap();
  }
}

// ---- bulk async copy global -> shared (TMA engine; completes on an mbarrier with byte count) -------------------
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// L2 prefetch of a contiguous global range (multiple of 16 bytes), fire and forget.
__device__ __forceinline__ void prefetch_l2(const void* gmem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(gmem_src), "r"(bytes) : "memory");
}

// ---- tensor memory -------------------------------------------------------------------------------------------
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(slot_in_smem)),
               "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {          // whole warp (the allocating one)
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

// 32 lanes x 16 consecutive 32-bit columns: thread `lane` of the warp receives row (lane base + lane), columns c..c+15.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&v)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3])
               : "r"(taddr)
               : "memory");
}
template <int W>
__device__ __forceinline__ void tmem_ldw(uint32_t taddr, uint32_t (&v)[W]);
template <>
__device__ __forceinline__ void tmem_ldw<4>(uint32_t taddr, uint32_t (&v)[4]) { tmem_ld4(taddr, v); }
template <>
__device__ __forceinline__ void tmem_ldw<16>(uint32_t taddr, uint32_t (&v)[16]) { tmem_ld16(taddr, v); }
template <>
__device__ __forceinline__ void tmem_ldw<8>(uint32_t taddr, uint32_t (&v)[8]) { tmem_ld8(taddr, v); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// ---- tcgen05.mma ---------------------------------------------------------------------------------------------
// Shared-memory operand descriptor, K-major canonical layout with 64-byte swizzle:
//   rows of 64 bytes (= 64 int8 along K), 8-row groups of 512 bytes (SBO), 16-byte pieces XOR-swizzled with
//   address bits [7,9)  (Swizzle<2,4,3>).  bits: [0,14) addr>>4 | [16,30) LBO>>4 (=1, unused) | [32,46) SBO>>4 |
//   [46,48) version = 1 | [61,64) layout = 4 (SWIZZLE_64B).
__device__ __forceinline__ uint64_t smem_desc_sw64(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
// The same descriptor split into its two words: only the low word (address field) changes between instructions, so the
// issue loop keeps one base per operand and adds byte offsets >> 4 (shared memory is < 256 KB: no carry out of [0,14)).
constexpr uint32_t DESC_HI_SW64 = (512u >> 4) | (1u << 14) | (4u << 29);
__device__ __forceinline__ uint32_t desc_lo_sw64(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ uint64_t desc_from_lo(uint32_t lo) { return ((uint64_t)DESC_HI_SW64 << 32) | (uint64_t)lo; }
// One lane of a converged warp (the lowest): the MMA warp walks its loop as a whole and only this lane issues.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile("{\n .reg .pred px;\n elect.sync _|px, 0xffffffff;\n selp.u32 %0, 1, 0, px;\n}\n" : "=r"(pred));
  return pred != 0;
}
// Instruction descriptor for kind::i8: s8 x s8 -> s32, both operands K-major, M = 128.
//   [4,6) D format = 2 (S32) | [7,10) A = 1 (signed) | [10,13) B = 1 (signed) | [17,23) N>>3 | [24,29) M>>4
__host__ __device__ constexpr uint32_t idesc_i8(int N) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((128u >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]^T, issued by ONE thread.
__device__ __forceinline__ void mma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same with the A operand read from tensor memory (128 lanes x 8 columns per 32-byte K step) instead of shared memory.
__device__ __forceinline__ void mma_i8_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// All previously issued MMAs of this thread arrive on the mbarrier when they have completed.
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}

// ---- CTA pairs (cta_group::2): the two CTAs of a cluster act as one M = 256 tensor-core tile ---------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// arrive on the mbarrier at the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n .reg .b32 ra;\n mapa.shared::cluster.u32 ra, %0, %1;\n mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n}\n" ::"r"(
          smem_u32(bar)),
      "r"(rank)
      : "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc2(uint32_t* slot_in_smem) {   // one warp (same warp id) in BOTH CTAs of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(slot_in_smem)), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "n"(COLS) : "memory");
}
// M = 256 across the pair: each CTA contributes its own 128 rows of A and half of the N rows of B (same shared-memory
// offsets in both CTAs) and receives its 128 rows of D in its own tensor memory.  Issued by the leader CTA only.
__host__ __device__ constexpr uint32_t idesc_i8_m256(int N) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((256u >> 4) << 24);
}
__device__ __forceinline__ void mma_i8_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of the pair's MMAs arrives on the mbarrier at this offset in BOTH CTAs
__device__ __forceinline__ void mma_commit_pair(uint64_t* bar) {
  asm volatile(
      "{\n .reg .b16 m;\n mov.b16 m, 3;\n tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n}\n" ::"r"(
          smem_u32(bar))
      : "memory");
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace tc
}  // namespace bocf
