// sm_100a primitives used by the tcgen05 kernels: mbarrier, bulk async copy (TMA engine, 1-D),
// TMEM allocation, UMMA descriptors / issue / commit, TMEM loads.  Inline PTX only.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace dvq {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier ----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
// try_wait with an explicit suspend-time hint: the thread sleeps in hardware until the phase completes
// (or the hint expires) instead of spinning — a polling loop without it returns every few dozen cycles
// and was measured to eat ~40 % of the SM's issue slots in the warp-specialised VQ kernel.
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity), "r"(100000u)   // ns
      : "memory");
  return done != 0;
}
// Bounded wait: a protocol bug must never hang the GPU.  On timeout the caller's error word is
// set and the wait returns false; every role then drains out of its loops.
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, volatile int* err_word, int code) {
  for (uint32_t spin = 0; spin < (1u << 20); ++spin) {
    if (mbar_try_wait(bar, parity)) return true;
    if ((spin & 63u) == 63u && *err_word != 0) return false;
  }
  *err_word = code;
  return false;
}

// ---- async proxy --------------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {  // st.shared -> visible to UMMA / bulk copies
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// 1-D bulk copy global -> shared (TMA engine), completion on an mbarrier via complete_tx
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// same, with an L2 evict_last policy: the tile is read again a few microseconds later
__device__ __forceinline__ void bulk_g2s_keep(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  uint64_t policy;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(policy));
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
               : "memory");
}

// ---- TMEM ---------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // same warp as alloc
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 32 lanes x 32 consecutive columns -> 32 registers per thread (thread = TMEM lane = tile row)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 0 -> 32 lanes x 32 consecutive columns (thread = TMEM lane); complete with tmem_st_wait() before reading them back
__device__ __forceinline__ void tmem_st32_zero(uint32_t taddr) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
      "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(0u)
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// the same wait carrying a register dependence on the loaded values, so that the compiler cannot schedule their
// consumers above it
__device__ __forceinline__ void tmem_ld_wait_dep32(uint32_t (&v)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                 "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
                 "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
                 "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
               :
               : "memory");
}

// ---- UMMA ---------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, K-major, no swizzle ("interleave"): 8 rows x 16 bytes core
// matrices whose rows are 16 B apart; core matrices LBO bytes apart along K and SBO bytes apart
// along M/N (bit layout: cute/arch/mma_sm100_desc.hpp, SmemDescriptor).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version 1 (Blackwell)
  return d;                // base_offset 0, lbo_mode 0, layout_type 0 (SWIZZLE_NONE)
}
// Instruction descriptor, kind::f16, A/B = F16 (0) or BF16 (1), D = F32, both K-major.
__host__ __device__ constexpr uint32_t make_idesc_f16(int m, int n, int ab_format) {
  return (1u << 4) | ((uint32_t)ab_format << 7) | ((uint32_t)ab_format << 10) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives when every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- the same primitives on 32-bit shared-window addresses ------------------------------------------
// (a kernel that keeps all its barriers in one shared struct addresses them as base + constant, which
//  saves the generic->shared conversion (S2R + LEA) at every arrive / wait site)
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx_a(uint32_t bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_a(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity), "r"(100000u)
      : "memory");
  return done != 0;
}
__device__ __forceinline__ int lds_volatile_a(uint32_t addr) {
  int v;
  asm volatile("ld.volatile.shared::cta.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_volatile_a(uint32_t addr, int v) {
  asm volatile("st.volatile.shared::cta.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
// bounded wait, lean fast path: one try_wait + branch when the phase has already completed; the error
// word is polled only every 64 failed tries
__device__ __forceinline__ bool mbar_wait_a(uint32_t bar, uint32_t parity, uint32_t err_addr, int code) {
  if (mbar_try_wait_a(bar, parity)) return true;
#pragma unroll 1
  for (uint32_t spin = 1; spin < (1u << 18); ++spin) {
    if (mbar_try_wait_a(bar, parity)) return true;
    if ((spin & 63u) == 0u && lds_volatile_a(err_addr) != 0) return false;
  }
  sts_volatile_a(err_addr, code);
  return false;
}
__device__ __forceinline__ void bulk_g2s_a(uint32_t smem_dst, const void* gmem_src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst),
               "l"(gmem_src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void bulk_g2s_keep_a(uint32_t smem_dst, const void* gmem_src, uint32_t bytes, uint32_t bar) {
  uint64_t policy;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(policy));
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_dst),
               "l"(gmem_src), "r"(bytes), "r"(bar), "l"(policy)
               : "memory");
}
// 2-D tiled TMA load (tensor map built by cuTensorMapEncodeTiled, passed as a __grid_constant__ kernel parameter):
// the box at element coordinates (c0 = innermost, c1) lands densely in shared memory, out-of-bounds elements as zeros;
// the mbarrier receives the full box byte count
__device__ __forceinline__ void tma_load_2d_a(uint32_t smem_dst, const void* tmap, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(smem_dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_load_2d_keep_a(uint32_t smem_dst, const void* tmap, int c0, int c1, uint32_t bar) {   // L2 evict_last
  uint64_t policy;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(policy));
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
               ::"r"(smem_dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void umma_commit_a(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// ---- CTA pair (cta_group::2): the two CTAs of a cluster on the two SMs of a TPC run ONE M = 256 MMA -----------------
// Each CTA supplies its own 128 rows of A and its own HALF of the B block (N / 2 codes) from its shared memory, at the same
// offsets; each CTA's TMEM receives its 128 rows x N columns.  Only a thread of the even CTA (cluster rank 0) issues;
// completion is committed to the same barrier offset in both CTAs (multicast).  (Operand split: cute/atom/mma_traits_sm100.hpp,
// SM100_MMA_F16BF16_2x1SM_SS: ALayout / BLayout / CLayout.)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t smem_addr, uint32_t cta_rank) {   // shared::cta address -> that CTA's shared::cluster address
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_bar_addr) {   // release at cluster scope
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar_addr) : "memory");
}
// 2-D tiled TMA load issued by either CTA of a pair into its OWN shared memory, completing (complete_tx) on an mbarrier that
// may live in the peer CTA (`bar_cluster` = shared::cluster address, e.g. the leader's barrier for both halves of an operand)
__device__ __forceinline__ void tma_load_2d_pair_a(uint32_t smem_dst, const void* tmap, int c0, int c1, uint32_t bar_cluster) {
  asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(smem_dst), "l"(tmap), "r"(bar_cluster), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint32_t cluster_bar_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_slot, uint32_t ncols) {  // one full warp of EACH CTA of the pair, same slot offset
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs of the pair once every MMA issued so far has completed
__device__ __forceinline__ void umma_commit_pair_a(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3)
               : "memory");
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

}  // namespace tc
}  // namespace dvq
