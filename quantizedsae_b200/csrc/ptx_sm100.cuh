// Thin inline-PTX wrappers for the sm_100a features the kernels use: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld / fences) and cluster helpers.
// Bit layouts of the UMMA descriptors follow the PTX ISA tables for tcgen05 (matrix
// descriptor, instruction descriptor).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace qsae {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrive on the barrier at the same smem offset in CTA `cta` of the cluster. Default semantics (release at CTA
// scope), NOT .release.cluster: the only users signal "this warp has drained its TMEM accumulator" (ordered by
// tcgen05.wait::ld + tcgen05.fence::before_thread_sync), and a cluster-scope release makes the warp wait until every
// global store it has issued is acknowledged by L2 -- ncu showed 14 % of the dense encoder's stall samples on that
// membar (profiles/r2s2_*): the epilogue's 192 KB of stores per tile were serialised with the next tile.
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// Bounded wait: a mis-programmed pipeline must trap, never hang the GPU.
#ifndef QSAE_MBAR_TIMEOUT_CYCLES
#define QSAE_MBAR_TIMEOUT_CYCLES (4000000000ll)  // ~2 s at 2 GHz
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > QSAE_MBAR_TIMEOUT_CYCLES) {
      printf("qsae: mbarrier timeout block (%d,%d) thread %d bar %u parity %u\n", blockIdx.x,
             blockIdx.y, threadIdx.x, smem_u32(bar), parity);
      __trap();
    }
  }
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* desc) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(desc) : "memory");
}
// 2D tiled load global -> shared::cta, completion on a local mbarrier
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* desc, uint64_t* bar,
                                            int32_t c0, int32_t c1, uint64_t cache_policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(desc), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(cache_policy)
      : "memory");
}
// multicast variant: the tile lands at the same smem offset in every CTA of `mask`, and each
// destination CTA's barrier (same offset) receives the complete_tx
__device__ __forceinline__ void tma_load_2d_mcast(void* smem_dst, const void* desc, uint64_t* bar,
                                                  int32_t c0, int32_t c1, uint16_t mask,
                                                  uint64_t cache_policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      ".multicast::cluster.L2::cache_hint [%0], [%1, {%4, %5}], [%2], %3, %6;" ::"r"(
          smem_u32(smem_dst)),
      "l"(desc), "r"(smem_u32(bar)), "h"(mask), "r"(c0), "r"(c1), "l"(cache_policy)
      : "memory");
}
// 2D tiled store shared::cta -> global (bulk async-group completion). Rows / columns of the box
// that fall outside the tensor are clipped by the hardware.
__device__ __forceinline__ void tma_store_2d(const void* desc, const void* smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(desc),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed bulk stores of this thread have finished READING their shared-memory source
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
// ... and have completed entirely (writes performed)
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// L2 cache policies (createpolicy encodings used by CUTLASS' TMA::CacheHintSm90)
constexpr uint64_t kPolicyEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kPolicyEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kPolicyEvictLast = 0x14F0000000000000ull;

// ---------------------------------------------------------------- tcgen05
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::f16 (bf16/fp16 in, fp32 accumulate)
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread arrive on `bar` when complete
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void umma_commit_mcast(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;" ::"r"(smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
// 32 lanes x 32 consecutive columns (one row of the accumulator per thread)
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// the same wait, with the destination registers of the outstanding load as operands: when other work sits between
// a tcgen05.ld and its wait, this keeps the compiler from reading (or copying) r before the load has landed
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]),
                 "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]),
                 "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]),
                 "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// ---------------------------------------------------------------- tcgen05, CTA pairs (cta_group::2)
// Two CTAs of a cluster (ranks 2i, 2i+1, same TPC) execute one MMA of M = 256: each holds its own
// 128 rows of A and half of the N columns of B in shared memory at identical offsets, each receives
// its 128 accumulator rows in its own TMEM. Only the leader (even rank) issues MMA and commit.
template <int kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_result) {   // one warp in EACH CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void umma_f16_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at this offset in every CTA of cta_mask when the pair's MMAs complete
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;" ::"r"(smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
// shared::cluster address of `local_addr` (a shared::cta address of this CTA) in CTA `rank`
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
// TMA load issued by either CTA of a pair; the completion bytes are credited to `bar_cluster_addr`,
// which may live in the peer CTA (the leader's "stage full" barrier)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const void* desc, uint32_t bar_cluster_addr,
                                                 int32_t c0, int32_t c1, uint64_t cache_policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(desc), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "l"(cache_policy)
      : "memory");
}

// K-major, 128-byte swizzled operand tile: rows of 128 B (64 bf16), 8-row atoms of 1024 B.
//   [0,14) start address >> 4 | [16,30) LBO >> 4 (unused with swizzle, 1) |
//   [32,46) SBO >> 4 = 1024 >> 4 | [46,48) version = 1 | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_desc_kmajor_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// MN-major, 128-byte swizzled operand tile: each K index is one row of 64 MN-consecutive bf16 (128 B), 8-row atoms
// of 1024 B (the layout a {64 x rows} TMA box of a row-major [K, MN] tensor lands in with SWIZZLE_128B).
//   [16,30) LBO >> 4: byte distance between consecutive 64-element MN columns of atoms |
//   [32,46) SBO >> 4: byte distance between consecutive groups of 8 K rows (1024 for a contiguous column)
// A K step of 16 rows advances the start address by 2 SBO.
__device__ __forceinline__ uint64_t umma_desc_mnmajor_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, dense
__host__ __device__ constexpr uint32_t umma_idesc_bf16_f32(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
// the same with the transpose bits: bit 15 = A is MN-major, bit 16 = B is MN-major
__host__ __device__ constexpr uint32_t umma_idesc_bf16_f32_major(int M, int N, bool a_mn, bool b_mn) {
  return umma_idesc_bf16_f32(M, N) | (a_mn ? (1u << 15) : 0u) | (b_mn ? (1u << 16) : 0u);
}

// ---------------------------------------------------------------- cluster
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// load one float from the shared memory of CTA `rank` of the cluster, at the offset of this CTA's `local_addr`
__device__ __forceinline__ float ld_dsmem_f32(uint32_t local_addr, uint32_t rank) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(mapa_u32(local_addr, rank)) : "memory");
  return v;
}

// ---------------------------------------------------------------- misc
// monotone map float -> uint32 (larger float <=> larger key); -0.0 < +0.0, NaNs sort by payload
__device__ __forceinline__ uint32_t float_to_key(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_to_float(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

}  // namespace qsae
