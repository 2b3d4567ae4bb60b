// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk[.tensor]), tcgen05 (MMA, TMEM).
// Written for this project; instruction syntax follows the PTX ISA 8.7 forms for sm_100a.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace abc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// Warp-uniform helpers: role code is executed by whole warps with warp-uniform control flow so that the compiler keeps
// descriptors / barrier addresses in uniform registers; only the issuing instruction itself is predicated on one lane.
__device__ __forceinline__ uint32_t warp_id_uniform() { return __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0); }
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, px;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(bar),
               "r"(bytes)
               : "memory");
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
// Bounded wait: a protocol bug traps (-> CUDA error on the host) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) {
      printf("abcnet: mbarrier timeout (block %d,%d thread %d bar 0x%x parity %u)\n", blockIdx.x, blockIdx.y,
             threadIdx.x, bar, parity);
      __trap();
    }
  }
}

// ----------------------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* desc) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(desc)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* desc, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar)
               : "memory");
}

// ----------------------------------------------------------------------------- tcgen05 / TMEM
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst) {   // whole warp
  const uint32_t ncols = kCols;
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {    // whole warp
  const uint32_t ncols = kCols;
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]; single thread issues on behalf of the CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same, descriptors given as (lo, hi) 32-bit halves so that the issuing thread only does 32-bit address arithmetic.
__device__ __forceinline__ void umma_bf16_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: A is M = 128 lanes (one row each) x K / 2 columns, two 16-bit elements per 32-bit column
// (the lower half holds the even K index), so a K step of 16 advances the A address by 8 columns.
__device__ __forceinline__ void umma_16_ts(uint32_t tmem_d, uint32_t tmem_a, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrive when all previously issued tcgen05 ops of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32-bit, 16 consecutive columns: thread i <- TMEM lane (lane_base + i), columns [c, c+16)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// the inverse: thread i -> TMEM lane (lane_base + i), columns [c, c+16); complete after tmem_st_wait()
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// barrier among `threads` threads (whole warps) of the CTA; id 0 is __syncthreads
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// ----------------------------------------------------------------------------- CTA pair (cta_group::2)
// Two CTAs of a (2,1,1) cluster sit on the two SMs of one TPC and execute ONE tcgen05.mma with M = 256: each CTA holds
// its own 128 rows of A and of the accumulator, and HALF of the B operand (N / 2 rows); the instruction is issued by one
// thread of the even ("leader") CTA. Halves the per-SM shared-memory operand traffic and the L2 -> SM weight stream.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t smem_dst) {   // one whole warp in EACH CTA of the pair
  const uint32_t ncols = kCols;
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  const uint32_t ncols = kCols;
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_lohi_pair(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                    uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the mbarrier at this offset in BOTH CTAs of the pair when all previously issued tcgen05 ops have completed
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(mask)
               : "memory");
}

// Shared-memory matrix descriptor, SWIZZLE_NONE ("interleave") canonical layouts:
//   K-major  : core matrix = 8 rows (M/N) x 16 bytes (8 bf16 along K), 128 contiguous bytes;
//              LBO = byte distance between core matrices adjacent in K,
//              SBO = byte distance between 8-row groups adjacent in M/N.
//   MN-major : core matrix = 8 K-rows x 16 bytes (8 bf16 along M/N);
//              LBO = distance between 8-K groups, SBO = distance between 8-element M/N groups.
// Bits: [0,14) start>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version=1 (sm_100), [61,64) layout=0.
__device__ __forceinline__ uint64_t umma_desc_hi(uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16) | (static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32) |
         (1ull << 46);
}
__device__ __forceinline__ uint64_t umma_desc(uint64_t hi, uint32_t smem_addr) {
  return hi | static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
}
// K-major operand in the 128-byte swizzle layout: one row = 64 bf16 (128 B), 8-row groups of 1024 B (SBO), the 16-byte
// chunk c of row r stored at chunk position c ^ (r % 8); the block must start on a 1024-byte boundary. A K step of 16
// elements advances the start address by 32 bytes. layout type (bits 61..63) = 2.
__device__ __forceinline__ uint64_t umma_desc_hi_sw128() {
  return (static_cast<uint64_t>(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// Instruction descriptor for kind::f16, BF16 x BF16 -> FP32.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn_major) << 15) |
         (static_cast<uint32_t>(b_mn_major) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
// Same with the 16-bit operand format as a parameter: A / B format fields (bits 7-9, 10-12) 0 = FP16, 1 = BF16; D = FP32.
__host__ __device__ constexpr uint32_t umma_idesc_16(int M, int N, int a_mn_major, int b_mn_major, bool fp16) {
  return umma_idesc_bf16(M, N, a_mn_major, b_mn_major) & ~(fp16 ? ((1u << 7) | (1u << 10)) : 0u);
}

}  // namespace abc
