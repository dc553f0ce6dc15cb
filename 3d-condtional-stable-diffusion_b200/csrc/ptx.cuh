// Inline-PTX wrappers for the sm_100a features the kernels use: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (alloc / mma / commit / ld / fences).  Every wait is bounded by a clock64 watchdog so a wrong
// descriptor shows up as a flag, never as a hung GPU.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// one lane of the (converged) warp: lets the compiler issue tcgen05 / TMA without per-lane serialisation loops
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
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
// Bounded wait: false (and *flag = code) after ~8e9 cycles (~4 s: longer than any stall a healthy launch can see; a real deadlock still surfaces as an error code instead of a hang).
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity, int* flag, int code) {
  if (mbar_try_wait(bar, parity)) return true;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 8000000000LL) {
      if (flag) atomicExch(flag, code);
      return false;
    }
  }
  return true;
}
// The same wait for roles that are NOT on the critical path (producers, epilogue and transform warps): between polls the warp sleeps,
// so it does not compete for issue slots with the one warp per sub-partition that paces the kernel (a spinning try_wait loop is ~6
// instructions per poll: four spinners per sub-partition left the MMA-issuing / transforming warp a fifth of the issue slots).
__device__ __forceinline__ bool mbar_wait_sleep(uint32_t bar, uint32_t parity, int* flag, int code, unsigned ns = 64) {
  if (mbar_try_wait(bar, parity)) return true;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(ns);
    if (clock64() - t0 > 8000000000LL) {
      if (flag) atomicExch(flag, code);
      return false;
    }
  }
  return true;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::
          "r"(dst),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// TMA store of a 5-D box from shared memory (bulk async-group completion)
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::
                   "l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed bulk groups of this thread have finished READING shared memory (the staging may be reused / the CTA may exit)
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

__device__ __forceinline__ void bulk_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

// ---------------------------------------------------------------- thread-block clusters
__device__ __forceinline__ uint32_t cluster_ctaid_x() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctaid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {  // every thread of every CTA of the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// The cluster barrier at a kernel's tail orders EXECUTION only (no CTA exits / frees TMEM while its peer may still touch it): every
// memory effect that matters has been waited for before (tcgen05.wait::ld, mbarrier phases, bulk-group reads), so the arrival needs no
// release fence.
// (The same form after barrier initialisation: fence.mbarrier_init.release.cluster has already published the barriers.)
__device__ __forceinline__ void cluster_sync_exit() {
  asm volatile("barrier.cluster.arrive.relaxed.aligned;\n\tbarrier.cluster.wait.aligned;" ::: "memory");
}
// distributed shared memory: address of `local_smem_addr` in CTA `rank` of the cluster, and a 4-byte load from it
__device__ __forceinline__ uint32_t mapa_shared(uint32_t local_smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ float ld_dsmem_f32(uint32_t cluster_addr) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(cluster_addr) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_dsmem_f32x4(uint32_t cluster_addr) {
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(cluster_addr) : "memory");
  return v;
}
// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::f16 (bf16 in, fp32 accumulate); one thread issues.
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 16 consecutive fp32 columns -> 16 registers per thread (thread = lane = row)
__device__ __forceinline__ void tc_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// ---------------------------------------------------------------- CTA pairs (cta_group::2): one MMA over two SMs
// The leader CTA (cluster rank 0) issues M = 256 MMAs whose A rows 0-127 / 128-255 and B rows 0-N/2-1 / N/2-N-1 come from the
// same shared-memory offsets of the two CTAs; D rows land in each CTA's own TMEM.  TMA loads of either CTA signal the
// LEADER's mbarrier; tcgen05.commit multicasts its arrive to the same barrier offset in both CTAs.
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t smem_dst, uint32_t ncols) {  // one whole warp in EACH CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_cg2() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_mma_f16_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_commit_cg2(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask)
               : "memory");
}
// TMA loads whose completion is signalled on an mbarrier that may live in the peer CTA (`bar` = shared::cluster address)
__device__ __forceinline__ void tma_load_5d_cg2(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::
          "r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_cg2(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::
          "r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {   // arrive on an mbarrier of any CTA of the cluster
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}

// SM100 UMMA shared-memory matrix descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor):
//  [0,14) start>>4  [16,30) LBO>>4  [32,46) SBO>>4  [46,48) version=1  [49,52) base_offset  [61,64) layout
constexpr uint64_t kLayoutSw128 = 2;
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                   uint64_t layout, uint32_t base_offset = 0) {
  return (uint64_t)((addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | ((uint64_t)(base_offset & 7u) << 49) |
         (layout << 61);
}
// Instruction descriptor, kind::f16: c=F32 (bit4), a/b format at bits 7 / 10 (0 = F16, 1 = BF16: the library's 16-bit
// storage type, common.cuh), K-major both, N>>3 @17, M>>4 @24.
#ifdef B200DM_ACT_FP16
constexpr uint32_t kIdescAB = 0u;
#define kTmapAct16 CU_TENSOR_MAP_DATA_TYPE_FLOAT16
#else
constexpr uint32_t kIdescAB = (1u << 7) | (1u << 10);
#define kTmapAct16 CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
#endif
__host__ __device__ constexpr uint32_t make_idesc_act(int m, int n) {
  return (1u << 4) | kIdescAB | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

}  // namespace ptx
