// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM).
// Everything here is device-only and header-only; no CUTLASS/CuTe dependency.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace av2v {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 rx;\n"
      ".reg .pred px;\n"
      "elect.sync rx|px, 0xffffffff;\n"
      "selp.b32 %0, 1, 0, px;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// make generic-proxy smem writes visible to the async proxy (TMA / tcgen05 operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug must trap, never hang the GPU.
#ifndef AV2V_WAIT_TIMEOUT_CYCLES
#define AV2V_WAIT_TIMEOUT_CYCLES (4000000000ll)
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > AV2V_WAIT_TIMEOUT_CYCLES) {
      printf("av2v: mbarrier wait timeout (block %d,%d thread %d bar %u parity %u)\n", blockIdx.x, blockIdx.y,
             threadIdx.x, smem_u32(bar), parity);
      __trap();
    }
  }
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// 2-D tiled load multicast to the CTAs in `cta_mask` of this cluster: the box lands at the same smem offset in each
// destination CTA and completes `bytes` on the mbarrier at the same offset in each of them.
__device__ __forceinline__ void tma_load_2d_mc(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                               uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, "
      "%4}], [%2], %5;" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(cta_mask)
      : "memory");
}
// ---- CTA-pair (cta_group::2) helpers
__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA loads into this CTA's smem whose completion bytes are signalled on a barrier of the pair's LEADER CTA
__device__ __forceinline__ void tma_load_2d_cg2(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_cg2(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1,
                                                int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
      "%5}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_cg2(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1,
                                                int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
      "%5, %6}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
template <int kPending>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPending) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read0() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ------------------------------------------------------------------ tcgen05 / TMEM
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {  // whole warp (the allocating one)
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all prior tcgen05.mma of this thread complete -> arrive(1) on mbarrier
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---- warp-convergent issue: EVERY lane of the issuing warp executes these with warp-uniform operands and `lead` true
// in one elected lane, which alone issues.  The operands then live in uniform registers; under a divergent
// `if (lane == 0)` the compiler wraps every UTCHMMA / UTCBAR in an ELECT + R2UR.BROADCAST + BRA.U.ANY "waterfall"
// loop that costs ~90 cycles per instruction (measured: the attention MMA thread spent 1800 of 2300 cycles per key
// tile issuing 16 MMAs — profiles/README.md).
__device__ __forceinline__ void umma_ss_w(uint32_t lead, uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p, q;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "setp.ne.b32 q, %5, 0;\n"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void umma_ts_w(uint32_t lead, uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p, q;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "setp.ne.b32 q, %5, 0;\n"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void umma_commit_w(uint32_t lead, uint64_t* bar) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %1, 0;\n"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n}\n" ::"r"(smem_u32(bar)),
      "r"(lead)
      : "memory");
}
__device__ __forceinline__ void umma_commit_mc_w(uint32_t lead, uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %2, 0;\n"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n}\n" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void umma_ss_cg2_w(uint32_t lead, uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p, q;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "setp.ne.b32 q, %5, 0;\n"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void umma_commit_cg2_mc_w(uint32_t lead, uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %2, 0;\n"
      "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n}\n" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask), "r"(lead)
      : "memory");
}

// ---- warp-convergent TMA / mbarrier issue (see umma_*_w above): uniform operands, one elected lane issues
__device__ __forceinline__ void mbar_arrive_expect_tx_w(uint32_t lead, uint64_t* bar, uint32_t bytes) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %2, 0;\n"
      "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n}\n" ::"r"(smem_u32(bar)), "r"(bytes), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_w(uint32_t lead, void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %5, 0;\n"
      "@q cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n}\n" ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_w(uint32_t lead, void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %6, 0;\n"
      "@q cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n}\n" ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_w(uint32_t lead, void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %7, 0;\n"
      "@q cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n}\n" ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_cg2_w(uint32_t lead, void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %5, 0;\n"
      "@q cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n}\n" ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_cg2_w(uint32_t lead, void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1, int c2) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %6, 0;\n"
      "@q cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n}\n" ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_cg2_w(uint32_t lead, void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1, int c2, int c3) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %7, 0;\n"
      "@q cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n}\n" ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_mc_w(uint32_t lead, void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, uint16_t cta_mask) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %6, 0;\n"
      "@q cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;\n}\n" ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(cta_mask), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void tma_store_3d_w(uint32_t lead, const CUtensorMap* m, const void* src, int c0, int c1, int c2) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %5, 0;\n"
      "@q cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];\n}\n" ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(lead)
      : "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx_w(uint32_t lead, uint32_t bar_addr, uint32_t bytes) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %2, 0;\n"
      "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n}\n" ::"r"(bar_addr), "r"(bytes), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_w(uint32_t lead, uint32_t dst_addr, const CUtensorMap* m, uint32_t bar_addr, int c0,
                                              int c1, int c2) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %6, 0;\n"
      "@q cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n}\n" ::"r"(
          dst_addr),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_addr), "r"(c0), "r"(c1), "r"(c2), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void tma_store_3d_w(uint32_t lead, const CUtensorMap* m, uint32_t src_addr, int c0, int c1, int c2) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %5, 0;\n"
      "@q cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];\n}\n" ::"l"(
          reinterpret_cast<uint64_t>(m)),
      "r"(src_addr), "r"(c0), "r"(c1), "r"(c2), "r"(lead)
      : "memory");
}

// 5-D tiled load (the residual block of a conv tile: channels x columns x rows x frames x slot)
__device__ __forceinline__ void tma_load_5d_w(uint32_t lead, uint32_t dst_addr, const CUtensorMap* m, uint32_t bar_addr, int c0,
                                              int c1, int c2, int c3, int c4) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %8, 0;\n"
      "@q cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];\n}\n" ::"r"(
          dst_addr),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(lead)
      : "memory");
}

// 5-D tiled store: a conv tile's block of pixels (channels x columns x rows x frames x slot), or with nearest-up x 2 fused into
// the conv, every second pixel / row of the output image
__device__ __forceinline__ void tma_store_5d_w(uint32_t lead, const CUtensorMap* m, uint32_t src_addr, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "{\n.reg .pred q;\n"
      "setp.ne.b32 q, %7, 0;\n"
      "@q cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];\n}\n" ::"l"(
          reinterpret_cast<uint64_t>(m)),
      "r"(src_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(lead)
      : "memory");
}

// cta_group::2 TMEM allocation: one warp in EACH CTA of the pair executes it
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
// D[tmem of both CTAs, 256 rows] (+)= A[smem, 128 rows per CTA] * B[smem, N/2 rows per CTA]; issued by the leader CTA only
__device__ __forceinline__ void umma_ss_cg2(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_cg2_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}

// ... and arrive(1) on the mbarrier at the same smem offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}

// Instruction descriptor, kind::f16, fp16 A/B, fp32 accumulate (cute/arch/mma_sm100_desc.hpp InstrDescriptor).
__host__ __device__ constexpr uint32_t make_idesc_f16(uint32_t M, uint32_t N, uint32_t a_mn_major,
                                                      uint32_t b_mn_major) {
  return (1u << 4)                    // c_format = F32
         | (0u << 7) | (0u << 10)     // a/b format = F16
         | (a_mn_major << 15) | (b_mn_major << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
// Shared-memory matrix descriptor (SmemDescriptor, version 1). Offsets are in bytes; layout_type 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t make_sdesc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                               uint32_t layout_type = 2u) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;  // version = 1 (Blackwell)
  d |= static_cast<uint64_t>(layout_type & 7u) << 61;
  return d;
}

// TMEM -> registers: this thread's lane (32*(warp%4)+lane), 32 consecutive fp32 columns.
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
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// registers -> TMEM, 16 consecutive 32-bit columns of this thread's lane
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}


// 2^x for x <= ~9 on the FMA pipe: x = n + f, n = round(x), f in [-0.5, 0.5]; 2^f by a degree-3 minimax polynomial
// (relative error < 7.5e-5, fitted in tools/exp2_poly_fit.py); 2^n by adding n to the exponent field.
__device__ __forceinline__ float ex2_poly(float x) {
  x = fmaxf(x, -125.0f);              // masked keys arrive as -inf; 2^-125 packs to 0 in fp16.  NOT lower: p can be just
                                      // below 1 (exponent 126), so n = -127 would wrap the exponent field into NaN
  const float t = x + 12582912.0f;    // 1.5 * 2^23: the integer n = round(x) lands in the low mantissa bits
  const float f = x - (t - 12582912.0f);
  float p = fmaf(f, 0.05517164245247841f, 0.2426111251115799f);
  p = fmaf(p, f, 0.6932609677314758f);
  p = fmaf(p, f, 0.9999280571937561f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(t) << 23));
}

// ---- packed fp32x2 arithmetic (FFMA2 / FADD2 on sm_100): two elements per issue slot.  The softmax loops are bounded by
// MUFU (ex2) and, once exponentials move to the FMA pipe, by instruction issue (profiles/r01_static_sass_analysis.txt).
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("{\n.reg .b64 ra, rb, rc, rd;\n"
      "mov.b64 ra, {%2, %3};\nmov.b64 rb, {%4, %5};\nmov.b64 rc, {%6, %7};\n"
      "fma.rn.f32x2 rd, ra, rb, rc;\n"
      "mov.b64 {%0, %1}, rd;\n}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  float2 d;
  asm("{\n.reg .b64 ra, rb, rd;\nmov.b64 ra, {%2, %3};\nmov.b64 rb, {%4, %5};\nadd.rn.f32x2 rd, ra, rb;\nmov.b64 {%0, %1}, rd;\n}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  float2 d;
  asm("{\n.reg .b64 ra, rb, rd;\nmov.b64 ra, {%2, %3};\nmov.b64 rb, {%4, %5};\nmul.rn.f32x2 rd, ra, rb;\nmov.b64 {%0, %1}, rd;\n}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}
// ex2_poly on two elements (same arithmetic per element, so tools/exp2_poly_fit.py covers it)
__device__ __forceinline__ float2 ex2_poly2(float2 x) {
  x.x = fmaxf(x.x, -125.0f);
  x.y = fmaxf(x.y, -125.0f);
  const float2 magic = make_float2(12582912.0f, 12582912.0f);
  const float2 t = fadd2(x, magic);
  const float2 n = fadd2(t, make_float2(-12582912.0f, -12582912.0f));
  const float2 f = ffma2(n, make_float2(-1.0f, -1.0f), x);
  float2 p = ffma2(f, make_float2(0.05517164245247841f, 0.05517164245247841f), make_float2(0.2426111251115799f, 0.2426111251115799f));
  p = ffma2(p, f, make_float2(0.6932609677314758f, 0.6932609677314758f));
  p = ffma2(p, f, make_float2(0.9999280571937561f, 0.9999280571937561f));
  return make_float2(__int_as_float(__float_as_int(p.x) + (__float_as_int(t.x) << 23)),
                     __int_as_float(__float_as_int(p.y) + (__float_as_int(t.y) << 23)));
}

}  // namespace av2v
