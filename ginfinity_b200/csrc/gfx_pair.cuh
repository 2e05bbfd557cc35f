// Inline-PTX wrappers for CTA pairs (thread-block clusters of two, tcgen05 cta_group::2):
// cluster rank and barrier, remote mbarrier arrives, paired TMEM allocation, M = 256 MMAs over
// both CTAs' tiles with multicast completion, register reallocation between warpgroups; and the
// host-side count of CTA pairs a GPU holds at once.
#pragma once
#include <stdint.h>

#include "gfx_common.cuh"
#include "gfx_umma.cuh"

namespace gfx {
namespace ptx {

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n"
               "barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same location in CTA `rank`
__device__ __forceinline__ uint32_t map_to_cta(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
// Arrive on a barrier of another CTA of the cluster.  Default semantics (release at CTA scope),
// as CUTLASS's ClusterBarrier::arrive does: what the arrival publishes is consumed by the tensor
// core (shared memory through the async proxy after fence.proxy.async, or TMEM after
// tcgen05.fence), never through the waiting thread's L1.  The cluster-scope forms cost a
// MEMBAR + ERRBAR per arrive and a CCTL.IVALL (L1 invalidate) per wait: 30 % of all stall
// samples in the first version of this kernel.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t *dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void mma2_f16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma2_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on `bar` (same offset in both CTAs of the pair) when all MMAs issued so far are done
__device__ __forceinline__ void mma2_commit(uint64_t *bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::
          "r"(smem_u32(bar)),
      "h"(uint16_t(3))
      : "memory");
}
// Register reallocation between warpgroups (4 consecutive warps): the launch gives every thread
// 64 registers (1024 threads); the utility warpgroup needs far fewer and the producers a few more.
template <int N>
__device__ __forceinline__ void reg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void reg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}

}  // namespace ptx

// *cap = how many CTA pairs of Kernel (2-CTA clusters of `threads` threads with `smem` bytes of
// dynamic shared memory) the current GPU holds at once, at most one per TPC.  Persistent pair
// kernels launch no more than that: which SMs are fused off differs from chip to chip, and a pair
// that does not fit waits for a whole wave to finish.  Asked once per kernel and device (a
// template instance per kernel, so two instantiations of one kernel template with different
// shared memory keep separate answers); one pair per TPC when the query fails.
template <auto Kernel>
int resident_pairs(int threads, int smem, int *cap) {
  static int resident[64] = {};                   // per device; 0 = not asked yet
  int device = 0;
  GFX_CUDA(cudaGetDevice(&device));
  if (device >= 0 && device < 64 && resident[device] == 0) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kNumSMs, 1, 1);
    cfg.blockDim = dim3(threads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2;
    attr.val.clusterDim.y = 1;
    attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    int max_clusters = 0;
    if (cudaOccupancyMaxActiveClusters(&max_clusters, Kernel, &cfg) != cudaSuccess || max_clusters < 1) {
      (void)cudaGetLastError();
      max_clusters = kNumSMs / 2;
    }
    resident[device] = max_clusters < kNumSMs / 2 ? max_clusters : kNumSMs / 2;
  }
  *cap = device >= 0 && device < 64 ? resident[device] : kNumSMs / 2;
  return GFX_OK;
}

}  // namespace gfx
