// sync.cuh -- synchronisation and data movement between the threads, groups and CTAs of a kernel: named barriers of a
// thread group, cluster rank / barrier / distributed shared memory, cp.async staging and shared-memory reductions.
#pragma once
#include "kernels.cuh"

namespace fheram {

// ---- named barriers (barrier 0 is __syncthreads) ----------------------------------------
// group grp of 256 threads: barrier 1 + grp
__device__ __forceinline__ void group_sync(int grp) { asm volatile("bar.sync %0, 256;" ::"r"(1 + grp) : "memory"); }
// group g of 128 threads: barrier 1 + g
__device__ __forceinline__ void gsync128(int g) { asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory"); }
// two groups of 128 threads on barrier id
__device__ __forceinline__ void pair_arrive(int id) { asm volatile("bar.arrive %0, 256;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void pair_sync(int id) { asm volatile("bar.sync %0, 256;" ::"r"(id) : "memory"); }

// ---- clusters ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
// address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_cluster_u64(uint32_t addr, unsigned long long v) {
  asm volatile("st.shared::cluster.u64 [%0], %1;" ::"r"(addr), "l"(v) : "memory");
}

// ---- cp.async ------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(const void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void cp_async_wait_n(int n) {
  switch (n) {
    case 0: cp_async_wait<0>(); break;
    case 1: cp_async_wait<1>(); break;
    case 2: cp_async_wait<2>(); break;
    case 3: cp_async_wait<3>(); break;
    case 4: cp_async_wait<4>(); break;
    case 5: cp_async_wait<5>(); break;
    case 6: cp_async_wait<6>(); break;
    case 7: cp_async_wait<7>(); break;
    case 8: cp_async_wait<8>(); break;
    case 9: cp_async_wait<9>(); break;
    default: cp_async_wait<10>(); break;
  }
}
__device__ __forceinline__ void red_add_u32(uint32_t* p, uint32_t v) {
  asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}

}  // namespace fheram
