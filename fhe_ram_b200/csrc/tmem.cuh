// tmem.cuh -- tensor memory as LANE-PRIVATE scratch (tcgen05.st / tcgen05.ld, no MMA involved): where the key-switch
// and external-product kernels park spectra, twiddles and matrix tiles.  Allocation, release and the fence / barrier /
// fence handoff that orders tensor-memory accesses across a CTA barrier.
#pragma once
#include "kernels.cuh"

namespace fheram {

// one warp: allocate NCOLS columns (base address to *slot in shared memory) and give up the allocation permit
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(NCOLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
// CTA barrier with the tensor-memory accesses before it ordered against those after it
__device__ __forceinline__ void tmem_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// end of the kernel: every thread is done with tensor memory, then the allocating warp frees the columns
template <int NCOLS>
__device__ __forceinline__ void tmem_free(uint32_t base, bool alloc_warp) {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (alloc_warp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(NCOLS) : "memory");
}

__device__ __forceinline__ void tm_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// 16 consecutive 32-bit columns of this thread's TMEM lane <-> 4 double2
__device__ __forceinline__ void tm_st4(uint32_t taddr, const double2 (&v)[4]) {
  uint32_t r[16];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    r[4 * j] = (uint32_t)__double2loint(v[j].x); r[4 * j + 1] = (uint32_t)__double2hiint(v[j].x);
    r[4 * j + 2] = (uint32_t)__double2loint(v[j].y); r[4 * j + 3] = (uint32_t)__double2hiint(v[j].y);
  }
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tm_ld4(uint32_t taddr, double2 (&v)[4]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  tm_wait_ld();
#pragma unroll
  for (int j = 0; j < 4; j++) {
    v[j].x = __hiloint2double((int)r[4 * j + 1], (int)r[4 * j]);
    v[j].y = __hiloint2double((int)r[4 * j + 3], (int)r[4 * j + 2]);
  }
}

}  // namespace fheram
