// transform_pad.cuh -- the 2048-point transform of kernels.cuh with PADDED exchange buffers.
//
// kernels.cuh keeps every 16-byte shared-memory access of the exchanges conflict free with XOR
// swizzles (S1/S2), which costs one LOP3 + one LEA per access.  Here the same accesses are made
// conflict free by padding instead, so that every address is a per-thread base register plus a
// compile-time immediate:
//   a warp's 256-element block occupies 288 slots;
//   P1(e) = e + 4 (e >> 5)   (4 slots after every 32 elements)  for the exchanges of passes 1-3,
//   P2(e) = e + (e >> 3)     (1 slot after every 8 elements)    for the exchange of passes 3-4.
// Access patterns (e within the block, q = lane >> 2, r = lane & 3), quarter-warps hit 8 banks:
//   A: e = lane + 32 m        -> P1 = lane + 36 m
//   B: e = 32 q + 4 m + r     -> P1 = 36 q + r + 4 m,   P2 = 36 q + r + 4 m + (m >> 1)
//   C: e = 8 lane + j         -> P2 = 9 lane + j
//   D: block level, element T + 256 m lives in block m at P1(T) = T + 4 (T >> 5)
// Arithmetic (butterflies, twiddles, order of operations) is identical to kernels.cuh, so spectra
// and results are bit-identical and the prepared matrices are shared.
#pragma once
#include "kernels.cuh"
#include "sync.cuh"
#include "tmem.cuh"

// timing ablations for tools/ablate.sh (results are garbage when non-zero): 1 no matrix loads, 2 no inverse
// transforms, 4 no forward transforms (k_ks4), 8 no warp-local exchanges, 16 no butterflies
#ifndef FHERAM_ABL
#define FHERAM_ABL 0
#endif
#define ABL_XCH if (!(FHERAM_ABL & 8))
#define ABL_BFLY if (!(FHERAM_ABL & 16))

namespace fheram {

constexpr int kBlk = 288;            // padded slots per warp block
constexpr int kWorkPad = 8 * kBlk;   // double2 slots of one exchange buffer (36 KiB)

struct PadAddr {
  double2* A;  // block + lane
  double2* B;  // block + 36 q + r
  double2* C;  // block + 9 lane
  double2* D;  // buffer + T + 4 w
};
__device__ __forceinline__ PadAddr pad_addr(double2* work, int T, int w, int lane) {
  double2* wb = work + kBlk * w;
  PadAddr p;
  p.A = wb + lane;
  p.B = wb + 36 * (lane >> 2) + (lane & 3);
  p.C = wb + 9 * lane;
  p.D = work + T + 4 * w;
  return p;
}

struct Tw4x { double2 a, b, c, d; };  // four twiddles of one pass

// pass-3/4 twiddles of thread (w, lane) parked in tensor memory columns ttw .. ttw + 31, and their loaders
__device__ __forceinline__ void park_tw34(uint32_t ttw, const Twiddles& tw, int w, int lane) {
  const Tw34 t = load_tw34(tw, w, lane);
  const double2 p3[4] = {t.a3, t.b3, t.c3, t.d3};
  const double2 p4[4] = {t.b4a, t.b4b, t.c4a, t.c4b};
  tm_st4(ttw, p3);
  tm_st4(ttw + 16, p4);
  tm_wait_st();
}
__device__ __forceinline__ Tw4x tm_tw3(uint32_t ttw) { double2 t[4]; tm_ld4(ttw, t); return Tw4x{t[0], t[1], t[2], t[3]}; }
__device__ __forceinline__ Tw4x tm_tw4(uint32_t ttw) { double2 t[4]; tm_ld4(ttw + 16, t); return Tw4x{t[0], t[1], t[2], t[3]}; }

// Split barrier protecting the exchange buffer between transforms (write-after-read): a warp
// RELEASES the buffer (one mbarrier arrival per warp) once it has read everything it needs, and a
// thread ACQUIRES it (waits for the 8 arrivals of the previous transform) right before its first store
// of the next transform -- hundreds to thousands of cycles later, so the wait is normally free.
struct BufSync {
  uint32_t mbar;   // shared-memory address of the mbarrier (8 bytes, 8-byte aligned)
  uint32_t phase;  // parity of the phase the next acquire waits for
};
// one thread: init; then __syncthreads(); then every warp calls buf_release once (phase 0 completes)
__device__ __forceinline__ void buf_init(uint32_t mbar) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 8;" ::"r"(mbar) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void buf_release(const BufSync& b) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(b.mbar) : "memory");
}
__device__ __forceinline__ void buf_acquire(BufSync& b) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(b.mbar), "r"(b.phase) : "memory");
  b.phase ^= 1u;
}

// pass 1 on x[m] = z[T + 256 m]; result to the exchange buffer (block level); the caller issues
// __syncthreads() before fwd_warp_passes_p
__device__ __forceinline__ void fwd_pass1_store_p(double2 (&x)[8], const PadAddr& p, BufSync& bs) {
  ABL_BFLY radix8_fwd<true>(x, c_tw_lo[1], c_tw_lo[2], c_tw_lo[4], c_tw_lo[6]);
  buf_acquire(bs);
#pragma unroll
  for (int m = 0; m < 8; m++) p.D[kBlk * m] = x[m];
}
// passes 2-4 of warp w after a block-level sync; returns the 8 final frequencies of this thread
// (spectrum positions 256 w + 32 j + lane).  tw3() / tw4() deliver (a3,b3,c3,d3) / (b4a,b4b,c4a,c4b).
template <typename F3, typename F4>
__device__ __forceinline__ void fwd_warp_passes_p(const PadAddr& p, int w, F3&& tw3, F4&& tw4, double2 (&x)[8],
                                                  const BufSync& bs) {
#pragma unroll
  for (int m = 0; m < 8; m++) x[m] = p.A[36 * m];
  ABL_BFLY radix8_fwd<true>(x, c_tw_lo[8 + w], c_tw_lo[16 + 2 * w], c_tw_lo[32 + 4 * w], c_tw_lo[32 + 4 * w + 2]);
  ABL_XCH {
#pragma unroll
    for (int m = 0; m < 8; m++) p.A[36 * m] = x[m];
    __syncwarp();
#pragma unroll
    for (int m = 0; m < 8; m++) x[m] = p.B[4 * m];
  }
  {
    const Tw4x t = tw3();
    ABL_BFLY radix8_fwd<true>(x, t.a, t.b, t.c, t.d);
  }
  ABL_XCH {
    __syncwarp();
#pragma unroll
    for (int m = 0; m < 8; m++) p.B[4 * m + (m >> 1)] = x[m];
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 8; j++) x[j] = p.C[j];
  }
  buf_release(bs);
  {
    const Tw4x t = tw4();
    ABL_BFLY {
      bf(x[0], x[2], t.a); bf(x[1], x[3], t.a); bf(x[4], x[6], t.b); bf(x[5], x[7], t.b);
      bf(x[0], x[1], t.c); bf(x[2], x[3], mul_i(t.c));
      bf(x[4], x[5], t.d); bf(x[6], x[7], mul_i(t.d));
    }
  }
}
// inverse: x[j] = this thread's 8 spectrum values; on return x[m] = M z[T + 256 m].
// Buffer protocol: buf_acquire() before the first store, buf_release() after the last load.
template <typename F3, typename F4>
__device__ __forceinline__ void inv_transform_p(double2 (&x)[8], const PadAddr& p, int w, F3&& tw3, F4&& tw4,
                                                BufSync& bs) {
  {
    const Tw4x t = tw4();
    ABL_BFLY {
      ibf(x[0], x[1], t.c); ibf(x[2], x[3], mul_i(t.c));
      ibf(x[4], x[5], t.d); ibf(x[6], x[7], mul_i(t.d));
      ibf(x[0], x[2], t.a); ibf(x[1], x[3], t.a); ibf(x[4], x[6], t.b); ibf(x[5], x[7], t.b);
    }
  }
  buf_acquire(bs);
  ABL_XCH {
#pragma unroll
    for (int j = 0; j < 8; j++) p.C[j] = x[j];
    __syncwarp();
#pragma unroll
    for (int m = 0; m < 8; m++) x[m] = p.B[4 * m + (m >> 1)];
  }
  {
    const Tw4x t = tw3();
    ABL_BFLY radix8_inv<true>(x, t.a, t.b, t.c, t.d);
  }
  ABL_XCH {
    __syncwarp();
#pragma unroll
    for (int m = 0; m < 8; m++) p.B[4 * m] = x[m];
    __syncwarp();
#pragma unroll
    for (int m = 0; m < 8; m++) x[m] = p.A[36 * m];
  }
  ABL_BFLY radix8_inv<true>(x, c_tw_lo[8 + w], c_tw_lo[16 + 2 * w], c_tw_lo[32 + 4 * w], c_tw_lo[32 + 4 * w + 2]);
#pragma unroll
  for (int m = 0; m < 8; m++) p.A[36 * m] = x[m];
  __syncthreads();
#pragma unroll
  for (int m = 0; m < 8; m++) x[m] = p.D[kBlk * m];
  buf_release(bs);
  ABL_BFLY radix8_inv<true>(x, c_tw_lo[1], c_tw_lo[2], c_tw_lo[4], c_tw_lo[6]);
}

// inv_transform_p with the block barrier restricted to the group and three
// hooks in the inverse (tile prefetch points, several hundred cycles apart)
template <typename F3, typename F4, typename H>
__device__ __forceinline__ void inv_transform_g(double2 (&x)[8], const PadAddr& p, int w, int grp, F3&& tw3, F4&& tw4,
                                                BufSync& bs, H&& hook) {
  hook(0);
  {
    const Tw4x t = tw4();
    ibf(x[0], x[1], t.c); ibf(x[2], x[3], mul_i(t.c));
    ibf(x[4], x[5], t.d); ibf(x[6], x[7], mul_i(t.d));
    ibf(x[0], x[2], t.a); ibf(x[1], x[3], t.a); ibf(x[4], x[6], t.b); ibf(x[5], x[7], t.b);
  }
  buf_acquire(bs);
#pragma unroll
  for (int j = 0; j < 8; j++) p.C[j] = x[j];
  __syncwarp();
#pragma unroll
  for (int m = 0; m < 8; m++) x[m] = p.B[4 * m + (m >> 1)];
  {
    const Tw4x t = tw3();
    radix8_inv<true>(x, t.a, t.b, t.c, t.d);
  }
  hook(1);
  __syncwarp();
#pragma unroll
  for (int m = 0; m < 8; m++) p.B[4 * m] = x[m];
  __syncwarp();
#pragma unroll
  for (int m = 0; m < 8; m++) x[m] = p.A[36 * m];
  radix8_inv<true>(x, c_tw_lo[8 + w], c_tw_lo[16 + 2 * w], c_tw_lo[32 + 4 * w], c_tw_lo[32 + 4 * w + 2]);
#pragma unroll
  for (int m = 0; m < 8; m++) p.A[36 * m] = x[m];
  group_sync(grp);
#pragma unroll
  for (int m = 0; m < 8; m++) x[m] = p.D[kBlk * m];
  buf_release(bs);
  hook(2);
  radix8_inv<true>(x, c_tw_lo[1], c_tw_lo[2], c_tw_lo[4], c_tw_lo[6]);
}

}  // namespace fheram
