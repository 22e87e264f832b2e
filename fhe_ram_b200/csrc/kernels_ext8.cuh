// kernels_ext8.cuh -- external-product chains (CoordinatePrepared::product / product_inplace,
// src/coordinate_prepared.rs:147-177) on the TWO-EXCHANGE transform of kernels_ks7.cuh, ONE ciphertext per SM.
//
// The round-1 kernel (k_ext3, since retired) ran its 14 transforms one after the other on 256 threads x 8 points
// (three shared-memory exchanges each), kept two of the six input spectra in shared memory (read back 8 times)
// and waited one L2 round trip per 32 KiB matrix tile.  Here one CTA of 512 threads = FOUR groups of 128
// threads owns the SM and one ciphertext:
//   forward     rows rho = 2 limb + col of the input: group g transforms rows g and g + 4 (16 points per thread,
//               passes of 4 + 4 + 3 stages, private 34 KiB exchange buffer per group, no lock);
//               ALL six spectra live in tensor memory (6 x 64 columns; thread t of every group is tensor-memory
//               lane t, so a spectrum written by one group is read by the three others without an exchange)
//   contraction group g owns output column g & 1, limbs {3, 2} (g < 2) or {1, 0}: per output 24 chunks of
//   + inverse   4 frequencies x 6 rows, the matrix chunk of step c + 1 in flight while chunk c is multiplied
//               (the tile stream never drains: no round trip per tile), then inverse16 and the word update
//   words       the ciphertext between the steps of a chain stays on chip as 51-bit words (kernels_ks3.cuh),
//               kept as two 32-bit halves lo = W mod 2^26 (+ carries), hi = W >> 26 (+ carries) with
//               W = lo + hi 2^26 (mod 2^51): the limb-3 group STORES its contribution (+ bias), the three other
//               contributions of the column are added with native 32-bit shared atomics (no return value, no
//               64-bit CAS loop, order free); every sum stays below 2^28.  The digits are bit fields of (lo, hi).
// Same integers as k_ext9 and the oracle's external product; the prepared GGSWs are in the frequency order of k_prepare7.
// Shared memory 4 (pass-2 twiddles) + 4 x 34 (exchange) + 64 (words) = 204 KiB, 512 tensor-memory columns.
#pragma once
#include "kernels_ks7.cuh"

// groups 2, 3 start contracting rows 0..3 while groups 0, 1 transform rows 4, 5 (0: all groups wait for the six rows)
// timing ablations (results are garbage): 1 no matrix stream, 2 no tensor-memory loads in the contraction
#ifndef FHERAM_EXT8_ABL
#define FHERAM_EXT8_ABL 0
#endif
// matrix stream of the contraction: 0 LDG.128 into registers (one chunk ahead), 1 cp.async staging in the exchange buffer
#ifndef FHERAM_EXT8_STREAM
#define FHERAM_EXT8_STREAM 1
#endif
#ifndef FHERAM_EXT8_STAGGER
#define FHERAM_EXT8_STAGGER 0
#endif

namespace fheram {

constexpr int kExt8Threads = 512;
constexpr size_t kExt8Smem = (size_t)256 * sizeof(double2) + (size_t)4 * kPad16 * sizeof(double2) +
                             (size_t)4 * kN * sizeof(uint32_t) + 32;

__device__ __forceinline__ void pair_arrive(int id) { asm volatile("bar.arrive %0, 256;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void pair_sync(int id) { asm volatile("bar.sync %0, 256;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void cp_async16(const void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void red_add_u32(uint32_t* p, uint32_t v) {
  asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
// digit fields of the word W = lo + hi 2^26 (limb 0 = bits 34..50, limb 1 = 17..33, limb 2 = 0..16)
__device__ __forceinline__ uint32_t word_field(uint32_t lo, uint32_t hi, int limb) {
  if (limb == 2) return lo & 0x1ffffu;
  if (limb == 1) return ((lo >> 17) + (hi << 9)) & 0x1ffffu;
  return ((hi + (lo >> 26)) >> 8) & 0x1ffffu;
}

__global__ void __launch_bounds__(kExt8Threads, 1) k_ext8(const VmpArgs A, const double2* __restrict__ tw16) {
  constexpr int NR = 6, LOUT = 4, NOUT = 2 * LOUT;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* tw2 = reinterpret_cast<double2*>(smem_raw);
  double2* bufs = tw2 + 256;
  uint32_t* xlo = reinterpret_cast<uint32_t*>(bufs + 4 * kPad16);  // [2 cols][N]
  uint32_t* xhi = xlo + 2 * kN;                                    // [2 cols][N]
  uint32_t* slot = xhi + 2 * kN;

  const int tid = threadIdx.x, g = tid >> 7, t = tid & 127;
  auto CT = [](int col, int limb) { return (limb * 2 + col) * kN; };

  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid < 256) tw2[tid] = __ldg(tw16 + tid);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *slot;
  const uint32_t tsp = tmem_base + ((uint32_t)(((tid >> 5) & 3) * 32) << 16);  // spectrum rho at column 64 rho
  const uint32_t ttw = tsp + 384;                                              // 7 pass-3 twiddles (28 columns)
  if (g == 0) {
    const Tw3x w = load_tw3x(tw16, t);
    const double2 p0[4] = {w.w8, w.w9a, w.w9b, w.w10[0]};
    const double2 p1[4] = {w.w10[1], w.w10[2], w.w10[3], w.w10[3]};
    tm_st4(ttw, p0);
    tm_st4(ttw + 16, p1);
    tm_wait_st();
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  auto t3f = [&]() {
    double2 p0[4], p1[4];
    tm_ld4(ttw, p0);
    tm_ld4(ttw + 16, p1);
    Tw3x w;
    w.w8 = p0[0]; w.w9a = p0[1]; w.w9b = p0[2]; w.w10[0] = p0[3];
    w.w10[1] = p1[0]; w.w10[2] = p1[1]; w.w10[3] = p1[2];
    return w;
  };
  const T16 tc{bufs + g * kPad16, tw2, nullptr, t, g};
  const int co = g & 1;                    // output column of this group
  uint32_t* clo = xlo + co * kN + t;       // its words, position t (+ 128 m, + 2048)
  uint32_t* chi = xhi + co * kN + t;
  const int pair_bar = 5 + co;             // barriers 1..4: the groups (gsync128)
  long long phase_t0 = A.phase_cycles ? clock64() : 0;
  // groups of a pair leave every CTA-wide barrier A.stagger cycles apart, so that one is in a register pass (FP64 pipe)
  // while the other exchanges (shared-memory pipe) instead of both queueing for the same unit
  auto skew = [&]() {};
  // SMs start a quarter of a step apart: the grid is uniform, so without it every SM streams its matrix tiles in the
  // same thousands of cycles and the L2 (21.8 TB/s in total, tools/tile_stage_probe.cu) is the bound of that phase
  if (A.stagger > 0) {
    const long long until = clock64() + (long long)A.stagger * (blockIdx.x & 3);
    while (clock64() < until) {}
  }

  for (int item = blockIdx.x; item < A.n_items; item += gridDim.x) {
    int* dst = A.dst + (size_t)item * A.ct_stride;
    const int* src;
    {
      long idx = item;
      if (A.src_div > 0) idx = item / A.src_div;
      else if (A.src_mod > 0) { int r = item % A.src_mod; idx = A.src_map ? A.src_map[r] : r; }
      src = A.src + idx * A.ct_stride;
    }
    const size_t mat_off = A.mat_div > 0 ? (size_t)(item / A.mat_div) * A.mat_stride : 0;

    for (int step = 0; step < A.n_steps; step++) {
      const double2* G = A.mat[step] + mat_off;
      PHASE_TICK(0);
      // ------------------------------ forward transforms: rows g and g + 4 ------------------------------
      auto fwd_row = [&](int rho) {
        const int col = rho & 1, limb = rho >> 1;
        double2 x[16];
        if (step == 0) {
          // the caller's limbs as they are (any int32), like k_ext9
          const int* p = src + CT(col, limb) + t;
          asm volatile("" : "+l"(p));
#pragma unroll
          for (int m = 0; m < 16; m++) x[m] = make_double2(int_f64(p[128 * m]), int_f64(p[128 * m + kM]));
        } else {
          const uint32_t* pl = xlo + col * kN + t;
          const uint32_t* ph = xhi + col * kN + t;
#pragma unroll
          for (int m = 0; m < 16; m++) {
            const uint32_t la = pl[128 * m], lb = pl[128 * m + kM];
            uint32_t ha = 0, hb = 0;
            if (limb != 2) { ha = ph[128 * m]; hb = ph[128 * m + kM]; }
            x[m] = make_double2(field_f64(word_field(la, ha, limb), 0u), field_f64(word_field(lb, hb, limb), 0u));
          }
        }
        PHASE_TICK(1);
        forward16(x, tc, t3f);
        PHASE_TICK(2);
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const double2 v[4] = {x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]};
          tm_st4(tsp + 64 * rho + 16 * q, v);
        }
      };
      fwd_row(g);
      tm_wait_st();
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();  // rows 0..3 visible to every group
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      skew();
      if (!FHERAM_EXT8_STAGGER) {
        if (g < 2) {
          fwd_row(g + 4);
          tm_wait_st();
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();  // six spectra visible to every group; every read of the old words is done
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      } else if (g < 2) {
        // rows 4 and 5 while groups 2 and 3 already contract rows 0..3 (their matrix stream then runs beside these
        // transforms and, one output later, beside the inverse transforms of groups 0 and 1)
        fwd_row(g + 4);
        tm_wait_st();
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        asm volatile("bar.arrive 7, 512;" ::: "memory");  // groups 2, 3 wait for it before their chunk 16
        asm volatile("bar.sync 8, 256;" ::: "memory");    // rows 4 and 5 of each other
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      }
      PHASE_TICK(7);

      // ----------------- contraction + inverse transform + word update: two outputs per group -----------------
      constexpr int kDepth = 4;
      double2* stage = tc.buf + t;  // slot (s, j) of this thread: stage[(4 s + j) * 128]
      auto stage_issue = [&](const double2* gp, int c) {
        const double2* np = gp + (size_t)(c >> 2) * NOUT * kM + 512 * (c & 3);
#pragma unroll
        for (int j = 0; j < 4; j++) cp_async16(stage + (4 * (c % kDepth) + j) * 128, np + 128 * j);
        cp_async_commit();
      };
      auto stage_begin = [&](const double2* gp) {
#pragma unroll
        for (int c = 0; c < kDepth - 1; c++) stage_issue(gp, c);
      };
#pragma unroll 1
      for (int k = 0; k < 2; k++) {
        const int l = (g < 2 ? 3 : 1) - k;
        const double2* gp = G + (size_t)(co * LOUT + l) * kM + t;  // + rho NOUT kM + 128 r
        // 24 chunks of (row rho = c >> 2, frequencies r = 4 (c & 3) .. + 3).  The matrix stream is staged by cp.async
        // (16 bytes per thread and value, thread-private slots, completion by groups: no registers and no scoreboard
        // held by the values in flight) in the group's exchange buffer, idle during the contraction: kDepth - 1
        // chunks (24 KiB per group) are in flight while one is multiplied.
        double2 cur[16];
#pragma unroll
        for (int r = 0; r < 16; r++) cur[r] = make_double2(0.0, 0.0);
#if FHERAM_EXT8_STREAM == 0
        // matrix chunk c + 1 requested (LDG.128 into registers) while chunk c is multiplied
        double2 gb[2][4];
#pragma unroll
        for (int j = 0; j < 4; j++) gb[0][j] = ldg_pinned(gp + 128 * j);
#pragma unroll
        for (int c = 0; c < 4 * NR; c++) {
          if (c + 1 < 4 * NR) {
            const double2* np = gp + (size_t)((c + 1) >> 2) * NOUT * kM + 512 * ((c + 1) & 3);
#pragma unroll
            for (int j = 0; j < 4; j++) gb[(c + 1) & 1][j] = ldg_pinned(np + 128 * j);
          }
          if (FHERAM_EXT8_STAGGER && c == 16 && k == 0 && g >= 2) {
            asm volatile("bar.sync 7, 512;" ::: "memory");
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          }
          double2 a[4];
          tm_ld4(tsp + 64 * (c >> 2) + 16 * (c & 3), a);
#pragma unroll
          for (int j = 0; j < 4; j++) {
            double2& acc = cur[4 * (c & 3) + j];
            const double2 m = gb[c & 1][j];
            acc.x = fma(a[j].x, m.x, fma(-a[j].y, m.y, acc.x));
            acc.y = fma(a[j].x, m.y, fma(a[j].y, m.x, acc.y));
          }
        }
#else
        if (k == 0) stage_begin(gp);
#pragma unroll
        for (int c = 0; c < 4 * NR; c++) {
          if (!(FHERAM_EXT8_ABL & 1)) {
            if (c + kDepth - 1 < 4 * NR) stage_issue(gp, c + kDepth - 1);
            else cp_async_commit();  // empty group: the wait below counts groups
          }
          if (FHERAM_EXT8_STAGGER && c == 16 && k == 0 && g >= 2) {
            // rows 4, 5 are complete, and with them every read of the old words (forward transforms of this step)
            asm volatile("bar.sync 7, 512;" ::: "memory");
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          }
          double2 m[4], a[4];
          if (FHERAM_EXT8_ABL & 1) {
#pragma unroll
            for (int j = 0; j < 4; j++) m[j] = make_double2(1.0 + c, 0.5 * j);
          } else {
            cp_async_wait<kDepth - 1>();
#pragma unroll
            for (int j = 0; j < 4; j++) m[j] = stage[(4 * (c % kDepth) + j) * 128];
          }
          if (FHERAM_EXT8_ABL & 2) {
#pragma unroll
            for (int j = 0; j < 4; j++) a[j] = make_double2(2.0 + c, 0.25 * j);
          } else {
            tm_ld4(tsp + 64 * (c >> 2) + 16 * (c & 3), a);
          }
#pragma unroll
          for (int j = 0; j < 4; j++) {
            double2& acc = cur[4 * (c & 3) + j];
            acc.x = fma(a[j].x, m[j].x, fma(-a[j].y, m[j].y, acc.x));
            acc.y = fma(a[j].x, m[j].y, fma(a[j].y, m[j].x, acc.y));
          }
        }
#endif
        gsync128(g);  // every staged value is read before the inverse transform's first store into the buffer
        PHASE_TICK(3);
        inverse16(cur, tc, t3f);
        if (FHERAM_EXT8_STREAM && k == 0) stage_begin(gp - kM);  // the next output (limb l - 1) streams during this one's word update
        PHASE_TICK(4);
        // cur[m] = vmp[t + 128 m] + i vmp[t + 128 m + 2048] of limb l: round, add into the words of column co
        if (l == 3) {
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const int off = 128 * (q & 15) + (q >> 4) * kM;
            const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
            const double tt = v + (kMagic52 + 65536.0);
            const int c3 = (int)__funnelshift_r((uint32_t)__double2loint(tt), (uint32_t)__double2hiint(tt), 17);
            const unsigned long long W = ((unsigned long long)(long long)c3 + kBias51) & kMask51;
            clo[off] = (uint32_t)W & 0x3ffffffu;
            chi[off] = (uint32_t)(W >> 26);
          }
          pair_arrive(pair_bar);  // the column's words exist: the other group of the pair may add
        } else if (l == 2) {
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const int off = 128 * (q & 15) + (q >> 4) * kM;
            const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
            const unsigned long long m = magic_bits(v + kMagic52);
            red_add_u32(clo + off, (uint32_t)m & 0x3ffffffu);
            red_add_u32(chi + off, (uint32_t)(m >> 26) & 0x1ffffffu);
          }
        } else if (l == 1) {
          pair_sync(pair_bar);
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const int off = 128 * (q & 15) + (q >> 4) * kM;
            const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
            const unsigned long long m = magic_bits(v + kMagic52);
            red_add_u32(clo + off, ((uint32_t)m & 0x1ffu) << 17);
            red_add_u32(chi + off, (uint32_t)(m >> 9) & 0x1ffffffu);
          }
        } else {
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const int off = 128 * (q & 15) + (q >> 4) * kM;
            const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
            const uint32_t m = (uint32_t)__double2loint(v + kMagic52);
            red_add_u32(chi + off, (m & 0x1ffffu) << 8);
          }
        }
        PHASE_TICK(5);
      }
      // every contribution landed before the next step's reads; every spectrum read precedes the next stores
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      skew();
    }  // steps

    // digits of the final words -> dst (coalesced)
#pragma unroll 4
    for (int m = 0; m < 8; m++) {
      const int i = tid + 512 * m;
#pragma unroll
      for (int col = 0; col < 2; col++) {
        const uint32_t lo = xlo[col * kN + i], hi = xhi[col * kN + i];
        dst[CT(col, 0) + i] = (int)word_field(lo, hi, 0) - 65536;
        dst[CT(col, 1) + i] = (int)word_field(lo, hi, 1) - 65536;
        dst[CT(col, 2) + i] = (int)word_field(lo, hi, 2) - 65536;
      }
    }
    __syncthreads();  // words reuse by the next item
    PHASE_TICK(6);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

}  // namespace fheram
