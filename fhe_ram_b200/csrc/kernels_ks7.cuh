// kernels_ks7.cuh -- trace chains on the wide launches, with the two-exchange transform of transform16.cuh
// (DESIGN.md 7.2 item 1).
//
// k_ks4 transforms one polynomial at a time with 256 threads x 8 points and three shared-memory exchanges;
// its register passes are shared-memory bound and its eight inverse transforms per step run one after the other.
// Here the two groups of 128 threads of a CTA work on two polynomials at once: group g owns output column g
// (contraction, inverse transform, in-place word accumulation of that column), the three forward transforms are
// split 2 + 1.  The groups take turns on one exchange buffer (a lock held from the first store to the last load of a
// transform's exchanges), which keeps the CTA at 34 + 64 (words) + 4 (twiddles) = 102 KiB, two CTAs per SM.
//   tensor memory (256 columns per CTA): per thread position three spectra (3 x 64 columns) + pass-3 twiddles (28).
// Integer side: the 51-bit words of words.cuh, accumulated in place as in k_ks4 (each position is owned by one
// thread of the column's group).  The matrix tiles are not double buffered (the registers hold 16 accumulators).
// Same integers as every other kernel; the frequency order of transform16.cuh, hence its own prepared trace keys.
#pragma once
#include "sync.cuh"
#include "tmem.cuh"
#include "transform16.cuh"
#include "words.cuh"

namespace fheram {

constexpr size_t kKs7Smem = (size_t)256 * sizeof(double2) + (size_t)kPad16 * sizeof(double2) +
                            (size_t)2 * kN * sizeof(long long) + 32;

// ======================================================================================
// k_ks7: chain of { rsh 1; x <- x +/- phi_g(KS(x)) }  (trace / one-sided packer levels)
// ======================================================================================
__global__ void __launch_bounds__(256, 2) k_ks7(const VmpArgs A, const double2* __restrict__ tw16) {
  constexpr int LOUT = 4, NOUT = 2 * LOUT;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* tw2 = reinterpret_cast<double2*>(smem_raw);
  double2* buf = tw2 + 256;
  unsigned long long* xp = reinterpret_cast<unsigned long long*>(buf + kPad16);  // [2 cols][N] words
  uint32_t* slot = reinterpret_cast<uint32_t*>(xp + 2 * kN);                     // +0 tmem base, +4 buffer lock

  const int tid = threadIdx.x, g = tid >> 7, t = tid & 127;
  auto CT = [](int col, int limb) { return (limb * 2 + col) * kN; };

  if (tid < 32) tmem_alloc<256>(slot);
  tw2[tid] = __ldg(tw16 + tid);
  if (tid == 0) slot[1] = 0u;
  tmem_sync();
  const uint32_t tmem_base = *slot;
  // thread position (quadrant = warp & 3, lane): both groups address the same columns
  const uint32_t tsp = tmem_base + ((uint32_t)(((tid >> 5) & 3) * 32) << 16);  // spectra rows at +0 / +64 / +128
  const uint32_t ttw = tsp + 192;                                             // 7 pass-3 twiddles (28 columns)
  if (g == 0) park_tw3x(ttw, tw16, t);
  tmem_sync();
  auto t3f = [&]() { return tm_tw3x(ttw); };
  const T16 tc{buf, tw2, slot + 1, t, g};
  const double sgn_d = A.sign < 0 ? -1.0 : 1.0;
  const uint32_t sgn_bit = A.sign < 0 ? 1u : 0u;
  const int co = g;                         // output column of this group
  unsigned long long* xc = xp + co * kN;    // its words
  long long phase_t0 = A.phase_cycles ? clock64() : 0;

  for (int item = blockIdx.x; item < A.n_items; item += gridDim.x) {
    int* dst = A.dst + (size_t)item * A.ct_stride;
    const int* src = item_src(A, item);
    const size_t mat_off = A.mat_div > 0 ? (size_t)(item / A.mat_div) * A.mat_stride : 0;

    // ------------------------------ prologue: x = rsh1(src * X^rk) ------------------------------
    {
      const int rk = trace_rot(A, item, A.rot_const);
#pragma unroll 4
      for (int m = 0; m < 16; m++) {
        const int i = tid + 256 * m;
        bool neg;
        const int j = rot_index(i, 2 * kN - rk, neg);
#pragma unroll
        for (int col = 0; col < 2; col++) {
          long long X = limbs_value(src[CT(col, 0) + j], src[CT(col, 1) + j], src[CT(col, 2) + j]);
          if (neg) X = -X;
          xp[col * kN + i] = rsh1_word(X);
        }
      }
    }
    __syncthreads();
    PHASE_TICK(0);

    for (int step = 0; step < A.n_steps; step++) {
      const double2* G = A.mat[step] + mat_off;
      const int ginv = A.gal_inv[step];
      const bool last = step + 1 == A.n_steps;
      // automorphism source of this thread's positions i = t + 128 m (+ 2048): e = i * ginv mod 2N
      const int e0 = (t * ginv) & (2 * kN - 1);
      const int d1 = (128 * ginv) & (2 * kN - 1);
      const int d2 = kM * (ginv & 3);
      // ------------- forward transforms: group 0 rows 0 and 2, group 1 row 1 and the body init -------------
      auto fwd_row = [&](int rho) {
        double2 x[16];
        const int s1 = rho == 0 ? 31 : (rho == 1 ? 17 : 0);
        const int s2 = rho == 0 ? 3 : 0;
        // opaque copy: otherwise the 32 gather addresses are hoisted out of the row loop and spilled
        int e0r = e0;
        asm volatile("" : "+r"(e0r));
#pragma unroll
        for (int m = 0; m < 16; m++) {
          const int ea = (e0r + m * d1) & (2 * kN - 1);
          const int eb = (ea + d2) & (2 * kN - 1);
          const unsigned long long wa = xp[kN + (ea & (kN - 1))];
          const unsigned long long wb = xp[kN + (eb & (kN - 1))];
          const uint32_t na = ea >= kN ? 0x80000000u : 0u, nb = eb >= kN ? 0x80000000u : 0u;
          x[m] = make_double2(
              field_f64((__funnelshift_r((uint32_t)wa, (uint32_t)(wa >> 32), s1) >> s2) & 0x1ffffu, na),
              field_f64((__funnelshift_r((uint32_t)wb, (uint32_t)(wb >> 32), s1) >> s2) & 0x1ffffu, nb));
        }
        forward16(x, tc, t3f);
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const double2 v[4] = {x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]};
          tm_st4(tsp + 64 * rho + 16 * q, v);
        }
      };
      if (g == 0) {
#pragma unroll 1
        for (int rr = 0; rr < 2; rr++) fwd_row(2 * rr);
      } else {
        fwd_row(1);
        // body-column accumulator init: x_body + s phi_g(x_body), 32 positions per thread, in two halves (the
        // gathers of both halves precede every store: one group barrier in between)
        unsigned long long v0[16], v1[16];
#pragma unroll
        for (int m = 0; m < 16; m++) {
          const int ea = (e0 + m * d1) & (2 * kN - 1);
          v0[m] = body_base(xp[ea & (kN - 1)], ((ea >= kN ? 1u : 0u) ^ sgn_bit) != 0, xp[t + 128 * m]);
        }
#pragma unroll
        for (int m = 0; m < 16; m++) {
          const int eb = (e0 + m * d1 + d2) & (2 * kN - 1);
          v1[m] = body_base(xp[eb & (kN - 1)], ((eb >= kN ? 1u : 0u) ^ sgn_bit) != 0, xp[t + 128 * m + kM]);
        }
        gsync128(1);  // every gather of the old body column precedes its stores
#pragma unroll
        for (int m = 0; m < 16; m++) { xp[t + 128 * m] = v0[m]; xp[t + 128 * m + kM] = v1[m]; }
      }
      tm_wait_st();
      tmem_sync();  // spectra and the body init are visible to both groups
      PHASE_TICK(2);

      // --------- contraction + inverse transform + in-place word accumulation, column `co` -----------
#pragma unroll 1
      for (int l = LOUT - 1; l >= 0; l--) {
        const int o = co * LOUT + l;
        double2 cur[16];
#pragma unroll
        for (int r = 0; r < 16; r++) cur[r] = make_double2(0.0, 0.0);
#pragma unroll 1
        for (int rho = 0; rho < 3; rho++) {
          const double2* gp = G + ((size_t)rho * NOUT + o) * kM + t;
#pragma unroll
          for (int hf = 0; hf < 2; hf++) {
            double2 gt[8];
#pragma unroll
            for (int r = 0; r < 8; r++) gt[r] = ldg_pinned(gp + 128 * (8 * hf + r));
#pragma unroll
            for (int q = 0; q < 2; q++) {
              double2 a[4];
              tm_ld4(tsp + 64 * rho + 32 * hf + 16 * q, a);
#pragma unroll
              for (int j = 0; j < 4; j++) cmac(cur[8 * hf + 4 * q + j], a[j], gt[4 * q + j]);
            }
          }
        }
        PHASE_TICK(3);
        inverse16(cur, tc, t3f);
        PHASE_TICK(4);
        // cur[m] = phi_g(vmp)[t + 128 m] + i phi_g(vmp)[t + 128 m + 2048]: round and add into the words
        if (l == 3) {
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const int i = t + 128 * (q & 15) + (q >> 4) * kM;
            const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
            xc[i] += limb_word(v, 3, sgn_d, true, 0u);
          }
        } else if (l == 2) {
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const int i = t + 128 * (q & 15) + (q >> 4) * kM;
            const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
            xc[i] += limb_word(v, 2, sgn_d, true, 0u);
          }
        } else if (l == 1) {
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const int i = t + 128 * (q & 15) + (q >> 4) * kM;
            const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
            xc[i] += limb_word(v, 1, sgn_d, true, 0u);
          }
        } else {
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const int i = t + 128 * (q & 15) + (q >> 4) * kM;
            const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
            const unsigned long long W = xc[i] + limb_word(v, 0, sgn_d, true, 0u);
            const unsigned long long U = W & kMask51;
            xc[i] = last ? U : rsh1_canon(U);
          }
        }
        PHASE_TICK(5);
      }
      // both columns complete before the next step's gathers; every spectrum read precedes the next stores
      tmem_sync();
    }  // steps

#pragma unroll 4
    for (int m = 0; m < 16; m++) {
      const int i = tid + 256 * m;
#pragma unroll
      for (int col = 0; col < 2; col++) put_digits(dst, col, i, xp[col * kN + i]);
    }
    __syncthreads();  // xp reuse by the next item
    PHASE_TICK(6);
  }
  tmem_free<256>(tmem_base, tid < 32);
}

}  // namespace fheram
