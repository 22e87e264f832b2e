// kernels_ks4.cuh -- k_ks3 (key switch on 51-bit words, padded transforms) with the matrix stream
// software-pipelined: words are accumulated in place in shared memory instead of 32 registers, the
// registers hold a second matrix tile, so the L2 round trip of tile t+1 overlaps the FMAs of tile t
// and the first tile of every output is fetched during the previous inverse transform.
// (tools/ablate: without matrix loads k_ks3 runs 76.8 K -> 58.1 K cycles per operation; the loads
// were three exposed L2 round trips per output.)  Same integers as k_ks3 / k_ks2 / k_vmp.
// Two-sided combine of GLWEPacker only: the wide launches of the packer tree (the trace kernels took its traces).
#pragma once
#include "kernels_ks3.cuh"

namespace fheram {

constexpr size_t kKs4Smem = (size_t)kWorkPad * sizeof(double2) + (size_t)2 * kN * sizeof(long long) + 16;

__global__ void __launch_bounds__(kThreads, 2) k_ks4(const VmpArgs A) {
  constexpr int R = 3, LOUT = 4, NOUT = 2 * LOUT;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* work = reinterpret_cast<double2*>(smem_raw);  // padded exchange buffer (transform_pad.cuh)
  unsigned long long* xp = reinterpret_cast<unsigned long long*>(work + kWorkPad);  // [2 cols][N] words
  uint32_t* tmem_base_s = reinterpret_cast<uint32_t*>(xp + 2 * kN);

  const int T = threadIdx.x, w = T >> 5, lane = T & 31;
  auto CT = [](int col, int limb) { return (limb * 2 + col) * kN; };

  if (w == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(tmem_base_s)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  BufSync bs{smem_u32(tmem_base_s + 2), 0u};  // exchange-buffer mbarrier in the same 16-byte slot
  if (T == 0) buf_init(bs.mbar);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_base_s;
  buf_release(bs);  // the buffer starts out free
  // this thread's 128 columns: spectra rows at +0/+32/+64, twiddles at +96 (pass 3) / +112 (pass 4)
  const uint32_t tsp = tmem_base + ((uint32_t)((w & 3) * 32) << 16) + 128 * (w >> 2);
  const uint32_t ttw = tsp + 96;
  {
    const Tw34 t = load_tw34(A.tw, w, lane);
    const double2 p3[4] = {t.a3, t.b3, t.c3, t.d3};
    const double2 p4[4] = {t.b4a, t.b4b, t.c4a, t.c4b};
    tm_st4(ttw, p3);
    tm_st4(ttw + 16, p4);
    tm_wait_st();
  }
  const int P0 = 256 * w + lane;
  const PadAddr pa = pad_addr(work, T, w, lane);
  auto tw3 = [&]() { double2 t[4]; tm_ld4(ttw, t); return Tw4x{t[0], t[1], t[2], t[3]}; };
  auto tw4 = [&]() { double2 t[4]; tm_ld4(ttw + 16, t); return Tw4x{t[0], t[1], t[2], t[3]}; };
  long long phase_t0 = A.phase_cycles ? clock64() : 0;

  for (int item = blockIdx.x; item < A.n_items; item += gridDim.x) {
    int* dst = A.dst + (size_t)item * A.ct_stride;
    // words of S = rsh1(a X^-t + b), [2 cols][N], in this CTA's global scratch
    unsigned long long* sw = A.scratch
        ? reinterpret_cast<unsigned long long*>(A.scratch + (size_t)blockIdx.x * A.ct_stride) : nullptr;
    const int* src = A.src + 2L * item * A.ct_stride;
    const size_t mat_off = A.mat_div > 0 ? (size_t)(item / A.mat_div) * A.mat_stride : 0;

    // ------------------------------ prologue (once per item) ---------------------------
    {
      // a1 = a X^-t;  D = rsh1(a1 - b) -> xp;  S = rsh1(a1 + b) -> sw
      const int* a = src;
      const int* b = src + A.ct_stride;
      const int tt = A.rot_const;
#pragma unroll 1
      for (int mc = 0; mc < 16; mc += 4) {
        int av[4][2][3], bv[4][2][3];
        bool ng[4];
#pragma unroll
        for (int mm = 0; mm < 4; mm++) {
          const int i = T + 256 * (mc + mm);
          const int j = rot_index(i, tt, ng[mm]);  // (a X^-t)[i] = +/- a[(i + t) mod 2N]
#pragma unroll
          for (int col = 0; col < 2; col++)
#pragma unroll
            for (int l = 0; l < 3; l++) { av[mm][col][l] = a[CT(col, l) + j]; bv[mm][col][l] = b[CT(col, l) + i]; }
        }
#pragma unroll
        for (int mm = 0; mm < 4; mm++) {
          const int i = T + 256 * (mc + mm);
#pragma unroll
          for (int col = 0; col < 2; col++) {
            long long Xa = limbs_value(av[mm][col][0], av[mm][col][1], av[mm][col][2]);
            if (ng[mm]) Xa = -Xa;
            const long long Xb = limbs_value(bv[mm][col][0], bv[mm][col][1], bv[mm][col][2]);
            xp[col * kN + i] = rsh1_word(Xa - Xb);
            sw[col * kN + i] = rsh1_word(Xa + Xb);
          }
        }
      }
    }
    __syncthreads();
    PHASE_TICK(0);

    double2 gA[8], gB[8];  // matrix tiles in flight (double buffer)
    {
      // first tile of the item: step 0, mask column, limb 3, row 0
      const double2* gp = A.mat[0] + mat_off + (size_t)(LOUT + LOUT - 1) * kM + P0;
#pragma unroll
      for (int j = 0; j < 8; j++) gA[j] = ldg_pinned(gp + 32 * j);
    }
    for (int step = 0; step < A.n_steps; step++) {
      const double2* G = A.mat[step] + mat_off;
      const int ginv = A.gal_inv[step];
      const bool last = step + 1 == A.n_steps;
      // automorphism source of this thread's positions i_q = T + 256 (q & 7) + 2048 (q >> 3):
      // e_q = i_q * ginv mod 2N (index e_q mod N, sign e_q >= N); e_q = e0 + (q & 7) d1 + (q >> 3) d2
      const int e0 = (T * ginv) & (2 * kN - 1);
      const int d1 = (256 * ginv) & (2 * kN - 1);
      const int d2 = kM * (ginv & 3);
      unsigned sgn = 0;  // bit q: phi_g flips the sign at position i_q

      // --------------------------- forward transforms ------------------------------
      {
        // phi_g(x) mask digits of the 16 input positions; the words are gathered again for every
        // limb (holding them across the three transforms costs 32 registers and spills)
#pragma unroll 1
        for (int rho = 0; rho < R; rho++) {
          double2 x[8];
          // digit rho = bits [17 (2 - rho), +17) of the word = (funnel(lo, hi, s1) >> s2) & (2^17 - 1)
          // (shift amounts kept loop-variant on purpose: with per-rho code the compiler hoists all
          // 48 digits out of the loop and spills them)
          const int s1 = rho == 0 ? 31 : (rho == 1 ? 17 : 0);
          const int s2 = rho == 0 ? 3 : 0;
          unsigned sg = 0;
#pragma unroll
          for (int m = 0; m < 8; m++) {
            const int ea = (e0 + m * d1) & (2 * kN - 1);
            const int eb = (ea + d2) & (2 * kN - 1);
            const unsigned long long wa = xp[kN + (ea & (kN - 1))];
            const unsigned long long wb = xp[kN + (eb & (kN - 1))];
            const uint32_t na = ea >= kN ? 0x80000000u : 0u, nb = eb >= kN ? 0x80000000u : 0u;
            sg |= (na >> (31 - m)) | (nb >> (23 - m));
            x[m] = make_double2(
                field_f64((__funnelshift_r((uint32_t)wa, (uint32_t)(wa >> 32), s1) >> s2) & 0x1ffffu, na),
                field_f64((__funnelshift_r((uint32_t)wb, (uint32_t)(wb >> 32), s1) >> s2) & 0x1ffffu, nb));
          }
          sgn = sg;
          if (!(FHERAM_ABL & 4)) {
            fwd_pass1_store_p(x, pa, bs);
            __syncthreads();
            fwd_warp_passes_p(pa, w, tw3, tw4, x, bs);
          }
          {
            const double2 lo[4] = {x[0], x[1], x[2], x[3]};
            const double2 hi[4] = {x[4], x[5], x[6], x[7]};
            tm_st4(tsp + 32 * rho, lo);
            tm_st4(tsp + 32 * rho + 16, hi);
          }
        }
        tm_wait_st();
      }
      PHASE_TICK(2);

      // --------------- contraction + inverse transform + word accumulation ---------
      // The words of the column being produced are accumulated IN PLACE in shared memory (own
      // positions only), which frees the 32 accumulator registers of k_ks3 for a second matrix
      // tile: the loads of tile t+1 are issued before the FMAs of tile t, and the first tile of
      // the next output is in flight during the inverse transform of the current one.
      // Mask column first: its old words were consumed by the forward gather; the body column's
      // old words are gathered (phi_g) into the accumulator behind one barrier.
#pragma unroll 1
      for (int cc = 0; cc < 2; cc++) {
        const int co = 1 - cc;
        unsigned long long* xc = xp + co * kN;
        if (co == 0) {
          // accumulator init: sigma (D_body[u] - bias)
          unsigned long long v0[16];
#pragma unroll
          for (int q = 0; q < 16; q++) {
            const int e = (e0 + (q & 7) * d1 + (q >> 3) * d2) & (2 * kN - 1);
            const unsigned long long b = xp[e & (kN - 1)] - kBias51;
            const bool ng = ((sgn >> q) & 1u) != 0;
            v0[q] = ng ? 0ull - b : b;
          }
          __syncthreads();  // every gather of the old body column precedes its stores
#pragma unroll
          for (int q = 0; q < 16; q++) xp[T + 256 * (q & 7) + (q >> 3) * kM] = v0[q];
        }
#pragma unroll 1
        for (int l = LOUT - 1; l >= 0; l--) {
          const int o = co * LOUT + l;
          double2 cur[8];
#pragma unroll
          for (int j = 0; j < 8; j++) cur[j] = make_double2(0.0, 0.0);
          // tiles rho = 0, 1, 2 of this output; gA holds rho = 0 on entry
          auto fma_tile = [&](const double2 (&g)[8], int rho) {
#pragma unroll
            for (int h = 0; h < 2; h++) {
              double2 a[4];
              tm_ld4(tsp + 32 * rho + 16 * h, a);
#pragma unroll
              for (int j = 0; j < 4; j++) {
                cur[4 * h + j].x = fma(a[j].x, g[4 * h + j].x, fma(-a[j].y, g[4 * h + j].y, cur[4 * h + j].x));
                cur[4 * h + j].y = fma(a[j].x, g[4 * h + j].y, fma(a[j].y, g[4 * h + j].x, cur[4 * h + j].y));
              }
            }
          };
          {
            const double2* gp = G + ((size_t)1 * NOUT + o) * kM + P0;
#pragma unroll
            for (int j = 0; j < 8; j++) gB[j] = ldg_pinned(gp + 32 * j);
          }
          fma_tile(gA, 0);
          {
            const double2* gp = G + ((size_t)2 * NOUT + o) * kM + P0;
#pragma unroll
            for (int j = 0; j < 8; j++) gA[j] = ldg_pinned(gp + 32 * j);
          }
          fma_tile(gB, 1);
          {
            // first tile of the next output: (co, l - 1), then column 0, then the next step's matrix
            const bool more = !(cc == 1 && l == 0 && last);
            const double2* Gn = (cc == 1 && l == 0) ? A.mat[last ? step : step + 1] + mat_off : G;
            const int on = l > 0 ? o - 1 : (cc == 0 ? LOUT - 1 : LOUT + LOUT - 1);
            const double2* gp = Gn + (size_t)on * kM + P0;
            if (more) {
#pragma unroll
              for (int j = 0; j < 8; j++) gB[j] = ldg_pinned(gp + 32 * j);
            }
          }
          fma_tile(gA, 2);
#pragma unroll
          for (int j = 0; j < 8; j++) gA[j] = gB[j];
          PHASE_TICK(3);
          inv_transform_p(cur, pa, w, tw3, tw4, bs);
          PHASE_TICK(4);
          // cur[m] = phi_g(vmp)[T + 256 m] (+ i * [.. + 2048]); round and add into the word
          if (l == 3) {
            // floor((s r + 2^16) / 2^17) with s the sign frame of the carry chain, the per-position
            // automorphism sign, for which floor((-r + 2^16) / 2^17) = -floor((r + 2^16 - 1) / 2^17)
#pragma unroll
            for (int q = 0; q < 16; q++) {
              const int i = T + 256 * (q & 7) + (q >> 3) * kM;
              const double v = (q < 8) ? cur[q & 7].x : cur[q & 7].y;
              const double t = v + __hiloint2double(0x43380000, (int)(65536u - ((sgn >> q) & 1u)));
              const int c3 = (int)__funnelshift_r((uint32_t)__double2loint(t), (uint32_t)__double2hiint(t), 17);
              if (co == 1) xc[i] = (unsigned long long)(long long)c3;  // D mask words are dead
              else xc[i] += (unsigned long long)(long long)c3;
            }
          } else if (l == 2) {
#pragma unroll
            for (int q = 0; q < 16; q++) {
              const int i = T + 256 * (q & 7) + (q >> 3) * kM;
              const double v = (q < 8) ? cur[q & 7].x : cur[q & 7].y;
              xc[i] += magic_bits(v + kMagic52);
            }
          } else if (l == 1) {
#pragma unroll
            for (int q = 0; q < 16; q++) {
              const int i = T + 256 * (q & 7) + (q >> 3) * kM;
              const double v = (q < 8) ? cur[q & 7].x : cur[q & 7].y;
              xc[i] += magic_bits(v + kMagic52) << 17;
            }
          } else {
            // last limb: finish the word
#pragma unroll
            for (int q = 0; q < 16; q++) {
              const int i = T + 256 * (q & 7) + (q >> 3) * kM;
              const double v = (q < 8) ? cur[q & 7].x : cur[q & 7].y;
              const double t = v + kMagic52;
              const unsigned long long W = xc[i] + ((unsigned long long)((uint32_t)__double2loint(t) << 2) << 32);
              // y = phi_g(normalize(KS(D)));  out = normalize(S - y) X^t:
              //   word = S - (R + k3) - sigma (D_body[u] - bias)
              const unsigned long long U = (sw[co * kN + i] - W) & kMask51;
              bool rneg;
              const int dd = rot_index(i, A.rot_const, rneg);  // a' * X^t
#pragma unroll
              for (int ll = 0; ll < 3; ll++) {
                const int dg = word_digit(U, ll);
                dst[CT(co, ll) + dd] = rneg ? -dg : dg;
              }
            }
          }
          PHASE_TICK(5);
        }
      }
    }  // steps

    __syncthreads();  // xp reuse by the next item
    PHASE_TICK(6);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (w == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base) : "memory");
}

}  // namespace fheram
