// kernels_ks6.cuh -- latency variant of k_ks5<TRACE> for very narrow launches (the 12-step trace on
// word_size ciphertexts at the end of every read, src/ram.rs:457; the write path's first trace, :572):
// one trace chain per CLUSTER of two CTAs (two SMs), 512 threads each.
//
//   CTA c of the cluster owns output column c (c = 1: mask, c = 0: body); inside a CTA the two groups of 8
//   warps take two of the four output limbs each (group 0: limbs 3 and 1, group 1: limbs 2 and 0) and add
//   their word contributions into the same shared-memory words with 64-bit shared atomics, so a step costs
//   two contraction + inverse-transform rounds instead of the four of k_ks5 (eight of k_ks4).
//   Both CTAs transform the three mask limbs themselves (the spectra live in their own tensor memory).
//   The only data that crosses SMs is the new mask column: CTA 1 writes each finished word into its own
//   shared memory and into CTA 0's (distributed shared memory, st.shared::cluster), ordered by two split
//   cluster barriers per step (arrive after the forward gathers / wait before the remote stores; arrive after
//   them / wait before the next step's gathers).
// Everything else (51-bit words, padded transforms, matrix tiles parked in tensor memory during the inverse
// transform) is k_ks5.  Same integers as every other generation (tests/test_gpu_kernel_variants.py: "ks6").
#pragma once
#include "sync.cuh"
#include "tmem.cuh"
#include "transform_pad.cuh"
#include "words.cuh"

namespace fheram {

template <int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(512, 1) k_ks6(const VmpArgs A) {
  static_assert(MODE == MODE_TRACE || MODE == MODE_COMBINE2 || MODE == MODE_MIXED, "key-switch modes only");
  constexpr int LOUT = 4, NOUT = 2 * LOUT;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* work_all = reinterpret_cast<double2*>(smem_raw);                         // [2 groups] exchange buffers
  unsigned long long* xp = reinterpret_cast<unsigned long long*>(work_all + 2 * kWorkPad);  // [2 cols][N] words
  uint32_t* slot = reinterpret_cast<uint32_t*>(xp + 2 * kN);  // +0 tmem base, +8/+16 mbarriers of the groups

  const int tid = threadIdx.x, grp = tid >> 8, T = tid & 255, w = T >> 5, lane = T & 31;
  const int co = (int)cluster_ctarank();  // output column of this CTA
  auto CT = [](int col, int limb) { return (limb * 2 + col) * kN; };

  if (tid < 32) tmem_alloc<512>(slot);
  BufSync bs{smem_u32(slot + 2 + 2 * grp), 0u};
  if (T == 0) buf_init(bs.mbar);
  tmem_sync();
  const uint32_t tmem_base = *slot;
  buf_release(bs);
  const uint32_t tsp = tmem_base + ((uint32_t)((w & 3) * 32) << 16) + 256 * (w >> 2);
  const uint32_t ttw = tsp + 96;
  const uint32_t tpark = tsp + 128 + 64 * grp;
  if (grp == 0) park_tw34(ttw, A.tw, w, lane);
  tmem_sync();

  const int P0 = 256 * w + lane;
  const PadAddr pa = pad_addr(work_all + grp * kWorkPad, T, w, lane);
  auto tw3 = [&]() { return tm_tw3(ttw); };
  auto tw4 = [&]() { return tm_tw4(ttw); };
  const double sgn_d = (MODE == MODE_TRACE && A.sign < 0) ? -1.0 : 1.0;
  const uint32_t sgn_bit = (MODE == MODE_TRACE && A.sign < 0) ? 1u : 0u;
  unsigned long long* xc = xp + co * kN;  // the words this CTA produces
  // CTA 0's copy of the mask column, as seen from CTA 1
  const uint32_t remote_mask = map_to_cta(smem_u32(xp + kN), 0);
  const int l_first = grp == 0 ? 3 : 2;   // this group's limbs: l_first, l_first - 2

  const int n_clusters = gridDim.x >> 1;
  for (int item = blockIdx.x >> 1; item < A.n_items; item += n_clusters) {
    int* dst = A.dst + (size_t)item * A.ct_stride;
    // COMBINE2: words of S = rsh1(a X^-t + b) of this CTA's column, in its global scratch
    unsigned long long* sw = A.scratch
        ? reinterpret_cast<unsigned long long*>(A.scratch + (size_t)blockIdx.x * A.ct_stride) : nullptr;
    const int* src;
    bool two = true;  // MODE_MIXED: the item has its second operand
    if constexpr (MODE == MODE_MIXED) {
      src = mixed_src(A, item, two);
    } else {
      long idx = item;
      if (MODE == MODE_COMBINE2) idx = 2L * item;
      else if (A.src_div > 0) idx = item / A.src_div;
      else if (A.src_mod > 0) { int r = item % A.src_mod; idx = A.src_map ? A.src_map[r] : r; }
      src = A.src + idx * A.ct_stride;
    }
    // this item's path: TRACE steps, or the two-sided combine (a constant unless MODE_MIXED)
    const bool trace = MODE == MODE_MIXED ? !two : MODE == MODE_TRACE;
    const size_t mat_off = A.mat_div > 0 ? (size_t)(item / A.mat_div) * A.mat_stride : 0;

    // -------- prologue: both CTAs need the mask column of x (TRACE) / D (COMBINE2), CTA 0 also the body --------
    // CTA 0: group 0 converts the body column, group 1 the mask column; CTA 1: both groups half of the mask
    {
      const int col = co == 0 ? grp : 1;
      const int m0 = co == 0 ? 0 : 8 * grp, m1 = co == 0 ? 16 : 8 * grp + 8;
      if (trace) {
        // x = rsh1(src * X^rk)  (MODE_MIXED: the one-sided combine, no rotation)
        const int rk = trace_rot(A, item, MODE == MODE_MIXED ? 0 : A.rot_const);
#pragma unroll 4
        for (int m = m0; m < m1; m++) {
          const int i = T + 256 * m;
          bool neg;
          const int j = rot_index(i, 2 * kN - rk, neg);
          long long X = limbs_value(src[CT(col, 0) + j], src[CT(col, 1) + j], src[CT(col, 2) + j]);
          if (neg) X = -X;
          xp[col * kN + i] = rsh1_word(X);
        }
      } else {
        // a1 = a X^-t;  D = rsh1(a1 - b) -> xp;  S = rsh1(a1 + b) -> sw (own column only)
        const int* a = src;
        const int* b = src + A.ct_stride;
        const int tt = A.rot_const;
#pragma unroll 1
        for (int mc = m0; mc < m1; mc += 8) {
          int av[8][3], bv[8][3];
          bool ng[8];
#pragma unroll
          for (int mm = 0; mm < 8; mm++) {
            const int i = T + 256 * (mc + mm);
            const int j = rot_index(i, tt, ng[mm]);  // (a X^-t)[i] = +/- a[(i + t) mod 2N]
#pragma unroll
            for (int l = 0; l < 3; l++) { av[mm][l] = a[CT(col, l) + j]; bv[mm][l] = b[CT(col, l) + i]; }
          }
#pragma unroll
          for (int mm = 0; mm < 8; mm++) {
            const int i = T + 256 * (mc + mm);
            long long Xa = limbs_value(av[mm][0], av[mm][1], av[mm][2]);
            if (ng[mm]) Xa = -Xa;
            const long long Xb = limbs_value(bv[mm][0], bv[mm][1], bv[mm][2]);
            xp[col * kN + i] = rsh1_word(Xa - Xb);
            if (col == co) sw[i] = rsh1_word(Xa + Xb);
          }
        }
      }
    }
    __syncthreads();

    double2 stage[8];
    const double2* gnext = A.mat[0] + mat_off + (size_t)(co * LOUT + l_first) * kM + P0;
    bool have_next = true;
    auto fetch = [&](int rho) {
      const double2* gp = gnext + (size_t)rho * NOUT * kM;
#pragma unroll
      for (int j = 0; j < 8; j++) stage[j] = ldg_pinned(gp + 32 * j);
    };
    auto park = [&](int which) {
      const double2 lo[4] = {stage[0], stage[1], stage[2], stage[3]};
      const double2 hi[4] = {stage[4], stage[5], stage[6], stage[7]};
      tm_st4(tpark + 32 * which, lo);
      tm_st4(tpark + 32 * which + 16, hi);
    };
    auto prefetch = [&](int point) {
      if (!have_next) return;
      if (point == 0) { fetch(1); }
      else if (point == 1) { park(0); fetch(2); }
      else { park(1); fetch(0); }
    };

    for (int step = 0; step < A.n_steps; step++) {
      const double2* G = A.mat[step] + mat_off;
      const int ginv = A.gal_inv[step];
      const bool last = step + 1 == A.n_steps;
      const int e0 = (T * ginv) & (2 * kN - 1);
      const int d1 = (256 * ginv) & (2 * kN - 1);
      const int d2 = kM * (ginv & 3);
      unsigned sgn = 0;
#pragma unroll
      for (int q = 0; q < 16; q++) sgn |= ((((e0 + (q & 7) * d1 + (q >> 3) * d2) & (2 * kN - 1)) >= kN) ? 1u : 0u) << q;

      // ------------- forward transforms: group 0 rows 0 and 1, group 1 row 2 (in both CTAs) ---------------
      if (step == 0) prefetch(0);
#pragma unroll 1
      for (int rho = (grp == 0 ? 0 : 2); rho < (grp == 0 ? 2 : 3); rho++) {
        double2 x[8];
        const int s1 = rho == 0 ? 31 : (rho == 1 ? 17 : 0);
        const int s2 = rho == 0 ? 3 : 0;
#pragma unroll
        for (int m = 0; m < 8; m++) {
          const int ea = (e0 + m * d1) & (2 * kN - 1);
          const int eb = (ea + d2) & (2 * kN - 1);
          const unsigned long long wa = xp[kN + (ea & (kN - 1))];
          const unsigned long long wb = xp[kN + (eb & (kN - 1))];
          const uint32_t na = ea >= kN ? 0x80000000u : 0u, nb = eb >= kN ? 0x80000000u : 0u;
          x[m] = make_double2(
              field_f64((__funnelshift_r((uint32_t)wa, (uint32_t)(wa >> 32), s1) >> s2) & 0x1ffffu, na),
              field_f64((__funnelshift_r((uint32_t)wb, (uint32_t)(wb >> 32), s1) >> s2) & 0x1ffffu, nb));
        }
        fwd_pass1_store_p(x, pa, bs);
        group_sync(grp);
        fwd_warp_passes_p(pa, w, tw3, tw4, x, bs);
        {
          const double2 lo[4] = {x[0], x[1], x[2], x[3]};
          const double2 hi[4] = {x[4], x[5], x[6], x[7]};
          tm_st4(tsp + 32 * rho, lo);
          tm_st4(tsp + 32 * rho + 16, hi);
        }
        if (step == 0 && rho != 1) prefetch(1);
      }
      if (co == 0 && grp == 1) {
        // body-column accumulator init: TRACE x_body + s phi_g(x_body); COMBINE2 sigma (D_body[u] - bias)
        unsigned long long v0[16];
#pragma unroll
        for (int q = 0; q < 16; q++) {
          const int i = T + 256 * (q & 7) + (q >> 3) * kM;
          const int e = (e0 + (q & 7) * d1 + (q >> 3) * d2) & (2 * kN - 1);
          const unsigned long long b = xp[e & (kN - 1)] - kBias51;
          const bool ng = (((sgn >> q) & 1u) ^ sgn_bit) != 0;
          v0[q] = (ng ? 0ull - b : b) + (trace ? xp[i] : 0ull);
        }
        group_sync(1);
#pragma unroll
        for (int q = 0; q < 16; q++) xp[T + 256 * (q & 7) + (q >> 3) * kM] = v0[q];
      }
      if (step == 0) prefetch(2);
      tm_wait_st();
      tmem_sync();  // spectra and the body init visible to both groups; every gather of the old mask words done
      if (trace) {
        cluster_arrive();  // phase A: this CTA no longer reads the old mask words
      } else if (co == 1) {
        // COMBINE2, mask column: the accumulator starts from zero (the D words were only needed by the gathers)
#pragma unroll
        for (int q = 0; q < 8; q++) xc[tid + 512 * q] = 0ull;
        __syncthreads();
      }

      // --------- this group's two limbs of column `co`: contraction, inverse, atomic word accumulation -------
#pragma unroll 1
      for (int k = 0; k < 2; k++) {
        const int l = l_first - 2 * k;
        double2 cur[8];
#pragma unroll
        for (int j = 0; j < 8; j++) cur[j] = make_double2(0.0, 0.0);
        auto fma_tile = [&](const double2 (&g)[8], int rho) {
#pragma unroll
          for (int h = 0; h < 2; h++) {
            double2 a[4];
            tm_ld4(tsp + 32 * rho + 16 * h, a);
#pragma unroll
            for (int j = 0; j < 4; j++) cmac(cur[4 * h + j], a[j], g[4 * h + j]);
          }
        };
        tm_wait_st();
        fma_tile(stage, 0);
#pragma unroll 1
        for (int rho = 1; rho < 3; rho++) {
          double2 g[8];
          {
            double2 lo[4], hi[4];
            tm_ld4(tpark + 32 * (rho - 1), lo);
            tm_ld4(tpark + 32 * (rho - 1) + 16, hi);
#pragma unroll
            for (int j = 0; j < 4; j++) { g[j] = lo[j]; g[4 + j] = hi[j]; }
          }
          fma_tile(g, rho);
        }
        // next output of this group: its second limb, or its first limb under the next step's matrix
        have_next = !(k == 1 && last);
        gnext = (k == 0 ? G : A.mat[last ? step : step + 1] + mat_off) +
                (size_t)(co * LOUT + (k == 0 ? l - 2 : l_first)) * kM + P0;
        inv_transform_g(cur, pa, w, grp, tw3, tw4, bs, prefetch);
        // word contribution of limb l: c3 | r2 | r1 << 17 | r0 << 34  (mod 2^51), added atomically because the
        // other group adds its limbs into the same words
#pragma unroll
        for (int q = 0; q < 16; q++) {
          const int i = T + 256 * (q & 7) + (q >> 3) * kM;
          const double v = (q < 8) ? cur[q & 7].x : cur[q & 7].y;
          unsigned long long add;
          if (l == 3) {
            const double t = trace ? fma(v, sgn_d, kMagic52 + 65536.0)
                                                : v + __hiloint2double(0x43380000, (int)(65536u - ((sgn >> q) & 1u)));
            add = (unsigned long long)(long long)(int)__funnelshift_r((uint32_t)__double2loint(t), (uint32_t)__double2hiint(t), 17);
          } else {
            const double t = fma(v, sgn_d, kMagic52);
            add = l == 2 ? magic_bits(t) : (l == 1 ? magic_bits(t) << 17 : (unsigned long long)((uint32_t)__double2loint(t) << 2) << 32);
          }
          atomicAdd(&xc[i], add);
        }
      }
      __syncthreads();   // all four limbs are in the words of this CTA's column
      if (trace) {
        cluster_wait();    // phase A complete: CTA 0 has gathered the old mask words, CTA 1 may overwrite them
        // ------- finish the words (mask to 51 bits, rsh for the next step); CTA 1 mirrors them into CTA 0 -------
#pragma unroll
        for (int q = 0; q < 8; q++) {
          const int i = tid + 512 * q;
          const unsigned long long U = xc[i] & kMask51;
          const unsigned long long Un = last ? U : rsh1_canon(U);
          xc[i] = Un;
          if (co == 1) st_cluster_u64(remote_mask + 8u * (uint32_t)i, Un);
        }
        cluster_arrive();  // phase B: new mask words written on both sides
        tmem_sync();
        cluster_wait();    // ... and visible before the next step's gathers
      } else {
        // y = phi_g(normalize(KS(D)));  out = normalize(S - y) X^t:  word = S - (R + k3) [- sigma (D_body[u] - bias)]
#pragma unroll
        for (int q = 0; q < 8; q++) {
          const int i = tid + 512 * q;
          put_digits_rot(dst, co, i, (sw[i] - xc[i]) & kMask51, A.rot_const);
        }
        tmem_sync();
      }
    }  // steps

    if (trace) {
      // copy-out: every CTA its own column, all 512 threads
#pragma unroll 4
      for (int q = 0; q < 8; q++) put_digits(dst, co, tid + 512 * q, xc[tid + 512 * q]);
    }
    // the next item's prologue rewrites the word buffers (CTA 0's mask column is also written by CTA 1)
    cluster_arrive();
    __syncthreads();
    cluster_wait();
  }
  tmem_free<512>(tmem_base, tid < 32);
}

}  // namespace fheram
