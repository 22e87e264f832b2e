// kernels_ks5.cuh -- key switch (trace chains, two-sided packer combine) with ONE operation per SM
// spread over a CTA of 512 threads = two groups of 8 warps.
//
// Why: tools/ablate shows k_ks4 is bound by per-CTA latency, not by a saturated unit: the
// contraction waits one L2 round trip per matrix tile (the registers of 256 threads hold 32 KiB in
// flight), and with two CTAs per SM there is no tensor memory or shared memory left to stage tiles.
// Here both groups work on the SAME ciphertext (group g owns output column g: contraction, inverse
// transforms and word accumulation of that column; the three forward transforms are split 2 + 1),
// so the input spectra, the twiddles and the word buffer exist once per SM:
//   tensor memory (512 columns, all of it): per thread position 3 spectra (96 columns) + pass-3/4
//     twiddles (32), shared by the two groups, + per group two parked matrix tiles (2 x 32);
//   shared memory: words [2][N] (64 KiB) + one padded exchange buffer per group (2 x 36 KiB).
// The three matrix tiles of the NEXT output are fetched during the inverse transform of the current
// one: 8 LDG.128 per thread into a 32-register staging buffer at three points of the transform, the
// first two batches parked in tensor memory (tcgen05.st), the last one kept in registers.  The
// contraction then reads tiles from registers / tensor memory and no longer waits on L2.
// A single operation per SM also finishes in about half the time, which is what the narrow stages
// of a single read need (top of the packer tree, the final trace on word_size ciphertexts).
// Integer side (51-bit words), transforms and results are those of k_ks4.
#pragma once
#include "sync.cuh"
#include "tmem.cuh"
#include "transform_pad.cuh"
#include "words.cuh"

namespace fheram {

constexpr int kThreads5 = 512;
constexpr size_t kKs5Smem = (size_t)2 * kWorkPad * sizeof(double2) + (size_t)2 * kN * sizeof(long long) + 32;

template <int MODE>
__global__ void __launch_bounds__(kThreads5, 1) k_ks5(const VmpArgs A) {
  static_assert(MODE == MODE_TRACE || MODE == MODE_COMBINE2 || MODE == MODE_MIXED, "key-switch modes only");
  constexpr int LOUT = 4, NOUT = 2 * LOUT;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* work_all = reinterpret_cast<double2*>(smem_raw);                         // [2 groups] exchange buffers
  unsigned long long* xp = reinterpret_cast<unsigned long long*>(work_all + 2 * kWorkPad);  // [2 cols][N] words
  uint32_t* slot = reinterpret_cast<uint32_t*>(xp + 2 * kN);  // +0 tmem base, +8/+16 mbarriers of the groups

  const int tid = threadIdx.x, grp = tid >> 8, T = tid & 255, w = T >> 5, lane = T & 31;
  auto CT = [](int col, int limb) { return (limb * 2 + col) * kN; };

  if (tid < 32) tmem_alloc<512>(slot);
  BufSync bs{smem_u32(slot + 2 + 2 * grp), 0u};
  if (T == 0) buf_init(bs.mbar);
  tmem_sync();
  const uint32_t tmem_base = *slot;
  buf_release(bs);  // the group's buffer starts out free
  // columns of thread position (w, lane), the same for both groups: spectra +0/+32/+64, twiddles +96
  // (pass 3) / +112 (pass 4); parked tiles of group g at +128 + 64 g (+0, +32)
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
  const int co = grp;                       // output column of this group
  unsigned long long* xc = xp + co * kN;    // its words
  long long phase_t0 = A.phase_cycles ? clock64() : 0;

  for (int item = blockIdx.x; item < A.n_items; item += gridDim.x) {
    int* dst = A.dst + (size_t)item * A.ct_stride;
    // COMBINE2: words of S = rsh1(a X^-t + b), [2 cols][N], in this CTA's global scratch
    unsigned long long* sw = A.scratch
        ? reinterpret_cast<unsigned long long*>(A.scratch + (size_t)blockIdx.x * A.ct_stride) : nullptr;
    bool two = true;  // MODE_MIXED: the item has its second operand
    const int* src = mode_src<MODE>(A, item, two);
    // this item's path: TRACE steps, or the two-sided combine (a constant unless MODE_MIXED)
    const bool trace = MODE == MODE_MIXED ? !two : MODE == MODE_TRACE;
    const size_t mat_off = A.mat_div > 0 ? (size_t)(item / A.mat_div) * A.mat_stride : 0;

    // ---------------- prologue (once per item): group g converts column g -----------------
    if (trace) {
      // x = rsh1(src * X^rk)  (MODE_MIXED: the one-sided combine, no rotation)
      const int rk = trace_rot(A, item, MODE == MODE_MIXED ? 0 : A.rot_const);
#pragma unroll 4
      for (int m = 0; m < 16; m++) xc[T + 256 * m] = trace_word(src, co, T + 256 * m, rk);
    } else {
      // a1 = a X^-t;  D = rsh1(a1 - b) -> xp;  S = rsh1(a1 + b) -> sw
      const int* a = src;
      const int* b = src + A.ct_stride;
      const int tt = A.rot_const;
#pragma unroll 1
      for (int mc = 0; mc < 16; mc += 8) {
        int av[8][3], bv[8][3];
        bool ng[8];
#pragma unroll
        for (int mm = 0; mm < 8; mm++) {
          const int i = T + 256 * (mc + mm);
          const int j = rot_index(i, tt, ng[mm]);  // (a X^-t)[i] = +/- a[(i + t) mod 2N]
#pragma unroll
          for (int l = 0; l < 3; l++) { av[mm][l] = a[CT(co, l) + j]; bv[mm][l] = b[CT(co, l) + i]; }
        }
#pragma unroll
        for (int mm = 0; mm < 8; mm++) {
          const int i = T + 256 * (mc + mm);
          long long Xa = limbs_value(av[mm][0], av[mm][1], av[mm][2]);
          if (ng[mm]) Xa = -Xa;
          const long long Xb = limbs_value(bv[mm][0], bv[mm][1], bv[mm][2]);
          xc[i] = rsh1_word(Xa - Xb);
          sw[co * kN + i] = rsh1_word(Xa + Xb);
        }
      }
    }
    __syncthreads();
    PHASE_TICK(0);

    // matrix tile staging: `stage` holds tile 0 of the next output when a contraction starts
    double2 stage[8];
    const double2* gnext = A.mat[0] + mat_off + (size_t)(co * LOUT + LOUT - 1) * kM + P0;  // (step 0, limb 3, row 0)
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
    // the three prefetch points: tile 1 -> park 0, tile 2 -> park 1, tile 0 -> registers
    auto prefetch = [&](int point) {
      if (!have_next || A.stagger < 0) return;  // stagger < 0: timing experiment without tile prefetch
      if (point == 0) { fetch(1); }
      else if (point == 1) { park(0); fetch(2); }
      else { park(1); fetch(0); }
    };

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
#pragma unroll
      for (int q = 0; q < 16; q++) sgn |= ((((e0 + (q & 7) * d1 + (q >> 3) * d2) & (2 * kN - 1)) >= kN) ? 1u : 0u) << q;

      // ------------- forward transforms: group 0 rows 0 and 1, group 1 row 2 ---------------
      if (step == 0) prefetch(0);
#pragma unroll 1
      for (int rho = (grp == 0 ? 0 : 2); rho < (grp == 0 ? 2 : 3); rho++) {
        double2 x[8];
        // digit rho = bits [17 (2 - rho), +17) of the word = (funnel(lo, hi, s1) >> s2) & (2^17 - 1)
#pragma unroll
        for (int m = 0; m < 8; m++) {
          const int ea = (e0 + m * d1) & (2 * kN - 1);
          x[m] = gather_digits(xp + kN, ea, (ea + d2) & (2 * kN - 1), rho);
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
      if (grp == 1) {
        // body-column accumulator init, done by the group with the lighter forward share:
        //   TRACE: x_body + s phi_g(x_body);  COMBINE2: sigma (D_body[u] - bias)
        unsigned long long v0[16];
#pragma unroll
        for (int q = 0; q < 16; q++) {
          const int i = T + 256 * (q & 7) + (q >> 3) * kM;
          const int e = (e0 + (q & 7) * d1 + (q >> 3) * d2) & (2 * kN - 1);
          const unsigned long long b = xp[e & (kN - 1)] - kBias51;
          const bool ng = (((sgn >> q) & 1u) ^ sgn_bit) != 0;
          v0[q] = (ng ? 0ull - b : b) + (trace ? xp[i] : 0ull);
        }
        group_sync(1);  // every gather of the old body column precedes its stores
#pragma unroll
        for (int q = 0; q < 16; q++) xp[T + 256 * (q & 7) + (q >> 3) * kM] = v0[q];
      }
      if (step == 0) prefetch(2);
      tm_wait_st();
      tmem_sync();  // spectra (tensor memory) and the body-column init are visible to both groups
      if (grp == 1 && A.stagger > 0) {
        // the groups run identical phase sequences: offset them so that one group's butterflies
        // overlap the other's shared-memory exchanges instead of colliding with its butterflies
        const long long t0 = clock64();
        while (clock64() - t0 < A.stagger) {}
      }
      PHASE_TICK(2);

      // --------- contraction + inverse transform + word accumulation, column `co` -----------
#pragma unroll 1
      for (int l = LOUT - 1; l >= 0; l--) {
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
        tm_wait_st();  // parked tiles of this output
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
        PHASE_TICK(3);
        // next output: limb l - 1 of this column, or limb 3 of the next step's matrix
        have_next = !(l == 0 && last);
        gnext = (l > 0 ? G : A.mat[last ? step : step + 1] + mat_off) +
                (size_t)(co * LOUT + (l > 0 ? l - 1 : LOUT - 1)) * kM + P0;
        inv_transform_g(cur, pa, w, grp, tw3, tw4, bs, prefetch);
        PHASE_TICK(4);
        // cur[m] = phi_g(vmp)[T + 256 m] (+ i * [.. + 2048]); round and add into the word
        if (l == 3) {
#pragma unroll
          for (int q = 0; q < 16; q++) {
            const int i = T + 256 * (q & 7) + (q >> 3) * kM;
            const double v = (q < 8) ? cur[q & 7].x : cur[q & 7].y;
            double t;
            if (trace) t = fma(v, sgn_d, kMagic52 + 65536.0);
            else t = v + __hiloint2double(0x43380000, (int)(65536u - ((sgn >> q) & 1u)));
            const int c3 = (int)__funnelshift_r((uint32_t)__double2loint(t), (uint32_t)__double2hiint(t), 17);
            if (!trace && co == 1) xc[i] = (unsigned long long)(long long)c3;  // D mask words are dead
            else xc[i] += (unsigned long long)(long long)c3;
          }
        } else if (l == 2) {
#pragma unroll
          for (int q = 0; q < 16; q++) {
            const int i = T + 256 * (q & 7) + (q >> 3) * kM;
            const double v = (q < 8) ? cur[q & 7].x : cur[q & 7].y;
            xc[i] += magic_bits(fma(v, sgn_d, kMagic52));
          }
        } else if (l == 1) {
#pragma unroll
          for (int q = 0; q < 16; q++) {
            const int i = T + 256 * (q & 7) + (q >> 3) * kM;
            const double v = (q < 8) ? cur[q & 7].x : cur[q & 7].y;
            xc[i] += magic_bits(fma(v, sgn_d, kMagic52)) << 17;
          }
        } else {
#pragma unroll
          for (int q = 0; q < 16; q++) {
            const int i = T + 256 * (q & 7) + (q >> 3) * kM;
            const double v = (q < 8) ? cur[q & 7].x : cur[q & 7].y;
            const double t = fma(v, sgn_d, kMagic52);
            const unsigned long long W = xc[i] + ((unsigned long long)((uint32_t)__double2loint(t) << 2) << 32);
            if (trace) {
              const unsigned long long U = W & kMask51;
              xc[i] = last ? U : rsh1_canon(U);
            } else {
              put_digits_rot(dst, co, i, (sw[co * kN + i] - W) & kMask51, A.rot_const);
            }
          }
        }
        PHASE_TICK(5);
      }
      // both columns complete (the next forward gathers the mask words, the next body init gathers
      // the body words) and every read of the spectra precedes the next forward's tensor-memory stores
      tmem_sync();
    }  // steps

    if (trace) {
#pragma unroll 4
      for (int m = 0; m < 16; m++) put_digits(dst, co, T + 256 * m, xc[T + 256 * m]);
    }
    __syncthreads();  // xp reuse by the next item
    PHASE_TICK(6);
  }
  tmem_free<512>(tmem_base, tid < 32);
}

}  // namespace fheram
