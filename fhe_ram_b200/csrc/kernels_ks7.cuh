// kernels_ks7.cuh -- trace chains with the TWO-EXCHANGE transform (DESIGN.md 7.2 item 1, tools/t2_transform_probe.cu).
//
// k_ks4 transforms one polynomial at a time with 256 threads x 8 points and three shared-memory exchanges;
// its register passes are shared-memory bound and its eight inverse transforms per step run one after the other.
// Here a polynomial is transformed by 128 threads x 16 points with passes of 4 + 4 + 3 stages (two exchanges), and
// the two groups of a CTA work on two polynomials at once: group g owns output column g (contraction, inverse
// transform, in-place word accumulation of that column), the three forward transforms are split 2 + 1.
//   thread / point maps of a group (t = thread in group, e = 11-bit point index):
//     pass 1 (stages 0-3):   e = t + 128 m          m  = e[10:7] in registers, uniform twiddles
//     pass 2 (stages 4-7):   e = 128 a + 8 m' + c   a = t >> 3, c = t & 7, m' = e[6:3]; twiddles per a (shared table)
//     pass 3 (stages 8-10):  e = 16 t + r           r  = e[3:0]; seven twiddles per thread (tensor memory)
//     spectrum value (t, r) is stored at position 128 r + t of the prepared matrices (k_prepare7)
//   exchange buffer: one polynomial, 16 blocks of 136 slots, P(e) = e + (e >> 4) (conflict free for all three
//   patterns); the two groups take turns on it (a lock held from the first store to the last load of a transform's
//   exchanges), which keeps the CTA at 34 + 64 (words) + 4 (twiddles) = 102 KiB, two CTAs per SM.
//   tensor memory (256 columns per CTA): per thread position three spectra (3 x 64 columns) + pass-3 twiddles (28).
// Integer side: the 51-bit words of kernels_ks3.cuh, accumulated in place as in k_ks4 (each position is owned by one
// thread of the column's group).  The matrix tiles are not double buffered (the registers hold 16 accumulators).
// Same integers as every other generation; its own private frequency order, hence its own prepared trace keys.
#pragma once
#include "kernels_ks6.cuh"

namespace fheram {

constexpr int kPad16 = 2176;
constexpr size_t kKs7Smem = (size_t)256 * sizeof(double2) + (size_t)kPad16 * sizeof(double2) +
                            (size_t)2 * kN * sizeof(long long) + 32;
constexpr int kTw16Len = 256 + 128 * 7;  // global table: pass-2 twiddles [16][16], then pass-3 twiddles [128][7]

// pass-1 twiddles zeta(s, b), s < 4, are the first 16 entries of c_tw_lo (kernels.cuh)

__device__ __forceinline__ void gsync128(int g) { asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory"); }

// stages sl = SL0 .. 3 of a 16-point register block; tw(sl, bl) = twiddle of local block bl at local stage sl
template <int SL0, typename F>
__device__ __forceinline__ void fwd16(double2 (&x)[16], F&& tw) {
#pragma unroll
  for (int sl = SL0; sl < 4; sl++) {
    const int half = 8 >> sl;
#pragma unroll
    for (int i = 0; i < 16; i++)
      if (!(i & half)) bf(x[i], x[i + half], tw(sl, i >> (4 - sl)));
  }
}
template <int SL0, typename F>
__device__ __forceinline__ void inv16(double2 (&x)[16], F&& tw) {
#pragma unroll
  for (int sl = 3; sl >= SL0; sl--) {
    const int half = 8 >> sl;
#pragma unroll
    for (int i = 0; i < 16; i++)
      if (!(i & half)) ibf(x[i], x[i + half], tw(sl, i >> (4 - sl)));
  }
}

// pass-3 twiddles of one thread: zeta(8, 2t), zeta(9, 4t), zeta(9, 4t+2), zeta(10, 8t + 2k); odd blocks = i * even
struct Tw3x { double2 w8, w9a, w9b, w10[4]; };
__device__ __forceinline__ double2 tw3x(const Tw3x& t3, int sl, int bl) {
  if (sl == 1) return (bl & 1) ? mul_i(t3.w8) : t3.w8;
  if (sl == 2) { const double2 w = (bl & 2) ? t3.w9b : t3.w9a; return (bl & 1) ? mul_i(w) : w; }
  const double2 w = t3.w10[bl >> 1];
  return (bl & 1) ? mul_i(w) : w;
}

struct T16 {
  double2* buf;        // exchange buffer (shared by the groups of the CTA when lock != nullptr)
  const double2* tw2;  // shared memory: [16 a][16]
  unsigned* lock;      // nullptr: the buffer is private to the group
  int t, g;
};
__device__ __forceinline__ void t16_lock(const T16& c) {
  if (c.lock) {
    if (c.t == 0) { while (atomicCAS(c.lock, 0u, 1u) != 0u) {} }
    gsync128(c.g);
  }
}
__device__ __forceinline__ void t16_unlock(const T16& c) {
  gsync128(c.g);  // every load of the group is done
  if (c.lock && c.t == 0) { __threadfence_block(); atomicExch(c.lock, 0u); }
}
// x[m] = z[t + 128 m] on entry, spectrum values (t, r) on exit; T3 returns the pass-3 twiddles when they are needed
template <typename T3>
__device__ __forceinline__ void forward16(double2 (&x)[16], const T16& c, T3&& t3f) {
  const int t = c.t, a = t >> 3, cc = t & 7;
  fwd16<0>(x, [&](int sl, int bl) { return c_tw_lo[(1 << sl) + bl]; });
  t16_lock(c);
#pragma unroll
  for (int m = 0; m < 16; m++) c.buf[t + (t >> 4) + 136 * m] = x[m];
  gsync128(c.g);
#pragma unroll
  for (int m = 0; m < 16; m++) x[m] = c.buf[136 * a + 8 * m + cc + (m >> 1)];
  // pass-2 twiddles of block a: zeta(s, 2 j + 1) = i zeta(s, 2 j), so only the even entries are loaded (8 instead of 15
  // LDS.128 per transform: the table reads were a fifth of the shared-memory wavefronts of a key switch)
  const double2* ta = c.tw2 + 16 * a;
  fwd16<0>(x, [&](int sl, int bl) {
    const double2 w = ta[(1 << sl) + (bl & ~1)];
    return (sl > 0 && (bl & 1)) ? mul_i(w) : w;
  });
#pragma unroll
  for (int m = 0; m < 16; m++) c.buf[136 * a + 8 * m + cc + (m >> 1)] = x[m];
  __syncwarp();
#pragma unroll
  for (int r = 0; r < 16; r++) x[r] = c.buf[136 * a + 17 * cc + r];
  t16_unlock(c);
  const Tw3x t3 = t3f();
  fwd16<1>(x, [&](int sl, int bl) { return tw3x(t3, sl, bl); });
}
// spectrum values (t, r) on entry, x[m] = M z[t + 128 m] on exit
template <typename T3>
__device__ __forceinline__ void inverse16(double2 (&x)[16], const T16& c, T3&& t3f) {
  const int t = c.t, a = t >> 3, cc = t & 7;
  {
    const Tw3x t3 = t3f();
    inv16<1>(x, [&](int sl, int bl) { return tw3x(t3, sl, bl); });
  }
  t16_lock(c);
#pragma unroll
  for (int r = 0; r < 16; r++) c.buf[136 * a + 17 * cc + r] = x[r];
  __syncwarp();
#pragma unroll
  for (int m = 0; m < 16; m++) x[m] = c.buf[136 * a + 8 * m + cc + (m >> 1)];
  const double2* ta = c.tw2 + 16 * a;
  inv16<0>(x, [&](int sl, int bl) {
    const double2 w = ta[(1 << sl) + (bl & ~1)];
    return (sl > 0 && (bl & 1)) ? mul_i(w) : w;
  });
#pragma unroll
  for (int m = 0; m < 16; m++) c.buf[136 * a + 8 * m + cc + (m >> 1)] = x[m];
  gsync128(c.g);
#pragma unroll
  for (int m = 0; m < 16; m++) x[m] = c.buf[t + (t >> 4) + 136 * m];
  t16_unlock(c);
  inv16<0>(x, [&](int sl, int bl) { return c_tw_lo[(1 << sl) + bl]; });
}
__device__ __forceinline__ Tw3x load_tw3x(const double2* tw16, int t) {
  const double2* p = tw16 + 256 + 7 * t;
  Tw3x r;
  r.w8 = __ldg(p); r.w9a = __ldg(p + 1); r.w9b = __ldg(p + 2);
#pragma unroll
  for (int k = 0; k < 4; k++) r.w10[k] = __ldg(p + 3 + k);
  return r;
}

// ======================================================================================
// vmp_prepare in the frequency order of the 16-point transform: out[(rho, o)][128 r + t]
// (same raw layout, scaling and phi_g convention as k_prepare); two polynomials per CTA
// ======================================================================================
struct Prep7Args {
  PrepArgs p;
  const double2* tw16;
  int n_polys;
};
constexpr size_t kPrep7Smem = (size_t)256 * sizeof(double2) + (size_t)2 * kPad16 * sizeof(double2);
__global__ void __launch_bounds__(256, 2) k_prepare7(const Prep7Args P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* tw2 = reinterpret_cast<double2*>(smem_raw);
  double2* bufs = tw2 + 256;
  const PrepArgs& A = P.p;
  const int g = threadIdx.x >> 7, t = threadIdx.x & 127;
  tw2[threadIdx.x] = __ldg(P.tw16 + threadIdx.x);
  __syncthreads();
  const int poly = blockIdx.x * 2 + g;
  const bool active = poly < P.n_polys;
  const int pidx = active ? poly : P.n_polys - 1;  // inactive group repeats the last polynomial (barriers stay matched)
  const int per_mat = A.rows * A.cin * 2 * A.lout;
  const int mat = pidx / per_mat;
  const int r0 = pidx % per_mat;
  const int o = r0 % (2 * A.lout);
  const int rho = r0 / (2 * A.lout);
  const int co = o / A.lout, limb = o % A.lout;
  const int row = rho / A.cin, ci = rho % A.cin;
  const int* p = A.raw + (size_t)mat * A.raw_stride + ((((size_t)row * A.cin + ci) * A.lout + limb) * 2 + co) * kN;
  double2 x[16];
#pragma unroll
  for (int m = 0; m < 16; m++) {
    const int i = t + 128 * m;
    const int u = (i * A.gal_inv) & (2 * kN - 1);
    const int u2 = (u + kM * (A.gal_inv & 3)) & (2 * kN - 1);
    const int v = p[u & (kN - 1)], v2 = p[u2 & (kN - 1)];
    x[m] = make_double2((double)(u >= kN ? -v : v), (double)(u2 >= kN ? -v2 : v2));
  }
  T16 c{bufs + g * kPad16, tw2, nullptr, t, g};
  forward16(x, c, [&]() { return load_tw3x(P.tw16, t); });
  if (active) {
    double2* out = A.out + (size_t)mat * A.out_stride + ((size_t)rho * 2 * A.lout + o) * kM;
#pragma unroll
    for (int r = 0; r < 16; r++) out[128 * r + t] = make_double2(x[r].x * (1.0 / kM), x[r].y * (1.0 / kM));
  }
}

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

  const int tid = threadIdx.x, g = tid >> 7, t = tid & 127, lane = tid & 31;
  auto CT = [](int col, int limb) { return (limb * 2 + col) * kN; };

  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tw2[tid] = __ldg(tw16 + tid);
  if (tid == 0) slot[1] = 0u;
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *slot;
  // thread position (quadrant = warp & 3, lane): both groups address the same columns
  const uint32_t tsp = tmem_base + ((uint32_t)(((tid >> 5) & 3) * 32) << 16);  // spectra rows at +0 / +64 / +128
  const uint32_t ttw = tsp + 192;                                             // 7 pass-3 twiddles (28 columns)
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
  const T16 tc{buf, tw2, slot + 1, t, g};
  const double sgn_d = A.sign < 0 ? -1.0 : 1.0;
  const uint32_t sgn_bit = A.sign < 0 ? 1u : 0u;
  const int co = g;                         // output column of this group
  unsigned long long* xc = xp + co * kN;    // its words
  long long phase_t0 = A.phase_cycles ? clock64() : 0;

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

    // ------------------------------ prologue: x = rsh1(src * X^rk) ------------------------------
    {
      int rk = A.rot_const;
      if (A.rot_mod > 0) rk += A.rot_mul * (item % A.rot_mod);
      rk &= (2 * kN - 1);
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
          const unsigned long long ba = xp[ea & (kN - 1)] - kBias51;
          const bool na = ((ea >= kN ? 1u : 0u) ^ sgn_bit) != 0;
          v0[m] = (na ? 0ull - ba : ba) + xp[t + 128 * m];
        }
#pragma unroll
        for (int m = 0; m < 16; m++) {
          const int eb = (e0 + m * d1 + d2) & (2 * kN - 1);
          const unsigned long long bb = xp[eb & (kN - 1)] - kBias51;
          const bool nb = ((eb >= kN ? 1u : 0u) ^ sgn_bit) != 0;
          v1[m] = (nb ? 0ull - bb : bb) + xp[t + 128 * m + kM];
        }
        gsync128(1);  // every gather of the old body column precedes its stores
#pragma unroll
        for (int m = 0; m < 16; m++) { xp[t + 128 * m] = v0[m]; xp[t + 128 * m + kM] = v1[m]; }
      }
      tm_wait_st();
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();  // spectra and the body init are visible to both groups
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
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
              for (int j = 0; j < 4; j++) {
                double2& c = cur[8 * hf + 4 * q + j];
                c.x = fma(a[j].x, gt[4 * q + j].x, fma(-a[j].y, gt[4 * q + j].y, c.x));
                c.y = fma(a[j].x, gt[4 * q + j].y, fma(a[j].y, gt[4 * q + j].x, c.y));
              }
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
            const double tt = fma(v, sgn_d, kMagic52 + 65536.0);
            const int c3 = (int)__funnelshift_r((uint32_t)__double2loint(tt), (uint32_t)__double2hiint(tt), 17);
            xc[i] += (unsigned long long)(long long)c3;
          }
        } else if (l == 2) {
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const int i = t + 128 * (q & 15) + (q >> 4) * kM;
            const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
            xc[i] += magic_bits(fma(v, sgn_d, kMagic52));
          }
        } else if (l == 1) {
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const int i = t + 128 * (q & 15) + (q >> 4) * kM;
            const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
            xc[i] += magic_bits(fma(v, sgn_d, kMagic52)) << 17;
          }
        } else {
#pragma unroll
          for (int q = 0; q < 32; q++) {
            const int i = t + 128 * (q & 15) + (q >> 4) * kM;
            const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
            const double tt = fma(v, sgn_d, kMagic52);
            const unsigned long long W = xc[i] + ((unsigned long long)((uint32_t)__double2loint(tt) << 2) << 32);
            const unsigned long long U = W & kMask51;
            xc[i] = last ? U : rsh1_canon(U);
          }
        }
        PHASE_TICK(5);
      }
      // both columns complete before the next step's gathers; every spectrum read precedes the next stores
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }  // steps

#pragma unroll 4
    for (int m = 0; m < 16; m++) {
      const int i = tid + 256 * m;
#pragma unroll
      for (int col = 0; col < 2; col++) {
        const unsigned long long U = xp[col * kN + i];
        dst[CT(col, 0) + i] = word_digit(U, 0);
        dst[CT(col, 1) + i] = word_digit(U, 1);
        dst[CT(col, 2) + i] = word_digit(U, 2);
      }
    }
    __syncthreads();  // xp reuse by the next item
    PHASE_TICK(6);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base) : "memory");
  (void)lane;
}

}  // namespace fheram
