// kernels_ext9.cuh -- latency variant of the external-product chain (CoordinatePrepared::product / product_inplace,
// src/coordinate_prepared.rs:147-177) for the narrowest launches (the second-coordinate products on word_size
// ciphertexts of every read and write, src/ram.rs:453-455): one chain per CLUSTER of eight CTAs (four with two output
// polynomials each), built like k_ks8 (kernels_ks8.cuh):
//   phase A   every CTA rebuilds the words of BOTH columns in its shared memory: bias + the four limb contributions of
//             the previous step per column, read from L2 (8 x 32 KiB), reduced mod 2^51 (step 0: the caller's limbs);
//   forward   groups 0, 1, 2 transform rows g and g + 3 of the six (limb, column) rows in two rounds -- the same six
//             transforms in every CTA, the spectra stay in the CTA's tensor memory;
//   output    group 3 (and group 0 with two polynomials per CTA) contracts the six spectra with ITS column of the GGSW
//             (24 chunks of 8 KiB through a cp.async ring of 7 (3) slots filled since the previous step; the rows of
//             round one are contracted while round two is transformed), runs ONE inverse transform and stores the
//             rounded, shifted result as the CTA's contribution slab in L2.
// One cluster barrier per step, no distributed shared memory, no atomics.  Same integers as k_ext8; the
// prepared GGSWs are in the frequency order of k_prepare7.
#pragma once
#include "kernels_ks8.cuh"

namespace fheram {

__host__ __device__ constexpr int ext9_ring(int cl) { return cl == 8 ? 7 : 3; }
constexpr size_t ext9_smem(int cl) {
  return (size_t)256 * sizeof(double2) + (size_t)3 * kPad16 * sizeof(double2) +
         (size_t)2 * kN * sizeof(unsigned long long) + (size_t)(8 / cl) * ext9_ring(cl) * 512 * sizeof(double2) + 32;
}

template <int CL>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(512, 1) k_ext9(const VmpArgs A, const double2* __restrict__ tw16) {
  static_assert(CL == 8 || CL == 4, "cluster of eight or four CTAs");
  constexpr int NR = 6, LOUT = 4, NOUT = 2 * LOUT, NCH = 4 * NR;
  constexpr int OPC = NOUT / CL;       // output polynomials per CTA
  constexpr int R = ext9_ring(CL);     // ring slots per output group
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* tw2 = reinterpret_cast<double2*>(smem_raw);
  double2* bufs = tw2 + 256;                                                          // exchange buffers of groups 0..2
  unsigned long long* xw = reinterpret_cast<unsigned long long*>(bufs + 3 * kPad16);  // [2 cols][N] words of the step
  double2* ring = reinterpret_cast<double2*>(xw + 2 * kN);
  uint32_t* slot = reinterpret_cast<uint32_t*>(ring + OPC * R * 512);

  const int tid = threadIdx.x, g = tid >> 7, t = tid & 127;
  const int rank = (int)cluster_ctarank();
  const bool out_group = g == 3 || (OPC == 2 && g == 0);
  const int og = g == 3 ? 0 : 1;
  const int o = rank * OPC + og;  // this group's output polynomial: column o >> 2, limb l
  const int l = o & 3;
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
  // group 3 runs its inverse transform in the exchange buffer of group 1 (idle after the forward transforms)
  const T16 tc{bufs + (g < 3 ? g : 1) * kPad16, tw2, nullptr, t, g};

  const int n_clusters = gridDim.x / CL, cluster_id = blockIdx.x / CL;
  // per cluster: contribution slabs C[2 parities][8 outputs][N]
  unsigned long long* Cs = reinterpret_cast<unsigned long long*>(A.scratch) + (size_t)cluster_id * kKs8ScratchWords;
  double2* stage = ring + og * (R * 512) + t;  // slot s, value j of this thread: stage[(4 s + j) * 128]
  auto ring_issue = [&](const double2* gp, int c, int s) {
    const double2* np = gp + (size_t)(c >> 2) * NOUT * kM + 512 * (c & 3);
#pragma unroll
    for (int j = 0; j < 4; j++) cp_async16(stage + (4 * s + j) * 128, np + 128 * j);
    cp_async_commit();
  };
  auto ring_fill = [&](const double2* Gmat) {
    const double2* gp = Gmat + (size_t)o * kM + t;
#pragma unroll
    for (int c = 0; c < R; c++) ring_issue(gp, c, c);
  };

  for (int item = cluster_id; item < A.n_items; item += n_clusters) {
    int* dst = A.dst + (size_t)item * A.ct_stride;
    const int* src;
    {
      long idx = item;
      if (A.src_div > 0) idx = item / A.src_div;
      else if (A.src_mod > 0) { int r = item % A.src_mod; idx = A.src_map ? A.src_map[r] : r; }
      src = A.src + idx * A.ct_stride;
    }
    const size_t mat_off = A.mat_div > 0 ? (size_t)(item / A.mat_div) * A.mat_stride : 0;
    if (out_group) ring_fill(A.mat[0] + mat_off);

    for (int step = 0; step < A.n_steps; step++) {
      const bool last = step + 1 == A.n_steps, first = step == 0;
      const unsigned long long* Cin = Cs + (size_t)((step + 1) & 1) * NOUT * kN;  // contributions of the previous step
      unsigned long long* Cout = Cs + (size_t)(step & 1) * NOUT * kN;
      // ---------------- phase A: words of both columns ----------------
      if (!first) {
        const ulonglong2* c2 = reinterpret_cast<const ulonglong2*>(Cin);
        ulonglong2* x2 = reinterpret_cast<ulonglong2*>(xw);
#pragma unroll 2
        for (int m = 0; m < 8; m++) {
          const int i2 = tid + 512 * m;                    // pair index in [2 cols][N / 2]
          const int col = i2 >> 11, p2 = i2 & (kN / 2 - 1);
          ulonglong2 w = make_ulonglong2(kBias51, kBias51);
#pragma unroll
          for (int ll = 0; ll < LOUT; ll++) {
            const ulonglong2 c = __ldcg(c2 + (size_t)(col * LOUT + ll) * (kN / 2) + p2);
            w.x += c.x; w.y += c.y;
          }
          x2[i2] = make_ulonglong2(w.x & kMask51, w.y & kMask51);
        }
        __syncthreads();
      }

      if (g < 3) {
        // ---------------- forward transforms: rows g (round one) and g + 3 (round two) ----------------
#pragma unroll 1
        for (int round = 0; round < 2; round++) {
          const int rho = g + 3 * round;
          const int col = rho & 1, limb = rho >> 1;
          double2 x[16];
          if (first) {
            // the caller's limbs as they are (any int32), like k_ext8
            const int* p = src + CT(col, limb) + t;
            asm volatile("" : "+l"(p));
#pragma unroll
            for (int m = 0; m < 16; m++) x[m] = make_double2(int_f64(p[128 * m]), int_f64(p[128 * m + kM]));
          } else {
            const unsigned long long* pw = xw + col * kN + t;
            const int s1 = limb == 0 ? 31 : (limb == 1 ? 17 : 0);
            const int s2 = limb == 0 ? 3 : 0;
#pragma unroll
            for (int m = 0; m < 16; m++) {
              const unsigned long long wa = pw[128 * m], wb = pw[128 * m + kM];
              x[m] = make_double2(
                  field_f64((__funnelshift_r((uint32_t)wa, (uint32_t)(wa >> 32), s1) >> s2) & 0x1ffffu, 0u),
                  field_f64((__funnelshift_r((uint32_t)wb, (uint32_t)(wb >> 32), s1) >> s2) & 0x1ffffu, 0u));
            }
          }
          forward16(x, tc, t3f);
#pragma unroll
          for (int q = 0; q < 4; q++) {
            const double2 v[4] = {x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]};
            tm_st4(tsp + 64 * rho + 16 * q, v);
          }
          tm_wait_st();
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          if (round == 0) asm volatile("bar.arrive 5, 512;" ::: "memory");            // rows 0..2 are in tensor memory
          else if (!out_group) asm volatile("bar.arrive 6, 512;" ::: "memory");       // rows 3..5
        }
      }
      if (out_group) {
        // ---------------- contraction, inverse transform, contribution of output o ----------------
        const double2* gp = A.mat[step] + mat_off + (size_t)o * kM + t;
        double2 cur[16];
#pragma unroll
        for (int r = 0; r < 16; r++) cur[r] = make_double2(0.0, 0.0);
        if (g == 3) {
          asm volatile("bar.sync 5, 512;" ::: "memory");
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
#pragma unroll
        for (int c = 0; c < NCH; c++) {
          if ((g == 3 && c == NCH / 2) || (g != 3 && c == 0)) {  // rows 3..5 (group 0 only starts after both rounds)
            asm volatile("bar.sync 6, 512;" ::: "memory");
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          }
          // chunks issued so far: min(24, R + c); pending after the wait: those beyond chunk c
          cp_async_wait_n((R + c < NCH ? R + c : NCH) - c - 1);
          double2 m[4], a[4];
          const int s = c % R;
#pragma unroll
          for (int j = 0; j < 4; j++) m[j] = stage[(4 * s + j) * 128];
          if (c + R < NCH) ring_issue(gp, c + R, s);  // refill the slot just read
          tm_ld4(tsp + 64 * (c >> 2) + 16 * (c & 3), a);
#pragma unroll
          for (int j = 0; j < 4; j++) {
            double2& acc = cur[4 * (c & 3) + j];
            acc.x = fma(a[j].x, m[j].x, fma(-a[j].y, m[j].y, acc.x));
            acc.y = fma(a[j].x, m[j].y, fma(a[j].y, m[j].x, acc.y));
          }
        }
        if (!last) ring_fill(A.mat[step + 1] + mat_off);  // lands during the inverse transform and the next forward
        inverse16(cur, tc, t3f);
        // cur[m] = vmp[t + 128 m] + i vmp[t + 128 m + 2048] of limb l: round, shift to the limb's place in the word
        unsigned long long* go = Cout + (size_t)o * kN + t;
#pragma unroll
        for (int q = 0; q < 32; q++) {
          const int off = 128 * (q & 15) + (q >> 4) * kM;
          const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
          unsigned long long add;
          if (l == 3) {
            const double tt = v + (kMagic52 + 65536.0);
            add = (unsigned long long)(long long)(int)__funnelshift_r((uint32_t)__double2loint(tt),
                                                                      (uint32_t)__double2hiint(tt), 17);
          } else {
            const double tt = v + kMagic52;
            add = l == 2 ? magic_bits(tt)
                         : (l == 1 ? magic_bits(tt) << 17 : (unsigned long long)((uint32_t)__double2loint(tt) << 2) << 32);
          }
          __stcg(go + off, add);
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      cluster_arrive();  // the contributions of this step are written
      cluster_wait();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }  // steps

    // ---------------- output: digits of the final words, 2 N / CL positions per CTA ----------------
    {
      const unsigned long long* Cin = Cs + (size_t)((A.n_steps + 1) & 1) * NOUT * kN;
#pragma unroll
      for (int m = 0; m < 2 * kN / CL / 512; m++) {
        const int wi = rank * (2 * kN / CL) + tid + 512 * m;
        const int col = wi >> 12, i = wi & (kN - 1);
        unsigned long long w = kBias51;
#pragma unroll
        for (int ll = 0; ll < LOUT; ll++) w += __ldcg(Cin + (size_t)(col * LOUT + ll) * kN + i);
        const unsigned long long U = w & kMask51;
        dst[CT(col, 0) + i] = word_digit(U, 0);
        dst[CT(col, 1) + i] = word_digit(U, 1);
        dst[CT(col, 2) + i] = word_digit(U, 2);
      }
    }
    cluster_arrive();  // the next item rewrites the slabs
    cluster_wait();
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

}  // namespace fheram
