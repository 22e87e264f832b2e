// kernels_ks8.cuh -- latency variant of the key-switch kernels for the narrowest launches (the 12-step trace on
// word_size ciphertexts at the end of every read, src/ram.rs:457, and at the start of every write, :572; the last
// levels of the packing tree, src/ram.rs:435-449): one chain per CLUSTER of EIGHT CTAs (eight SMs), 512 threads each,
// one of the eight output polynomials (column, limb) of a key switch per CTA -- or of FOUR CTAs with two output
// polynomials each (groups 3 and 0, a shorter prefetch ring) for launches of up to a quarter of the SM count.
//
// k_ks6 (two CTAs) runs 2 forward + 2 (contraction + inverse) rounds one after the other per step and mirrors the new
// mask column over distributed shared memory (8.8 B/clk, tools/dsmem_probe.cu): 18.3 us per step.  Here a step is
//   phase A   every CTA rebuilds the mask words in its shared memory: old word + the four limb contributions of the
//             previous step, read from L2 (4 x 32 KiB, coalesced), reduced mod 2^51 and shifted (rsh 1);
//   forward   groups 0, 1, 2 (128 threads x 16 points, transform16.cuh) transform one mask limb each -- the same three
//             transforms in all eight CTAs, the spectra stay in the CTA's tensor memory;
//   output    group 3 contracts the three spectra with ITS column of the key (the 96 KiB were prefetched by cp.async
//             into a ring of 11 x 8 KiB since the previous step's contraction ended: no L2 round trip on the critical
//             path), runs ONE inverse transform and STORES the rounded, shifted result as the CTA's contribution slab;
//   body      nobody transforms the body column: its base term x + s phi_g(x) is rebuilt from the previous base and
//             contributions by groups 1, 2 of every CTA for an eighth of the positions, beside group 3's work.
// The contributions travel through L2 (two sets of eight slabs that alternate between the steps, plain stores, no
// atomics, nothing to clear), ordered by ONE cluster barrier per step.  No distributed shared memory.
// MODE_COMBINE2 (GLWEPacker two-sided combine, one step): the words are D = rsh1(a X^-t - b), the base term of the
// body column is s phi_g(D_body) only, and the output is normalize(S - y) X^t with S = rsh1(a X^-t + b) rebuilt from the
// operands at the end.
// MODE_MIXED (the packer level of a tree whose width is not a power of two): per item either MODE_COMBINE2 or one
// MODE_TRACE step without rotation (the one-sided combine), chosen by the operand table (mixed_src, kernels.cuh).
// Same integers as every other generation (tests/test_gpu_kernel_variants.py: "ks8"); keys in the order of k_prepare7.
#pragma once
#include "sync.cuh"
#include "tmem.cuh"
#include "transform16.cuh"
#include "words.cuh"

namespace fheram {

// per-phase cycles of ONE CTA (cluster 0, rank = A.stagger): thread 0 (group 0) slots 0..3 = phase A, forward,
// base term, barrier; thread 384 (group 3) slots 4..7 = wait for the spectra, contraction, inverse, contribution
#define KS8_TICK(slot_)                                                          \
  do {                                                                           \
    if (prof && (tid == 0 || tid == 384)) {                                      \
      const long long now_ = clock64();                                          \
      A.phase_cycles[(slot_)] += now_ - pt0;                                     \
      pt0 = now_;                                                                \
    }                                                                            \
  } while (0)

// staged 8 KiB chunks (of the 12 of one output column) per output group
__host__ __device__ constexpr int ks8_ring(int cl) { return cl == 8 ? 11 : 5; }
constexpr size_t ks8_smem(int cl) {
  return (size_t)256 * sizeof(double2) + (size_t)3 * kPad16 * sizeof(double2) + (size_t)kN * sizeof(unsigned long long) +
         (size_t)(8 / cl) * ks8_ring(cl) * 512 * sizeof(double2) + 32;
}

template <int CL, int MODE>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(512, 1) k_ks8(const VmpArgs A, const double2* __restrict__ tw16) {
  static_assert(CL == 8 || CL == 4, "cluster of eight or four CTAs");
  static_assert(MODE == MODE_TRACE || MODE == MODE_COMBINE2 || MODE == MODE_MIXED, "key-switch modes only");
  constexpr int LOUT = 4, NOUT = 2 * LOUT;
  constexpr int OPC = NOUT / CL;      // output polynomials per CTA
  constexpr int R = ks8_ring(CL);     // ring slots per output group
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* tw2 = reinterpret_cast<double2*>(smem_raw);
  double2* bufs = tw2 + 256;                                                          // exchange buffers of groups 0..2
  unsigned long long* xm = reinterpret_cast<unsigned long long*>(bufs + 3 * kPad16);  // mask words of the step
  double2* ring = reinterpret_cast<double2*>(xm + kN);
  uint32_t* slot = reinterpret_cast<uint32_t*>(ring + OPC * R * 512);

  const int tid = threadIdx.x, g = tid >> 7, t = tid & 127;
  const int rank = (int)cluster_ctarank();
  // output groups: group 3 (idle during the forward transforms) and, with two polynomials per CTA, group 0
  const bool out_group = g == 3 || (OPC == 2 && g == 0);
  const int og = g == 3 ? 0 : 1;
  const int o = rank * OPC + og;        // this group's output polynomial: column co (0 body, 1 mask), limb l
  const int l = o & 3;                  // (column o >> 2: 0 body, 1 mask)
  auto CT = [](int col, int limb) { return (limb * 2 + col) * kN; };

  if (tid < 32) tmem_alloc<256>(slot);
  if (tid < 256) tw2[tid] = __ldg(tw16 + tid);
  tmem_sync();
  const uint32_t tmem_base = *slot;
  const uint32_t tsp = tmem_base + ((uint32_t)(((tid >> 5) & 3) * 32) << 16);  // spectra rows at +0 / +64 / +128
  const uint32_t ttw = tsp + 192;                                             // 7 pass-3 twiddles (28 columns)
  if (g == 0) park_tw3x(ttw, tw16, t);
  tmem_sync();
  auto t3f = [&]() { return tm_tw3x(ttw); };
  // group 3 runs its inverse transform in the exchange buffer of group 1 (idle after the forward transforms)
  const T16 tc{bufs + (g < 3 ? g : 1) * kPad16, tw2, nullptr, t, g};
  const double sgn_d = (MODE == MODE_TRACE && A.sign < 0) ? -1.0 : 1.0;
  const uint32_t sgn_bit = (MODE == MODE_TRACE && A.sign < 0) ? 1u : 0u;

  const int n_clusters = gridDim.x / CL, cluster_id = blockIdx.x / CL;
  // per cluster: contribution slabs C[2 parities][8 outputs][N], body base terms B[2 parities][N]
  unsigned long long* Cs = reinterpret_cast<unsigned long long*>(A.scratch) + (size_t)cluster_id * kKs8ScratchWords;
  unsigned long long* Bs = Cs + (size_t)2 * NOUT * kN;
  const bool prof = A.phase_cycles != nullptr && cluster_id == 0 && rank == A.stagger;
  long long pt0 = 0;
  double2* stage = ring + og * (R * 512) + t;  // slot s, value j of this thread: stage[(4 s + j) * 128]

  for (int item = cluster_id; item < A.n_items; item += n_clusters) {
    int* dst = A.dst + (size_t)item * A.ct_stride;
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
    if (out_group) ring_fill<R>(stage, A.mat[0] + mat_off + (size_t)o * kM + t);

    // MODE_MIXED: the one-sided combine has no rotation
    const int rk = MODE == MODE_TRACE ? trace_rot(A, item, A.rot_const) : (MODE == MODE_MIXED && trace ? 0 : A.rot_const);
    // the words before step 0 of column col at position i:
    // TRACE x = rsh1(src X^rk);  COMBINE2 D = rsh1(a X^-t - b) (plus = false) or S = rsh1(a X^-t + b) (plus = true)
    auto x_src = [&](int col, int i, bool plus) {
      if (trace) {
        return trace_word(src, col, i, rk);
      } else {
        const int* pa = src;
        const int* pb = src + A.ct_stride;
        bool ng;
        const int j = rot_index(i, rk, ng);  // (a X^-t)[i] = +/- a[(i + t) mod 2N]
        long long Xa = limbs_value(pa[CT(col, 0) + j], pa[CT(col, 1) + j], pa[CT(col, 2) + j]);
        if (ng) Xa = -Xa;
        const long long Xb = limbs_value(pb[CT(col, 0) + i], pb[CT(col, 1) + i], pb[CT(col, 2) + i]);
        return rsh1_word(plus ? Xa + Xb : Xa - Xb);
      }
    };
    // ---- prologue: every CTA builds the mask words of step 0 itself
#pragma unroll 4
    for (int m = 0; m < 8; m++) xm[tid + 512 * m] = x_src(1, tid + 512 * m, false);
    __syncthreads();

    for (int step = 0; step < A.n_steps; step++) {
      const int ginv = A.gal_inv[step];
      const bool last = step + 1 == A.n_steps, first = step == 0;
      const unsigned long long* Cin = Cs + (size_t)((step + 1) & 1) * NOUT * kN;  // contributions of the previous step
      unsigned long long* Cout = Cs + (size_t)(step & 1) * NOUT * kN;
      const unsigned long long* Bin = Bs + (size_t)((step + 1) & 1) * kN;         // body base term of the previous step
      unsigned long long* Bout = Bs + (size_t)(step & 1) * kN;
      // ---------------- phase A: mask words of this step ----------------
      if (prof) pt0 = clock64();
      if (!first) {
        const ulonglong2* c4 = reinterpret_cast<const ulonglong2*>(Cin + (size_t)LOUT * kN);
        ulonglong2* x2 = reinterpret_cast<ulonglong2*>(xm);
#pragma unroll
        for (int m = 0; m < 4; m++) {
          const int i2 = tid + 512 * m;
          ulonglong2 w = x2[i2];
#pragma unroll
          for (int ll = 0; ll < LOUT; ll++) {
            const ulonglong2 c = __ldcg(c4 + (size_t)ll * (kN / 2) + i2);
            w.x += c.x; w.y += c.y;
          }
          x2[i2] = make_ulonglong2(rsh1_canon(w.x & kMask51), rsh1_canon(w.y & kMask51));
        }
        __syncthreads();
      }
      if (tid == 0) KS8_TICK(0); else if (prof && tid == 384) pt0 = clock64();

      // automorphism source of this thread's positions i = t + 128 m (+ 2048): e = i * ginv mod 2N
      const int e0 = (t * ginv) & (2 * kN - 1);
      const int d1 = (128 * ginv) & (2 * kN - 1);
      const int d2 = kM * (ginv & 3);
      if (g < 3) {
        // ---------------- forward transform of mask limb g ----------------
        {
          const int rho = g;
          double2 x[16];
#pragma unroll
          for (int m = 0; m < 16; m++) {
            const int ea = (e0 + m * d1) & (2 * kN - 1);
            x[m] = gather_digits(xm, ea, (ea + d2) & (2 * kN - 1), rho);
          }
          forward16(x, tc, t3f);
#pragma unroll
          for (int q = 0; q < 4; q++) {
            const double2 v[4] = {x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]};
            tm_st4(tsp + 64 * rho + 16 * q, v);
          }
        }
        tm_wait_st();
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        if (!out_group) asm volatile("bar.arrive 5, 512;" ::: "memory");  // the spectra are in tensor memory
        KS8_TICK(1);
        if (g >= 1) {
          // body column base term (TRACE x_body + s phi_g(x_body), COMBINE2 s phi_g(D_body)) for this CTA's share of
          // the positions: N / CL, 256 threads
          auto x_body = [&](int j) {
            if (first) return x_src(0, j, false);
            unsigned long long w = __ldcg(Bin + j);
#pragma unroll
            for (int ll = 0; ll < LOUT; ll++) w += __ldcg(Cin + (size_t)ll * kN + j);
            return rsh1_canon(w & kMask51);
          };
#pragma unroll
          for (int h = 0; h < kN / CL / 256; h++) {
            const int i = (kN / CL) * rank + (tid - 128) + 256 * h;
            const int e = (i * ginv) & (2 * kN - 1);
            const unsigned long long b = x_body(e & (kN - 1)) - kBias51;
            const bool ng = ((e >= kN ? 1u : 0u) ^ sgn_bit) != 0;
            __stcg(Bout + i, (ng ? 0ull - b : b) + (trace ? x_body(i) : 0ull));
          }
        }
      }
      if (out_group) {
        // ---------------- contraction, inverse transform, contribution of (co, l) ----------------
        asm volatile("bar.sync 5, 512;" ::: "memory");
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        KS8_TICK(4);
        const double2* gp = A.mat[step] + mat_off + (size_t)o * kM + t;
        double2 cur[16];
#pragma unroll
        for (int r = 0; r < 16; r++) cur[r] = make_double2(0.0, 0.0);
#pragma unroll
        for (int c = 0; c < 12; c++) {
          // chunks issued so far: min(12, R + c); pending after the wait: those beyond chunk c
          cp_async_wait_n((R + c < 12 ? R + c : 12) - c - 1);
          double2 m[4], a[4];
          const int s = c % R;
#pragma unroll
          for (int j = 0; j < 4; j++) m[j] = stage[(4 * s + j) * 128];
          if (c + R < 12) ring_issue(stage, gp, c + R, s);  // refill the slot just read
          tm_ld4(tsp + 64 * (c >> 2) + 16 * (c & 3), a);
#pragma unroll
          for (int j = 0; j < 4; j++) cmac(cur[4 * (c & 3) + j], a[j], m[j]);
        }
        KS8_TICK(5);
        if (!last) ring_fill<R>(stage, A.mat[step + 1] + mat_off + (size_t)o * kM + t);  // lands during the inverse and the next forward
        inverse16(cur, tc, t3f);
        KS8_TICK(6);
        // cur[m] = phi_g(vmp)[t + 128 m] + i phi_g(vmp)[t + 128 m + 2048] of limb l: round, shift to the limb's place
        unsigned long long* go = Cout + (size_t)o * kN + t;
        unsigned sgn = 0;
        if (!trace && l == 3) {
          // the carry chain runs in the pre-automorphism sign frame of each position (see k_ks3)
#pragma unroll
          for (int m = 0; m < 16; m++) {
            const int ea = (e0 + m * d1) & (2 * kN - 1);
            const int eb = (ea + d2) & (2 * kN - 1);
            sgn |= (ea >= kN ? 1u : 0u) << m;
            sgn |= (eb >= kN ? 1u : 0u) << (16 + m);
          }
        }
#pragma unroll
        for (int q = 0; q < 32; q++) {
          const int off = 128 * (q & 15) + (q >> 4) * kM;
          const double v = (q < 16) ? cur[q & 15].x : cur[q & 15].y;
          unsigned long long add;
          if (l == 3) {
            const double tt = trace ? fma(v, sgn_d, kMagic52 + 65536.0)
                                                 : v + __hiloint2double(0x43380000, (int)(65536u - ((sgn >> q) & 1u)));
            add = (unsigned long long)(long long)(int)__funnelshift_r((uint32_t)__double2loint(tt),
                                                                      (uint32_t)__double2hiint(tt), 17);
          } else {
            const double tt = fma(v, sgn_d, kMagic52);
            add = l == 2 ? magic_bits(tt)
                         : (l == 1 ? magic_bits(tt) << 17 : (unsigned long long)((uint32_t)__double2loint(tt) << 2) << 32);
          }
          __stcg(go + off, add);
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      if (tid == 0) KS8_TICK(2); else KS8_TICK(7);
      cluster_arrive();  // the contributions and the body base term of this step are written
      cluster_wait();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (tid == 0) KS8_TICK(3);
    }  // steps

    // ---------------- output: digits of the final words, 2 N / CL positions per CTA ----------------
    {
      const unsigned long long* Cin = Cs + (size_t)((A.n_steps + 1) & 1) * NOUT * kN;
      const unsigned long long* Bin = Bs + (size_t)((A.n_steps + 1) & 1) * kN;
#pragma unroll
      for (int m = 0; m < 2 * kN / CL / 512; m++) {
        const int wi = rank * (2 * kN / CL) + tid + 512 * m;
        const int col = wi >> 12, i = wi & (kN - 1);
        unsigned long long w = col == 1 ? (trace ? xm[i] : 0ull) : __ldcg(Bin + i);
#pragma unroll
        for (int ll = 0; ll < LOUT; ll++) w += __ldcg(Cin + (size_t)(col * LOUT + ll) * kN + i);
        if (trace) {
          const unsigned long long U = w & kMask51;
          dst[CT(col, 0) + i] = word_digit(U, 0);
          dst[CT(col, 1) + i] = word_digit(U, 1);
          dst[CT(col, 2) + i] = word_digit(U, 2);
        } else {
          // y = phi_g(normalize(KS(D)));  out = normalize(S - y) X^t
          const unsigned long long U = (x_src(col, i, true) - w) & kMask51;
          bool rneg;
          const int dd = rot_index(i, A.rot_const, rneg);  // a' * X^t
#pragma unroll
          for (int ll = 0; ll < 3; ll++) {
            const int dg = word_digit(U, ll);
            dst[CT(col, ll) + dd] = rneg ? -dg : dg;
          }
        }
      }
    }
    cluster_arrive();  // the next item rewrites the slabs and the mask words
    cluster_wait();
  }
  tmem_free<256>(tmem_base, tid < 32);
}

}  // namespace fheram
