// transform16.cuh -- the TWO-EXCHANGE transform (DESIGN.md 7.2 item 1, tools/t2_transform_probe.cu): a polynomial is
// transformed by 128 threads x 16 points with passes of 4 + 4 + 3 stages (two shared-memory exchanges).
//   thread / point maps of a group (t = thread in group, e = 11-bit point index):
//     pass 1 (stages 0-3):   e = t + 128 m          m  = e[10:7] in registers, uniform twiddles
//     pass 2 (stages 4-7):   e = 128 a + 8 m' + c   a = t >> 3, c = t & 7, m' = e[6:3]; twiddles per a (shared table)
//     pass 3 (stages 8-10):  e = 16 t + r           r  = e[3:0]; seven twiddles per thread (tensor memory)
//     spectrum value (t, r) is stored at position 128 r + t of the prepared matrices (k_prepare7)
//   exchange buffer: one polynomial, 16 blocks of 136 slots, P(e) = e + (e >> 4) (conflict free for all three
//   patterns).  The frequency order is private to this transform, hence its own prepared keys and GGSWs (k_prepare7).
#pragma once
#include "kernels.cuh"
#include "sync.cuh"
#include "tmem.cuh"

namespace fheram {

constexpr int kPad16 = 2176;
constexpr int kTw16Len = 256 + 128 * 7;  // global table: pass-2 twiddles [16][16], then pass-3 twiddles [128][7]

// pass-1 twiddles zeta(s, b), s < 4, are the first 16 entries of c_tw_lo (kernels.cuh)

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

// the seven pass-3 twiddles of thread t parked in tensor memory columns ttw .. ttw + 27, and their loader
__device__ __forceinline__ void park_tw3x(uint32_t ttw, const double2* tw16, int t) {
  const Tw3x w = load_tw3x(tw16, t);
  const double2 p0[4] = {w.w8, w.w9a, w.w9b, w.w10[0]};
  const double2 p1[4] = {w.w10[1], w.w10[2], w.w10[3], w.w10[3]};
  tm_st4(ttw, p0);
  tm_st4(ttw + 16, p1);
  tm_wait_st();
}
__device__ __forceinline__ Tw3x tm_tw3x(uint32_t ttw) {
  double2 p0[4], p1[4];
  tm_ld4(ttw, p0);
  tm_ld4(ttw + 16, p1);
  Tw3x w;
  w.w8 = p0[0]; w.w9a = p0[1]; w.w9b = p0[2]; w.w10[0] = p0[3];
  w.w10[1] = p1[0]; w.w10[2] = p1[1]; w.w10[3] = p1[2];
  return w;
}

// cp.async matrix stream of a contraction over 128 threads, prepared matrices in this frequency order (k_prepare7).
// Chunk c of output column gp (+ rho NOUT kM + 128 r, NOUT = 8 outputs) is row rho = c >> 2, frequencies
// r = 4 (c & 3) .. + 3; it goes to slot s of this thread's staging area stage[(4 s + j) * 128], one commit group per chunk
__device__ __forceinline__ void ring_issue(double2* stage, const double2* gp, int c, int s) {
  const double2* np = gp + (size_t)(c >> 2) * 8 * kM + 512 * (c & 3);
#pragma unroll
  for (int j = 0; j < 4; j++) cp_async16(stage + (4 * s + j) * 128, np + 128 * j);
  cp_async_commit();
}
// chunks 0 .. R - 1 into slots 0 .. R - 1
template <int R>
__device__ __forceinline__ void ring_fill(double2* stage, const double2* gp) {
#pragma unroll
  for (int c = 0; c < R; c++) ring_issue(stage, gp, c, c);
}

}  // namespace fheram
