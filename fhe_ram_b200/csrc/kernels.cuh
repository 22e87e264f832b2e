// kernels.cuh -- sm_100a device code for the FHE-RAM hot path (N = 4096, base2k = 17).
//
// What these kernels replace (reference = phantomzone-org/fhe-ram; the arithmetic lives in
// its un-vendored Poulpy 0.3.2 FFT64 backend, SURVEY.md section 2.1):
//   vec_znx_dft_apply + vmp_apply_dft_to_dft + vec_znx_idft_apply_consume +
//   vec_znx_big_{add_small,automorphism,normalize} + the small rsh/rotate/add/sub ops that
//   glwe_external_product / glwe_automorphism[_add] / GLWEPacker::combine / glwe_trace issue
//   (call sites: src/coordinate_prepared.rs:156-175, src/ram.rs:435,457,540,572,616-629).
//
// One CTA (256 threads) owns one ciphertext operation.  A polynomial of N = 4096 integer
// coefficients is folded to M = 2048 complex points z_j = a_j + i a_{j+M} and transformed by
// a "shifted" radix-2 decimation: stage s, block b uses the single twiddle
//   zeta(s,b) = exp(i pi (1/4 + bitrev_s(b)) / 2^s)
// (Cooley-Tukey butterflies forward, Gentleman-Sande inverse), which evaluates the polynomial
// at the odd 4M-th roots psi^(4k+1) without a separate twist pass.  The frequency order is
// private: the prepared matrices are produced by the same transform.
//
// Thread/data mapping (e = 11-bit element index, T = thread, w = warp, l = lane):
//   pass 1 (stages 0-2, bits 10..8): T holds e = T + 256 m            (global loads coalesced)
//   block exchange through shared memory
//   pass 2 (stages 3-5, bits  7..5): warp w holds block w, lane l holds 256w + l + 32 m
//   pass 3 (stages 6-8, bits  4..2): lane (q,r) holds 256w + 32q + 4m + r
//   pass 4 (stages 9-10,bits  1..0): lane l holds 256w + 8l + j
//   final spectrum position of (T, j): 256w + 32j + l   (conflict-free, thread-private)
// Passes 2-4 only need __syncwarp; XOR swizzles S1/S2 keep every 16-byte access
// bank-conflict free.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace fheram {

constexpr int kN = 4096;
constexpr int kM = 2048;
constexpr int kLogN = 12;
constexpr int kK = 17;          // base2k
constexpr int kThreads = 256;

// Twiddle tables (device global memory), built on the host in long double.
struct Twiddles {
  const double2* tw6;    // [64]   zeta(6, B)
  const double2* tw7c;   // [64]   zeta(7, 2B)
  const double2* tw8c;   // [128]  zeta(8, 2k)
  const double2* tw9;    // [512]  zeta(9, b)
  const double2* tw10c;  // [512]  zeta(10, 2k)
};
// zeta(s,b) for s < 6 at index (1<<s)+b  (1 KiB, uniform / warp-uniform accesses only)
__constant__ double2 c_tw_lo[64];

// read-only 16-byte global load that the compiler may not sink past barriers (prefetch slots)
__device__ __forceinline__ double2 ldg_pinned(const double2* p) {
  double2 v;
  asm volatile("ld.global.nc.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ double2 mul_i(double2 w) { return make_double2(-w.y, w.x); }
// acc += a g (complex multiply-accumulate of the contraction)
__device__ __forceinline__ void cmac(double2& acc, const double2 a, const double2 g) {
  acc.x = fma(a.x, g.x, fma(-a.y, g.y, acc.x));
  acc.y = fma(a.x, g.y, fma(a.y, g.x, acc.y));
}
__device__ __forceinline__ double2 conj_(double2 w) { return make_double2(w.x, -w.y); }

// forward butterfly: (x, y) <- (x + w y, x - w y), 6 FP64 FMA-pipe ops
__device__ __forceinline__ void bf(double2& x, double2& y, const double2 w) {
  double xr = fma(w.x, y.x, fma(-w.y, y.y, x.x));
  double xi = fma(w.x, y.y, fma(w.y, y.x, x.y));
  y.x = fma(2.0, x.x, -xr);
  y.y = fma(2.0, x.y, -xi);
  x.x = xr;
  x.y = xi;
}
// inverse butterfly: (x, y) <- (x + y, (x - y) conj(w)), w passed un-conjugated
__device__ __forceinline__ void ibf(double2& x, double2& y, const double2 w) {
  double dr = x.x - y.x, di = x.y - y.y;
  x.x += y.x;
  x.y += y.y;
  y.x = fma(dr, w.x, di * w.y);
  y.y = fma(di, w.x, -(dr * w.y));
}

// radix-8 group over register index bits (2,1,0) = (first, second, third stage).
// wA: stage-A twiddle; wB0: twiddle of the first stage-B block (second = i*wB0);
// wC0, wC2: first/third stage-C blocks (second = i*wC0, fourth = i*wC2).
template <bool WITH_A>
__device__ __forceinline__ void radix8_fwd(double2 (&x)[8], double2 wA, double2 wB0, double2 wC0,
                                           double2 wC2) {
  if (WITH_A) {
    bf(x[0], x[4], wA); bf(x[1], x[5], wA); bf(x[2], x[6], wA); bf(x[3], x[7], wA);
  }
  const double2 wB1 = mul_i(wB0);
  bf(x[0], x[2], wB0); bf(x[1], x[3], wB0); bf(x[4], x[6], wB1); bf(x[5], x[7], wB1);
  bf(x[0], x[1], wC0); bf(x[2], x[3], mul_i(wC0));
  bf(x[4], x[5], wC2); bf(x[6], x[7], mul_i(wC2));
}
template <bool WITH_A>
__device__ __forceinline__ void radix8_inv(double2 (&x)[8], double2 wA, double2 wB0, double2 wC0,
                                           double2 wC2) {
  ibf(x[0], x[1], wC0); ibf(x[2], x[3], mul_i(wC0));
  ibf(x[4], x[5], wC2); ibf(x[6], x[7], mul_i(wC2));
  const double2 wB1 = mul_i(wB0);
  ibf(x[0], x[2], wB0); ibf(x[1], x[3], wB0); ibf(x[4], x[6], wB1); ibf(x[5], x[7], wB1);
  if (WITH_A) {
    ibf(x[0], x[4], wA); ibf(x[1], x[5], wA); ibf(x[2], x[6], wA); ibf(x[3], x[7], wA);
  }
}

// swizzles on the element index (bits 5 and below / bits 5..3 only -> valid on local or global e)
__device__ __forceinline__ int S1(int e) { return e ^ (((e >> 5) & 1) << 2); }
__device__ __forceinline__ int S2(int e) { return e ^ ((e >> 3) & 7); }

struct Tw34 {  // per-thread twiddles of passes 3 and 4 (loaded once, reused across polynomials)
  double2 a3, b3, c3, d3;      // zeta(6,B), zeta(7,2B), zeta(8,4B), zeta(8,4B+2)
  double2 b4a, b4b, c4a, c4b;  // zeta(9,2B4), zeta(9,2B4+1), zeta(10,4B4), zeta(10,4B4+2)
};
__device__ __forceinline__ Tw34 load_tw34(const Twiddles& tw, int w, int lane) {
  Tw34 t;
  const int B = 8 * w + (lane >> 2);
  t.a3 = __ldg(tw.tw6 + B);
  t.b3 = __ldg(tw.tw7c + B);
  t.c3 = __ldg(tw.tw8c + 2 * B);
  t.d3 = __ldg(tw.tw8c + 2 * B + 1);
  const int B4 = 32 * w + lane;
  t.b4a = __ldg(tw.tw9 + 2 * B4);
  t.b4b = __ldg(tw.tw9 + 2 * B4 + 1);
  t.c4a = __ldg(tw.tw10c + 2 * B4);
  t.c4b = __ldg(tw.tw10c + 2 * B4 + 1);
  return t;
}

// ---- forward transform pieces -------------------------------------------------------
// pass 1 on x[m] = z[T + 256 m]; result stored to spec[S1(e)]
__device__ __forceinline__ void fwd_pass1_store(double2 (&x)[8], double2* spec, int T) {
  radix8_fwd<true>(x, c_tw_lo[1], c_tw_lo[2], c_tw_lo[4], c_tw_lo[6]);
#pragma unroll
  for (int m = 0; m < 8; m++) spec[S1(T + 256 * m)] = x[m];
}
// passes 2-4 of warp w on its 256-element block of `spec` (after a block-level sync);
// leaves the spectrum in final layout spec[256w + 32j + lane].
__device__ __forceinline__ void fwd_warp_passes(double2* spec, int w, int lane, const Tw34& t) {
  double2* base = spec + 256 * w;
  double2 x[8];
#pragma unroll
  for (int m = 0; m < 8; m++) x[m] = base[S1(lane + 32 * m)];
  radix8_fwd<true>(x, c_tw_lo[8 + w], c_tw_lo[16 + 2 * w], c_tw_lo[32 + 4 * w],
                   c_tw_lo[32 + 4 * w + 2]);
#pragma unroll
  for (int m = 0; m < 8; m++) base[S1(lane + 32 * m)] = x[m];
  __syncwarp();
  const int qr = 32 * (lane >> 2) + (lane & 3);
#pragma unroll
  for (int m = 0; m < 8; m++) x[m] = base[S1(qr + 4 * m)];
  radix8_fwd<true>(x, t.a3, t.b3, t.c3, t.d3);
  __syncwarp();
#pragma unroll
  for (int m = 0; m < 8; m++) base[S2(qr + 4 * m)] = x[m];
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 8; j++) x[j] = base[S2(8 * lane + j)];
  // pass 4 = stages 9,10: stage-B twiddles differ per half (two stage-9 blocks)
  {
    bf(x[0], x[2], t.b4a); bf(x[1], x[3], t.b4a); bf(x[4], x[6], t.b4b); bf(x[5], x[7], t.b4b);
    bf(x[0], x[1], t.c4a); bf(x[2], x[3], mul_i(t.c4a));
    bf(x[4], x[5], t.c4b); bf(x[6], x[7], mul_i(t.c4b));
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 8; j++) base[32 * j + lane] = x[j];
}

// ---- inverse transform pieces -------------------------------------------------------
// x[j] = spectrum values in final layout (thread-private).  Runs stages 10..3 inside the warp
// using `work` (block-shared 2048 x double2), then the block exchange and stages 2..0.
// On return x[m] = M * z[T + 256 m].  `pre_sync2` runs between the two block barriers (after
// the previous users of registers are dead) -- used to gather epilogue operands.
template <typename F>
__device__ __forceinline__ void inv_transform(double2 (&x)[8], double2* work, int T, int w,
                                              int lane, const Tw34& t, F&& pre_sync2) {
  double2* wb = work + 256 * w;
  {
    ibf(x[0], x[1], t.c4a); ibf(x[2], x[3], mul_i(t.c4a));
    ibf(x[4], x[5], t.c4b); ibf(x[6], x[7], mul_i(t.c4b));
    ibf(x[0], x[2], t.b4a); ibf(x[1], x[3], t.b4a); ibf(x[4], x[6], t.b4b); ibf(x[5], x[7], t.b4b);
  }
#pragma unroll
  for (int j = 0; j < 8; j++) wb[S2(8 * lane + j)] = x[j];
  __syncwarp();
  const int qr = 32 * (lane >> 2) + (lane & 3);
#pragma unroll
  for (int m = 0; m < 8; m++) x[m] = wb[S2(qr + 4 * m)];
  radix8_inv<true>(x, t.a3, t.b3, t.c3, t.d3);
  __syncwarp();
#pragma unroll
  for (int m = 0; m < 8; m++) wb[S1(qr + 4 * m)] = x[m];
  __syncwarp();
#pragma unroll
  for (int m = 0; m < 8; m++) x[m] = wb[S1(lane + 32 * m)];
  radix8_inv<true>(x, c_tw_lo[8 + w], c_tw_lo[16 + 2 * w], c_tw_lo[32 + 4 * w],
                   c_tw_lo[32 + 4 * w + 2]);
#pragma unroll
  for (int m = 0; m < 8; m++) wb[S1(lane + 32 * m)] = x[m];
  __syncthreads();
  pre_sync2();
#pragma unroll
  for (int m = 0; m < 8; m++) x[m] = work[S1(T + 256 * m)];
  __syncthreads();
  radix8_inv<true>(x, c_tw_lo[1], c_tw_lo[2], c_tw_lo[4], c_tw_lo[6]);
}

// ---- integer helpers (balanced base-2^17 digits) -------------------------------------
__device__ __forceinline__ long long sext17(long long x) { return (x << 47) >> 47; }
__device__ __forceinline__ int sext17i(int x) {
  int r;
  asm("bfe.s32 %0, %1, 0, 17;" : "=r"(r) : "r"(x));
  return r;
}

// Poulpy's vec_znx_rsh_inplace(k = 1) on a 3-limb coefficient, step by step in 32-bit
// arithmetic (oracle vz_rsh_inplace: shift by one limb, left-shift by 16 inside the
// normalisation): equals the balanced digits of ceil(X/2), X = a0 2^34 + a1 2^17 + a2.
__device__ __forceinline__ void rsh1_3(int a0, int a1, int a2, int& d0, int& d1, int& d2) {
  int carry = (a2 + 1) >> 1;                 // limb shifted out: carry only (digit -(a2&1) dropped)
  int dpc = (-(a1 & 1) << 16) + carry;       // low bit of limb 1 lands on top of limb 2
  d2 = sext17i(dpc);
  carry = ((a1 + 1) >> 1) + ((dpc - d2) >> 17);
  dpc = (-(a0 & 1) << 16) + carry;
  d1 = sext17i(dpc);
  carry = ((a0 + 1) >> 1) + ((dpc - d1) >> 17);
  d0 = sext17i(carry);
}

// automorphism X -> X^g on coefficient index i: returns destination index, sets neg
__device__ __forceinline__ int auto_index(int i, int g, bool& neg) {
  int e = (i * g) & (2 * kN - 1);
  neg = e >= kN;
  return e & (kN - 1);
}
// multiplication by X^k (k taken mod 2N, non-negative): destination of coefficient i
__device__ __forceinline__ int rot_index(int i, int k, bool& neg) {
  int e = (i + k) & (2 * kN - 1);
  neg = e >= kN;
  return e & (kN - 1);
}

// ======================================================================================
// Work description shared by all vmp-class launches
// ======================================================================================
constexpr int kMaxSteps = 12;

enum Mode : int {
  MODE_TRACE = 1,    // chain of { rsh 1; x <- x +/- phi_g(KS(x)) }  (trace / one-sided combine)
  MODE_COMBINE2 = 2, // GLWEPacker two-sided combine
  MODE_AUTO = 3,     // x <- phi_g(normalize(KS(x)))  (glwe_automorphism)
  MODE_EXPAND = 4,   // GGSW expand row: (KS_tsk(mask), + body on the mask column)
  MODE_MIXED = 5,    // GLWEPacker level whose pairs may lack their second operand: per item the two-sided
                     // combine (COMBINE2) or the one-sided one (one TRACE step, no rotation)
};

struct VmpArgs {
  int n_items;
  // source ciphertexts: item -> src + src_map[item % src_mod] * ct_stride (src_map may be null:
  // identity on item % src_mod; src_mod == 0: index = item)
  const int* src;
  const int* src_map;
  int src_mod;
  int src_div;       // if > 0: index = item / src_div (takes precedence over src_mod)
  // second operand of COMBINE2: a = src[2*item], b = src[2*item+1]
  // MODE_MIXED: pair p = item % src_div of group item / src_div; op = src_map[p] (offset << 1 | has_b):
  //   a = src[group * src_mod + (op >> 1)], b = the ciphertext after a when op & 1 (else the one-sided combine)
  int* dst;          // item -> dst + item * ct_stride
  int* scratch;      // per-CTA scratch: gridDim.x * 2 * ct_stride ints
  long ct_stride;    // ints per ciphertext
  // matrices: step s of item -> mat[s] + (item / mat_div) * mat_stride   (mat_div 0: shared)
  const double2* mat[kMaxSteps];
  int gal[kMaxSteps];      // automorphism exponent g (mod 2N, positive) per step
  int gal_inv[kMaxSteps];  // g^-1 mod 2N: phi_g(x)[j] = +/- x[j * g^-1 mod 2N]
  int mat_div;
  long mat_stride;         // in double2
  int n_steps;
  int sign;                // MODE_TRACE: +1 automorphism_add, -1 automorphism_sub_negate
  int rot_mod;             // MODE_TRACE pre-rotation: X^(rot_mul * (item % rot_mod)) (0: none)
  int rot_mul;
  int rot_const;           // added rotation (mod 2N), e.g. COMBINE2's t
  Twiddles tw;
  // optional per-phase cycle counters (debug / DESIGN.md phase breakdown): gridDim.x * 8 slots
  // 0 prologue, 1 forward pass 1, 2 forward warp passes, 3 contraction, 4 inverse, 5 epilogue, 6 rest
  long long* phase_cycles;
  int stagger;  // k_ks5: cycles by which group 1 trails group 0 after a CTA barrier (tuning knob)
};
// MODE_MIXED operands of `item`: returns a; two = whether b (the ciphertext after a) is present
__device__ __forceinline__ const int* mixed_src(const VmpArgs& A, int item, bool& two) {
  const int op = A.src_map[item % A.src_div];
  two = (op & 1) != 0;
  return A.src + ((long)(item / A.src_div) * A.src_mod + (op >> 1)) * A.ct_stride;
}
// source ciphertext of `item` through src_div / src_mod / src_map
__device__ __forceinline__ const int* item_src(const VmpArgs& A, int item) {
  long idx = item;
  if (A.src_div > 0) idx = item / A.src_div;
  else if (A.src_mod > 0) { int r = item % A.src_mod; idx = A.src_map ? A.src_map[r] : r; }
  return A.src + idx * A.ct_stride;
}
// the same for the key-switch modes: COMBINE2 reads the pair at 2 item, MODE_MIXED the operand table (two = b present)
template <int MODE>
__device__ __forceinline__ const int* mode_src(const VmpArgs& A, int item, bool& two) {
  if constexpr (MODE == MODE_MIXED) return mixed_src(A, item, two);
  else if constexpr (MODE == MODE_COMBINE2) return A.src + 2L * item * A.ct_stride;
  else return item_src(A, item);
}
#define PHASE_TICK(ph)                                                      \
  do {                                                                      \
    if (A.phase_cycles && threadIdx.x == 0) {                               \
      const long long now_ = clock64();                                     \
      A.phase_cycles[(size_t)blockIdx.x * 8 + (ph)] += now_ - phase_t0;     \
      phase_t0 = now_;                                                      \
    }                                                                       \
  } while (0)

// ======================================================================================
// The fused kernel: glwe_automorphism and the GGSW expand rows of the inverse address.
// Key-switch modes use keys prepared as phi_g(K) (k_prepare with gal_inv): since
// phi_g(sum_r a_r * K_r) = sum_r phi_g(a_r) * phi_g(K_r), transforming phi_g(x) instead of x makes
// the inverse transform deliver phi_g(KS(x)) directly in natural coefficient order, so every
// epilogue works on the thread's own positions (no scatter) and only reads of the small input
// are gathered.
//   R     limbs of the input ciphertext that are transformed (mask column only)
//   LOUT  limbs of the matrix / big result;   LRES  limbs kept after normalisation
// Shared memory: R spectra (32 KiB each) + 32 KiB work.
// ======================================================================================
template <int R, int LOUT, int LRES, int MODE>
__global__ void __launch_bounds__(kThreads, 1) k_vmp(const VmpArgs A) {
  static_assert(MODE == MODE_AUTO || MODE == MODE_EXPAND, "automorphism / expand only");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double2* spectra = reinterpret_cast<double2*>(smem_raw);
  double2* work = spectra + (size_t)R * kM;

  const int T = threadIdx.x, w = T >> 5, lane = T & 31;
  const Tw34 tw = load_tw34(A.tw, w, lane);
  constexpr int NOUT = 2 * LOUT;
  // layout of a ciphertext buffer: [limb][col][N]
  auto CT = [](int col, int limb) { return (limb * 2 + col) * kN; };

  long long phase_t0 = A.phase_cycles ? clock64() : 0;
  for (int item = blockIdx.x; item < A.n_items; item += gridDim.x) {
    int* dst = A.dst + (size_t)item * A.ct_stride;

    const int* src = item_src(A, item);
    const size_t mat_off = A.mat_div > 0 ? (size_t)(item / A.mat_div) * A.mat_stride : 0;

    for (int step = 0; step < A.n_steps; step++) {
      const double2* G = A.mat[step] + mat_off;
      PHASE_TICK(0);
      // input of the transforms
      const int* xin = src;
      constexpr bool PERM = MODE == MODE_AUTO;
      const int ginv = A.gal_inv[step];

      // --------------------------- forward transforms ------------------------------
      // integer limbs of row rho+1 are requested while row rho is converted and transformed
      auto load_row = [&](int rho, int (&v)[16]) {
        const int* p = xin + CT(1, rho);
#pragma unroll
        for (int m = 0; m < 8; m++) {
          const int i = T + 256 * m;
          if (PERM) {
            // phi_g(x)[i] and phi_g(x)[i + M]: (i + M) g^-1 = i g^-1 + M (g^-1 mod 4)  (mod 2N)
            const int u = (i * ginv) & (2 * kN - 1);
            const int u2 = (u + kM * (ginv & 3)) & (2 * kN - 1);
            const int a = p[u & (kN - 1)], b = p[u2 & (kN - 1)];
            v[m] = u >= kN ? -a : a;
            v[m + 8] = u2 >= kN ? -b : b;
          } else {
            v[m] = p[i];
            v[m + 8] = p[i + kM];
          }
        }
      };
      int nx[16];
      load_row(0, nx);
#pragma unroll 1
      for (int rho = 0; rho < R; rho++) {
        double2 x[8];
#pragma unroll
        for (int m = 0; m < 8; m++) x[m] = make_double2((double)nx[m], (double)nx[m + 8]);
        if (rho + 1 < R) load_row(rho + 1, nx);
        fwd_pass1_store(x, spectra + (size_t)rho * kM, T);
      }
      __syncthreads();
      PHASE_TICK(1);
#pragma unroll 1
      for (int rho = 0; rho < R; rho++) fwd_warp_passes(spectra + (size_t)rho * kM, w, lane, tw);
      PHASE_TICK(2);
      // no barrier needed: the contraction reads only what this thread wrote

      // --------------- contraction + inverse transform + epilogue ------------------
      // Both output columns of limb l are contracted together (each input spectrum value is read
      // from shared memory once for two outputs); carries fit 32 bits (|big| < 2^47).
      // (A register prefetch of the next output's matrix rows across the inverse transform was
      // measured and does not overlap: the L2 port runs at ~55 B/clk/SM either way.)
      const int P0 = 256 * w + lane;
      int carryA[16], carryB[16];    // running carry of column 0 / column 1
#pragma unroll
      for (int q = 0; q < 16; q++) { carryA[q] = 0; carryB[q] = 0; }
#pragma unroll 1
      for (int l = LOUT - 1; l >= 0; l--) {
        double2 cur[8], nxt[8];
#pragma unroll
        for (int j = 0; j < 8; j++) { cur[j] = make_double2(0.0, 0.0); nxt[j] = make_double2(0.0, 0.0); }
#pragma unroll(R <= 4 ? R : 2)
        for (int rho = 0; rho < R; rho++) {
          const double2* gp = G + ((size_t)rho * NOUT + l) * kM + P0;
          const double2* ap = spectra + (size_t)rho * kM + P0;
          double2 g0[8], g1[8];
#pragma unroll
          for (int j = 0; j < 8; j++) { g0[j] = __ldg(gp + 32 * j); g1[j] = __ldg(gp + (size_t)LOUT * kM + 32 * j); }
#pragma unroll
          for (int j = 0; j < 8; j++) {
            const double2 a = ap[32 * j];
            cmac(cur[j], a, g0[j]);
            cmac(nxt[j], a, g1[j]);
          }
        }
        PHASE_TICK(3);
#pragma unroll 1
        for (int co = 0; co < 2; co++) {
          const bool has_small = l < R;  // the small operand has R limbs
          inv_transform(cur, work, T, w, lane, tw, [&]() {});
          PHASE_TICK(4);
          int sv[16];  // small global operands of this output, requested together
          if (MODE == MODE_EXPAND && co == 1 && has_small) {
#pragma unroll
            for (int q = 0; q < 16; q++) sv[q] = xin[CT(0, l) + T + 256 * (q & 7) + (q >> 3) * kM];
          } else if (MODE == MODE_AUTO && co == 0 && has_small) {
#pragma unroll
            for (int q = 0; q < 16; q++) {
              bool ng;
              sv[q] = xin[CT(0, l) + auto_index(T + 256 * (q & 7) + (q >> 3) * kM, ginv, ng)];
            }
          }
          // cur[m] = M * phi_g(vmp)[T + 256 m] (natural order; plain vmp for EXPAND)
#pragma unroll
          for (int q = 0; q < 16; q++) {
            const int i = T + 256 * (q & 7) + (q >> 3) * kM;
            const double v = (q < 8) ? cur[q & 7].x : cur[q & 7].y;
            long long big = __double2ll_rn(v);
            bool neg = false;
            if (MODE == MODE_EXPAND) {
              if (co == 1 && has_small) big += (long long)sv[q];
            } else {
              // phi(normalize(KS(x))): run the carry chain in the pre-automorphism sign frame
              auto_index(i, ginv, neg);
              if (neg) big = -big;
              if (co == 0 && has_small) big += (long long)sv[q];
            }
            const long long t = big + (long long)carryA[q];
            const int c = (int)((t + 65536) >> kK);
            const int dg = (int)t - (c << kK);
            carryA[q] = c;
            if (l < LRES) dst[CT(co, l) + i] = neg ? -dg : dg;
          }
          PHASE_TICK(5);
          // rotate the per-column state so the loop body always works on (cur, carryA)
#pragma unroll
          for (int j = 0; j < 8; j++) { const double2 t = cur[j]; cur[j] = nxt[j]; nxt[j] = t; }
#pragma unroll
          for (int q = 0; q < 16; q++) { int t = carryA[q]; carryA[q] = carryB[q]; carryB[q] = t; }
        }
      }
    }  // steps

    __syncthreads();  // spectra reuse by the next item
    PHASE_TICK(6);
  }
}

// ======================================================================================
// vmp_prepare: raw int32 limbs of a GGSW / GGLWE -> spectra in contraction layout.
// raw layout (MatZnx): [row][ci][limb][co][N];  out: [rho = row*CIN+ci][o = co*LOUT+limb][M]
// one CTA per (matrix, rho, o) polynomial.
// ======================================================================================
struct PrepArgs {
  const int* raw;      // n_mat matrices, raw_stride ints apart
  double2* out;        // out_stride double2 apart
  long raw_stride, out_stride;
  int rows, cin, lout; // polys per matrix = rows*cin*2*lout
  int gal_inv;         // 1: plain; else prepare phi_g(matrix) (g^-1 mod 2N), see k_vmp
  Twiddles tw;
};
__global__ void __launch_bounds__(kThreads, 2) k_prepare(const PrepArgs A) {
  __shared__ __align__(16) double2 spec[kM];
  const int T = threadIdx.x, w = T >> 5, lane = T & 31;
  const int per_mat = A.rows * A.cin * 2 * A.lout;
  const int mat = blockIdx.x / per_mat;
  int r = blockIdx.x % per_mat;
  const int o = r % (2 * A.lout);
  const int rho = r / (2 * A.lout);
  const int co = o / A.lout, limb = o % A.lout;
  const int row = rho / A.cin, ci = rho % A.cin;
  const int* p = A.raw + (size_t)mat * A.raw_stride +
                 ((((size_t)row * A.cin + ci) * A.lout + limb) * 2 + co) * kN;
  double2 x[8];
#pragma unroll
  for (int m = 0; m < 8; m++) {
    const int i = T + 256 * m;
    const int u = (i * A.gal_inv) & (2 * kN - 1);
    const int u2 = (u + kM * (A.gal_inv & 3)) & (2 * kN - 1);
    const int v = p[u & (kN - 1)], v2 = p[u2 & (kN - 1)];
    x[m] = make_double2((double)(u >= kN ? -v : v), (double)(u2 >= kN ? -v2 : v2));
  }
  fwd_pass1_store(x, spec, T);
  __syncthreads();
  const Tw34 tw = load_tw34(A.tw, w, lane);
  fwd_warp_passes(spec, w, lane, tw);
  __syncwarp();
  double2* out = A.out + (size_t)mat * A.out_stride + ((size_t)rho * 2 * A.lout + o) * kM;
#pragma unroll
  for (int j = 0; j < 8; j++) {
    // the 1/M of the inverse transform is folded into the prepared matrix (exact: power of two)
    const double2 v = spec[256 * w + 32 * j + lane];
    out[256 * w + 32 * j + lane] = make_double2(v.x * (1.0 / kM), v.y * (1.0 / kM));
  }
}

// ======================================================================================
// Element-wise helpers
// ======================================================================================
// int64 host limbs -> int32 device limbs, flags values outside int32
__global__ void k_i64_to_i32(const long long* in, int* out, size_t n, int* err) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    long long v = in[i];
    if (v > 0x3fffffffLL || v < -0x40000000LL) *err = 1;
    out[i] = (int)v;
  }
}
__global__ void k_i32_to_i64(const int* in, long long* out, size_t n) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) out[i] = (long long)in[i];
}

// to[item] = normalize(to[item] - sub[item] + add[item / add_div])   (3-limb ciphertexts)
// (ram.rs:574-576 write_first_step and ram.rs:617,625-626 write_mid_step)
__global__ void k_sub_add_normalize(int* to, const int* sub, const int* add, int add_div,
                                    int n_items, long ct_stride) {
  const size_t total = (size_t)n_items * 2 * kN;
  size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  for (; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int item = (int)(idx / (2 * kN));
    const int r = (int)(idx % (2 * kN));  // col*N + i
    int* t = to + (size_t)item * ct_stride;
    const int* s = sub + (size_t)item * ct_stride;
    const int* a = add + (size_t)(add_div > 0 ? item / add_div : item) * ct_stride;
    long long c = 0;
#pragma unroll
    for (int l = 2; l >= 0; l--) {
      const int off = l * 2 * kN + r;
      long long v = (long long)t[off] - s[off] + a[off] + c;
      long long d = sext17(v);
      c = (v - d) >> kK;
      t[off] = (int)d;
    }
  }
}
// dst[item] = src[map[item % mod]]  (whole ciphertexts; packer feed order when no one-sided
// level precedes the tree)
__global__ void k_gather(int* dst, const int* src, const int* map, int mod, int n_items, long ct_stride) {
  const size_t total = (size_t)n_items * ct_stride;
  size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  for (; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int item = (int)(idx / ct_stride);
    const long off = (long)(idx % ct_stride);
    dst[idx] = src[(size_t)map[item % mod] * ct_stride + off];
  }
}
// dst[item] = src[item] * X^k  (glwe_rotate, ram.rs:629), k in [0, 2N)
__global__ void k_rotate(int* dst, const int* src, int k, int n_items, long ct_stride) {
  const size_t total = (size_t)n_items * ct_stride;
  size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  for (; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx & (kN - 1));
    bool neg;
    const int j = rot_index(i, k, neg);
    const int v = src[idx];
    dst[idx - i + j] = neg ? -v : v;
  }
}
// dst[item] = src[item]  (glwe_copy, ram.rs:526,535)
__global__ void k_copy(int* dst, const int* src, size_t n) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  for (; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}
// dst[item] = src[tab[item].x] * X^tab[item].y, tab[item].y in [0, 2N), or zeros where tab[item].x < 0 (the per-item
// glwe_rotate of the plaintext-address calls: polynomial h seen from coefficient j, and the spread of a shard's results
// into a zero-filled arena).  Limbs move as values: the wrapped ones are negated, so -2^16 becomes +2^16.
__global__ void k_gather_rotate(int* dst, const int* src, const int2* tab, int n_items, long ct_stride) {
  const size_t total = (size_t)n_items * ct_stride;
  size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  for (; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int item = (int)(idx / ct_stride);
    const long off = (long)(idx % ct_stride);
    const int2 t = tab[item];
    if (t.x < 0) { dst[idx] = 0; continue; }
    const int i = (int)(off & (kN - 1));
    bool neg;
    const int j = rot_index(i, 2 * kN - t.y, neg);  // (a X^k)[i] = +/- a[(i - k) mod 2N]
    const int v = src[(size_t)t.x * ct_stride + off - i + j];
    dst[idx] = neg ? -v : v;
  }
}
// data[dst0 + s dst_stride] = normalize(data[...] - T[s] X^k + w[s] X^k) for s < n_items, k in [0, 2N)   (3-limb
// ciphertexts; write_plain: write_first_step of src/ram.rs:574-576 on one polynomial seen from coefficient j).  The
// sum is exact in integers and normalised once, as k_sub_add_normalize does.
__global__ void k_plain_update(int* data, const int* T, const int* w, int k, int dst0, int dst_stride, int n_items,
                               long ct_stride) {
  const size_t total = (size_t)n_items * 2 * kN;
  size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  for (; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int item = (int)(idx / (2 * kN));
    const int r = (int)(idx % (2 * kN));  // col*N + i
    const int i = r & (kN - 1);
    bool neg;
    const int e = rot_index(i, 2 * kN - k, neg);
    int* t = data + (size_t)(dst0 + item * dst_stride) * ct_stride;
    const int* tt = T + (size_t)item * ct_stride;
    const int* ww = w + (size_t)item * ct_stride;
    long long c = 0;
#pragma unroll
    for (int l = 2; l >= 0; l--) {
      const int off = l * 2 * kN + r, src = off - i + e;
      long long x = (long long)ww[src] - tt[src];
      if (neg) x = -x;
      const long long v = (long long)t[off] + x + c;
      const long long d = sext17(v);
      c = (v - d) >> kK;
      t[off] = (int)d;
    }
  }
}

}  // namespace fheram
