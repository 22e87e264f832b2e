// words.cuh -- the integer side of a key switch / external product on 51-bit WORDS (every kernel that keeps a
// ciphertext on chip between the steps of a chain).
//
// A normalised 3-limb coefficient (balanced base-2^17 digits a0,a1,a2 in [-2^16, 2^16)) is kept
// on chip as the biased word
//     U = sum_l (a_l + 2^16) << 17 (2 - l)          (51 bits; the digits are plain bit fields)
// i.e. U = X + bias with X = a0 2^34 + a1 2^17 + a2 and bias = 2^16 + 2^33 + 2^50.  Because the
// balanced digits of a value are unique and the top carry of vec_znx_big_normalize is dropped,
// "normalise" is simply "reduce mod 2^51", and everything Poulpy does limb by limb between two
// transforms collapses to a few 64-bit additions per coefficient:
//   * glwe_rsh(1)          X -> ceil(X / 2)                 (kernels.cuh: rsh1_3 computes its digits)
//   * vec_znx_big_normalize of the 4-limb product r_0..r_3 plus small operands
//                          V = sum_{l<3} r_l << 17 (2 - l)  +  floor((r_3 + 2^16) / 2^17)  +  smalls
//   * the inverse transform's rounding: v + 1.5 2^52 puts round(v) mod 2^51 in the low mantissa
//     bits (one DFMA, no F2I), and digits enter the forward transform as (2^52 + field) - (2^52 +
//     2^16) (one DADD, no I2F).
// Reference semantics: GLWE trace / GLWEPacker::combine as issued from src/ram.rs:435-457,540,572,
// 616-629 (Poulpy 0.3.2 glwe_trace, glwe_packer; oracle/fheram_oracle.c glwe_trace, pack_combine).
#pragma once
#include "kernels.cuh"

namespace fheram {

constexpr unsigned long long kBias51 = (1ull << 16) | (1ull << 33) | (1ull << 50);
constexpr unsigned long long kMask51 = (1ull << 51) - 1;
constexpr double kMagic52 = 6755399441055744.0;  // 1.5 * 2^52

// u64 scratch per cluster of the cluster kernels k_ks8 / k_ext9 (576 KiB): contribution slabs C[2 parities][8 outputs][N]
// (the words of step s are a base plus the four limb contributions of their column), then body base terms B[2][N]
constexpr size_t kKs8ScratchWords = (size_t)2 * 8 * kN + 2 * kN;

// value of three (not necessarily canonical) limbs
__device__ __forceinline__ long long limbs_value(int a0, int a1, int a2) {
  return ((long long)a0 << 34) + ((long long)a1 << 17) + (long long)a2;
}
// biased word of ceil(X / 2) for an arbitrary value X (wraps mod 2^51 like the dropped top carry)
__device__ __forceinline__ unsigned long long rsh1_word(long long X) {
  return ((unsigned long long)((X + 1) >> 1) + kBias51) & kMask51;
}
// the same for a canonical word (value U - bias in the digit range: cannot wrap)
__device__ __forceinline__ unsigned long long rsh1_canon(unsigned long long U) {
  return ((U + 1) >> 1) + (kBias51 >> 1);
}
__device__ __forceinline__ int word_digit(unsigned long long U, int l) {
  return (int)((uint32_t)(U >> (17 * (2 - l))) & 0x1ffffu) - 65536;
}
// +/-(field - 2^16) as a double; negbit = 0 or 0x80000000
__device__ __forceinline__ double field_f64(uint32_t f, uint32_t negbit) {
  const double x = __hiloint2double((int)(0x43300000u | negbit), (int)f);       // +/-(2^52 + f)
  const double c = __hiloint2double((int)(0xC3300000u ^ negbit), 65536);        // -/+(2^52 + 2^16)
  return x + c;
}
// integer bits of a double produced by "+ kMagic52": congruent to round(v) mod 2^51
__device__ __forceinline__ unsigned long long magic_bits(double t) {
  return ((unsigned long long)(uint32_t)__double2hiint(t) << 32) | (uint32_t)__double2loint(t);
}

// int32 -> double as (2^52 + 2^31 + v) - (2^52 + 2^31)
__device__ __forceinline__ double int_f64(int v) {
  return __hiloint2double(0x43300000, (int)((uint32_t)v ^ 0x80000000u)) - 4503601774854144.0;
}

// ---- operand words before step 0 ----------------------------------------------------------
// trace chains: x = rsh1(src X^rk) at position i of column col
__device__ __forceinline__ unsigned long long trace_word(const int* src, int col, int i, int rk) {
  bool neg;
  const int j = rot_index(i, 2 * kN - rk, neg);
  long long X = limbs_value(src[(0 * 2 + col) * kN + j], src[(1 * 2 + col) * kN + j], src[(2 * 2 + col) * kN + j]);
  if (neg) X = -X;
  return rsh1_word(X);
}
// pre-rotation X^rk of trace item `item` (rk0 plus the per-item rotation of VmpArgs::rot_mod), mod 2N
__device__ __forceinline__ int trace_rot(const VmpArgs& A, int item, int rk0) {
  int rk = rk0;
  if (A.rot_mod > 0) rk += A.rot_mul * (item % A.rot_mod);
  return rk & (2 * kN - 1);
}

// ---- forward transform input ----------------------------------------------------------------
// digit rho of the word w as +/-(digit) (negbit = 0 or 0x80000000): bits [17 (2 - rho), +17) = (funnel(lo, hi, s1) >> s2)
__device__ __forceinline__ double digit_f64(unsigned long long w, int rho, uint32_t negbit) {
  const int s1 = rho == 0 ? 31 : (rho == 1 ? 17 : 0);
  const int s2 = rho == 0 ? 3 : 0;
  return field_f64((__funnelshift_r((uint32_t)w, (uint32_t)(w >> 32), s1) >> s2) & 0x1ffffu, negbit);
}
// phi_g gather of digit rho at the source pair (ea, eb) of a folded position: words[e mod N], negated for e >= N
__device__ __forceinline__ double2 gather_digits(const unsigned long long* words, int ea, int eb, int rho) {
  const unsigned long long wa = words[ea & (kN - 1)];
  const unsigned long long wb = words[eb & (kN - 1)];
  const uint32_t na = ea >= kN ? 0x80000000u : 0u, nb = eb >= kN ? 0x80000000u : 0u;
  return make_double2(digit_f64(wa, rho, na), digit_f64(wb, rho, nb));
}

// ---- word update after the inverse transform -------------------------------------------------
// base term of the body column at a position: sigma (x_body[e] - bias) with sign ng (phi_g and the trace sign), + add
// (TRACE: x_body[i]; COMBINE2: 0)
__device__ __forceinline__ unsigned long long body_base(unsigned long long xe, bool ng, unsigned long long add) {
  const unsigned long long b = xe - kBias51;
  return (ng ? 0ull - b : b) + add;
}
// contribution of output limb l to its word: round(s v) at bits 17 (2 - l) for l < 3, the carry
// floor((s v + 2^16) / 2^17) for l = 3.  The combine (trace = false) runs the carry chain in the pre-automorphism sign
// frame of the position, for which floor((-r + 2^16) / 2^17) = -floor((r + 2^16 - 1) / 2^17): f = 1 where phi_g
// negates the position, and s = 1
__device__ __forceinline__ unsigned long long limb_word(double v, int l, double s, bool trace, uint32_t f) {
  unsigned long long add;
  if (l == 3) {
    const double t = trace ? fma(v, s, kMagic52 + 65536.0) : v + __hiloint2double(0x43380000, (int)(65536u - f));
    add = (unsigned long long)(long long)(int)__funnelshift_r((uint32_t)__double2loint(t), (uint32_t)__double2hiint(t), 17);
  } else {
    const double t = fma(v, s, kMagic52);
    add = l == 2 ? magic_bits(t) : (l == 1 ? magic_bits(t) << 17 : (unsigned long long)((uint32_t)__double2loint(t) << 2) << 32);
  }
  return add;
}

// ---- output ----------------------------------------------------------------------------------
// the three digits of the canonical word U to position i of column col of ciphertext ct ([limb][col][N])
__device__ __forceinline__ void put_digits(int* ct, int col, int i, unsigned long long U) {
  ct[(0 * 2 + col) * kN + i] = word_digit(U, 0);
  ct[(1 * 2 + col) * kN + i] = word_digit(U, 1);
  ct[(2 * 2 + col) * kN + i] = word_digit(U, 2);
}
// the same times X^t (the combine's a' X^t): position i goes to (i + t) mod 2N with its sign
__device__ __forceinline__ void put_digits_rot(int* ct, int col, int i, unsigned long long U, int t) {
  bool rneg;
  const int dd = rot_index(i, t, rneg);
#pragma unroll
  for (int ll = 0; ll < 3; ll++) {
    const int dg = word_digit(U, ll);
    ct[(ll * 2 + col) * kN + dd] = rneg ? -dg : dg;
  }
}

}  // namespace fheram
