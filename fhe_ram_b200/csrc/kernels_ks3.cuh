// kernels_ks3.cuh -- the integer side of a key switch / external product on 51-bit WORDS instead of per-limb digits
// (helpers used by every later kernel).
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
// This replaces k_ks2's digit carry chains, packed-field inserts and the separate rsh pass (about
// 60 K of its 126 K warp instructions per key switch).  Transforms, contraction, tensor-memory use
// and the two-CTAs-per-SM footprint are those of k_ks2; results are bit-identical (same integers).
// Reference semantics: GLWE trace / GLWEPacker::combine as issued from src/ram.rs:435-457,540,572,
// 616-629 (Poulpy 0.3.2 glwe_trace, glwe_packer; oracle/fheram_oracle.c glwe_trace, pack_combine).
#pragma once
#include "kernels_ks2.cuh"
#include "transform_pad.cuh"

// timing ablations for tools/ablate.sh (results are garbage when non-zero): 1 no matrix loads,
// 2 no inverse transforms, 4 no forward transforms
#ifndef FHERAM_ABL
#define FHERAM_ABL 0
#endif

namespace fheram {

constexpr unsigned long long kBias51 = (1ull << 16) | (1ull << 33) | (1ull << 50);
constexpr unsigned long long kMask51 = (1ull << 51) - 1;
constexpr double kMagic52 = 6755399441055744.0;  // 1.5 * 2^52

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

// (k_ks3, the first word-domain key-switch kernel -- register accumulators, one tile in flight -- was retired in round 2:
// k_ks4 does the same with in-place word accumulation and two tiles in flight, k_ks7 with the two-exchange transform.
// k_ext3, the round-1 external product on the padded transform, was retired after k_ext8 / k_ext9 took every launch.)

}  // namespace fheram
