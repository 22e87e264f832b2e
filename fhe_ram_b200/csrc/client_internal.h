// Internal interface between the client-side code (client.cpp) and the GPU bulk-encryption path
// (fheram_cuda.cu).  Not part of the C ABI.
#pragma once
#include <cstddef>
#include <cstdint>

#include "../../include/fheram.h"

// key and absolute position (in 32-bit words) of a Source's ChaCha20 stream
void fheram_source_tell(const fheram_source* s, uint32_t key[8], uint64_t* word_pos);
// advance the stream by n 32-bit words without producing them
void fheram_source_skip_words(fheram_source* s, uint64_t n);
// n draws of the GLWE encryption noise (sigma 3.2, bound 6 sigma), exactly as glwe_encrypt draws them
void fheram_source_noise_i8(fheram_source* s, int8_t* out, size_t n);
// the noise draw that starts `word_offset` words past the Source's position (the Source is not advanced)
int8_t fheram_source_noise_at(const fheram_source* s, uint64_t word_offset);
// the n_ggsw monomials +/- X^pos an address value is encoded as (src/address.rs:102-108,
// src/coordinate.rs:148-179); returns n_ggsw or a negative status
int fheram_address_monomials(const fheram_params* p, uint32_t value, int32_t* pos, int32_t* sign);
// range checks of every field the digit tables / size helpers index with (n_decomp <= 8, max_addr <= N^2, ...);
// 0 or FHERAM_ERR_INVALID with fheram_last_error set
int fheram_params_check(const fheram_params* p);

// ---- decryption (fheram_decrypt_ram on the CPU, k_glwe_decrypt on the device) ----
// v = (sum_j pt_j 2^(K (S-1-j))) >> vsh is the phase of a coefficient at precision k_ct (vsh = S K - k_ct) and
// ls = k_ct - k_pt the scale of the plaintext; 0 or FHERAM_ERR_INVALID when k_pt >= k_ct or S K > 62
int fheram_decode_shifts(const fheram_params* p, int* vsh, int* ls);
#ifdef __CUDACC__
#define FHERAM_HD __host__ __device__
#else
#define FHERAM_HD
#endif
// value_raw = round_half_away(v / 2^ls), as fheram_decrypt_word's llround((double)v / 2^ls) (|v| < 2^53 is exact in
// double); value = value_raw reduced into [-2^(k_pt-1), 2^(k_pt-1)); err = v - value_raw 2^ls, exact
FHERAM_HD inline void fheram_decode(int64_t v, int ls, int k_pt, int16_t* value, int64_t* err) {
  const int64_t half = (int64_t)1 << (ls - 1);
  const int64_t raw = v >= 0 ? (v + half) >> ls : -((half - v) >> ls);
  *err = v - raw * ((int64_t)1 << ls);
  *value = (int16_t)((int64_t)((uint64_t)raw << (64 - k_pt)) >> (64 - k_pt));
}
