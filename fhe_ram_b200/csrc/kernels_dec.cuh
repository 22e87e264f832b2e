// Bulk GLWE secret-key decryption on the device (DESIGN.md 3.7): the resident RAM (fheram_ram_decrypt_sk) and
// coefficient 0 of read results (fheram_decrypt_words_device).  The same numbers as client.cpp's fheram_decrypt_ram /
// fheram_decrypt_word: pt = normalize(body + mask * s), then fheram_decode (client_internal.h).
#pragma once
#include "client_internal.h"
#include "kernels.cuh"

namespace fheram {

struct DecArgs {
  const int* in;              // GLWE j at in + j * ct_stride, [limb][col][N] int32 (col 0 = body)
  long ct_stride;
  int n_glwe, size;           // limbs per GLWE
  const double2* sk_spec;     // [M] prepared secret (1/M folded in)
  int vsh, ls, k_pt;          // v >>= vsh, then fheram_decode(v, ls, k_pt)
  short* values;              // outputs; err may be null
  long long* err;
  // coef0 != 0: entry j = coefficient 0 of GLWE j.  Else GLWE j = s * n_poly + hp (a RAM's [word_size][n_poly]
  // layout) writes coefficient i to entry (hp * N + i) * word_size + s while its address
  // (shard + n_shards * hp) * N + i is below max_addr
  int coef0;
  int n_poly, word_size, shard, n_shards;
  unsigned long long max_addr;
  Twiddles tw;
};

// dynamic shared memory: the transform buffer and the phase accumulators (acc below; in registers they would spill)
constexpr size_t kDecSmem = kM * sizeof(double2) + kN * sizeof(unsigned long long);

// One CTA per GLWE (grid-stride), limb by limb.
__global__ void __launch_bounds__(kThreads, 2) k_glwe_decrypt(const DecArgs A) {
  extern __shared__ __align__(16) double2 dsm[];
  double2* spec = dsm;
  unsigned long long* acc = (unsigned long long*)(dsm + kM);  // thread T owns the 16 coefficients it normalizes
  const int T = threadIdx.x, w = T >> 5, lane = T & 31;

  for (int j = blockIdx.x; j < A.n_glwe; j += gridDim.x) {
    const int* ct = A.in + (size_t)j * A.ct_stride;
    // acc = sum_l (b_l + a_l s) 2^(K (size-1-l)) modulo 2^64.  Normalization with the top carry dropped depends only on
    // acc mod 2^(K size) (the balanced digits are a complete residue system), so one 64-bit word per coefficient
    // replaces the carry chain of client.cpp's normalize, which runs on acc after the last limb
#pragma unroll
    for (int q = 0; q < 16; q++) acc[T + 256 * (q & 7) + (q >> 3) * kM] = 0;

#pragma unroll 1
    for (int l = A.size - 1; l >= 0; l--) {
      // ---- a_l * s by the negacyclic transform.  Exact for every limb the device stores: |a_l| < 2^20 and s ternary
      //      give |a_l * s| <= N 2^20 = 2^32, and the FP64 transform error stays far below 1/2 there ----
      const int* a = ct + ((size_t)l * 2 + 1) * kN;
      const Tw34 tw = load_tw34(A.tw, w, lane);  // per limb (L1 hits): not live across the decode
      double2 x[8];
#pragma unroll
      for (int m = 0; m < 8; m++)
        x[m] = make_double2((double)__ldg(a + T + 256 * m), (double)__ldg(a + T + 256 * m + kM));
      fwd_pass1_store(x, spec, T);
      __syncthreads();
      fwd_warp_passes(spec, w, lane, tw);
      __syncwarp();
#pragma unroll
      for (int jj = 0; jj < 8; jj++) {
        const double2 u = spec[256 * w + 32 * jj + lane];
        const double2 s = __ldg(A.sk_spec + 256 * w + 32 * jj + lane);
        x[jj] = make_double2(u.x * s.x - u.y * s.y, u.x * s.y + u.y * s.x);
      }
      __syncwarp();
      // its last barrier follows the last read of spec, so the next limb may overwrite it
      inv_transform(x, spec, T, w, lane, tw, [] {});
      const int* b = ct + (size_t)l * 2 * kN;
      const int sh = kK * (A.size - 1 - l);
#pragma unroll
      for (int q = 0; q < 16; q++) {
        const int i = T + 256 * (q & 7) + (q >> 3) * kM;
        const long long t = (long long)__ldg(b + i) + __double2ll_rn((q < 8) ? x[q & 7].x : x[q & 7].y);
        acc[i] += (unsigned long long)t << sh;
      }
    }
    // ---- pt = the balanced base-2^K digits of acc mod 2^(K size), v = sum_j pt_j 2^(K (size-1-j)), decode ----
    const int top = 64 - kK * A.size;
#pragma unroll
    for (int q = 0; q < 16; q++) {
      const int i = T + 256 * (q & 7) + (q >> 3) * kM;
      size_t e;
      if (A.coef0) {
        if (i != 0) continue;
        e = j;
      } else {
        const int s = j / A.n_poly, hp = j % A.n_poly;
        const unsigned long long addr = (unsigned long long)(A.shard + A.n_shards * hp) * kN + i;
        if (addr >= A.max_addr) continue;
        e = ((size_t)hp * kN + i) * A.word_size + s;
      }
      long long r = (long long)(acc[i] << top) >> top, v = 0;
      for (int l = A.size - 1, sh = 0; l >= 0; l--, sh += kK) {
        const long long dg = sext17(r);
        r = (r - dg) >> kK;
        v += dg * (1ll << sh);
      }
      int16_t val;
      int64_t er;
      fheram_decode(v >> A.vsh, A.ls, A.k_pt, &val, &er);
      A.values[e] = val;
      if (A.err) A.err[e] = er;
    }
  }
}

}  // namespace fheram
