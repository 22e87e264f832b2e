// Bulk GLWE secret-key encryption on the device (SURVEY.md 8(f).1): Ram::encrypt_sk
// (src/ram.rs:129-167,334-380) and Address::encrypt_sk (src/address.rs:86-109, one GGSW row =
// two GLWE, src/coordinate.rs:145-179).  Same limbs as client.cpp's glwe_encrypt on the same
// Sources: the mask is the Source's ChaCha20 stream regenerated here from (key, word position),
// the noise is drawn on the host (libm in the sampler) and arrives as one int8 per coefficient.
#pragma once
#include "kernels.cuh"

namespace fheram {

struct EncArgs {
  int* out;                   // GLWE j at out + j * ct_stride, [limb][col][N] int32 (col 0 = body)
  long ct_stride;
  int n_glwe, size;           // limbs per GLWE
  int nl, sh;                 // noise: limb nl += e << sh   (k_noise = (nl + 1) K - sh)
  const double2* sk_spec;     // [M] prepared secret (1/M folded in)
  const signed char* noise;   // [n_glwe][N], or (noise_by_seq) indexed by stream * glwe_per_stream + seq[j]
  int noise_by_seq;
  const signed char* pt;      // dense plaintext, one signed byte per coefficient, or null
  int pt_l, pt_sh;            //   limb pt_l += v << pt_sh   (encode at k_pt, src/ram.rs:364-368)
  const int* mono;            // per GLWE monomial +/- X^pos: pos | neg << 12 | limb << 16 | col << 24, or null
  const short* poly;          // [n_poly][N] small plaintext polynomials (key-switching keys: s, s * s), or null
  const int* poly_sel;        // per GLWE: polynomial index | limb << 16 (added to the body as is: GGLWE row `limb`)
  const int* sk_sel;          // per GLWE: which prepared secret (sk_spec + sk_sel[j] * 2 M) the mask is multiplied by; null: 0
  const uint32_t* keys;       // [n_streams][8] ChaCha20 keys
  const unsigned long long* word0;  // [n_streams] stream position (32-bit words) of the first mask draw
  int glwe_per_stream;        // GLWE j draws from stream j / glwe_per_stream ...
  const int* seq;             // ... as that stream's seq[j]-th GLWE (null: j % glwe_per_stream)
  Twiddles tw;
};

__device__ __forceinline__ uint32_t rotl32(uint32_t v, int n) { return __funnelshift_l(v, v, n); }
#define FHERAM_QR(a, b, c, d)                   \
  a += b; d ^= a; d = rotl32(d, 16);            \
  c += d; b ^= c; b = rotl32(b, 12);            \
  a += b; d ^= a; d = rotl32(d, 8);             \
  c += d; b ^= c; b = rotl32(b, 7);
// one ChaCha20 block (client.cpp fheram_source::refill): 64-bit block counter in words 12, 13
__device__ __forceinline__ void chacha20_block(const uint32_t* key, unsigned long long counter, uint32_t (&o)[16]) {
  uint32_t s[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u};
#pragma unroll
  for (int i = 0; i < 8; i++) s[4 + i] = key[i];
  s[12] = (uint32_t)counter; s[13] = (uint32_t)(counter >> 32); s[14] = 0; s[15] = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) o[i] = s[i];
#pragma unroll 2
  for (int r = 0; r < 10; r++) {
    FHERAM_QR(o[0], o[4], o[8], o[12]) FHERAM_QR(o[1], o[5], o[9], o[13])
    FHERAM_QR(o[2], o[6], o[10], o[14]) FHERAM_QR(o[3], o[7], o[11], o[15])
    FHERAM_QR(o[0], o[5], o[10], o[15]) FHERAM_QR(o[1], o[6], o[11], o[12])
    FHERAM_QR(o[2], o[7], o[8], o[13]) FHERAM_QR(o[3], o[4], o[9], o[14])
  }
#pragma unroll
  for (int i = 0; i < 16; i++) o[i] += s[i];
}
#undef FHERAM_QR

// Seeded ciphertexts (fheram.h fheram_seed): the mask of every GLWE regenerated from its Source's ChaCha20 stream, the
// body copied from int64 limbs or unpacked from 17-bit fields (fheram_pack17) in the same pass.
struct Seed {                 // layout of fheram_seed
  uint32_t key[8];
  unsigned long long word0;   // stream position (32-bit words) of the first mask draw
};
struct ExpandArgs {
  int* out;                   // GLWE j at out + j * ct_stride, [limb][col][N] int32 (col 0 = body)
  long ct_stride;
  int n_glwe, size;           // limbs per GLWE
  const long long* body64;    // bodies [n_glwe][size][N] as int64 limbs, or
  const uint32_t* body17;     //   as packed 17-bit fields (limb i = bits [17 i, 17 i + 17))
  int* err;                   // set when an int64 body limb lies outside +-2^30 (k_i64_to_i32's rule)
  const Seed* seeds;          // [n_streams]
  int glwe_per_stream;        // GLWE j draws from stream j / glwe_per_stream ...
  const int* seq;             // ... as that stream's seq[j]-th GLWE (null: j % glwe_per_stream)
};
// One CTA per (GLWE, limb), grid-stride.  Mask coefficient i of limb l of the stream's GLWE jl is the low 17 bits,
// sign-extended, of stream word word0 + 2 ((jl size + l) N + i): each thread produces whole ChaCha20 blocks, the
// coefficients whose low words fall in them go through shared memory so that the stores to the mask column coalesce.
__global__ void __launch_bounds__(kThreads) k_glwe_expand(const ExpandArgs A) {
  __shared__ __align__(16) int a_s[kN];
  const int T = threadIdx.x;
  for (long item = blockIdx.x; item < (long)A.n_glwe * A.size; item += gridDim.x) {
    const int j = (int)(item / A.size), l = (int)(item % A.size);
    const int stream = j / A.glwe_per_stream, jl = A.seq ? A.seq[j] : j % A.glwe_per_stream;
    const Seed& sd = A.seeds[stream];
    uint32_t key_s[8];
#pragma unroll
    for (int i = 0; i < 8; i++) key_s[i] = __ldg(sd.key + i);
    int* ob = A.out + (size_t)j * A.ct_stride + (size_t)l * 2 * kN;
    int* oa = ob + kN;
    const unsigned long long base = __ldg(&sd.word0) + 2ull * ((unsigned long long)jl * A.size + l) * kN;
    const unsigned long long b0 = base >> 4;
    const int r = (int)(base & 15);
    const int nblk = ((r + 2 * kN - 2) >> 4) + 1;
    for (int blk = T; blk < nblk; blk += kThreads) {
      uint32_t o[16];
      chacha20_block(key_s, b0 + blk, o);
#pragma unroll
      for (int k = 0; k < 16; k++) {
        const int off = blk * 16 + k - r;
        if (off >= 0 && off < 2 * kN && !(off & 1)) a_s[off >> 1] = sext17i((int)(o[k] & 0x1ffffu));
      }
    }
    __syncthreads();
    for (int i = T; i < kN / 4; i += kThreads) reinterpret_cast<int4*>(oa)[i] = reinterpret_cast<const int4*>(a_s)[i];
    const size_t t = (size_t)j * A.size + l;  // body limb t of the input
    if (A.body64) {
      const long long* in = A.body64 + t * kN;
      for (int i = T; i < kN; i += kThreads) {
        const long long v = in[i];
        if (v > 0x3fffffffLL || v < -0x40000000LL) *A.err = 1;
        ob[i] = (int)v;
      }
    } else {
      const uint32_t* in = A.body17 + t * (kN * 17 / 32);  // kN * 17 bits: a whole number of words
      for (int i = T; i < kN; i += kThreads) {
        const int bit = 17 * i, w = bit >> 5, sh = bit & 31;
        unsigned long long two = in[w];
        if (sh > 15) two |= (unsigned long long)in[w + 1] << 32;
        ob[i] = sext17i((int)((uint32_t)(two >> sh) & 0x1ffffu));
      }
    }
    __syncthreads();  // a_s is rewritten by the next item
  }
}

// Encryption noise on the device: sample k of a stream is client.cpp's fheram_source::gauss(3.2, 19.2) on the
// stream words 4k .. 4k+3 (two 53-bit uniforms, Box-Muller cosine branch, rounded to the nearest integer), as
// long as no earlier draw of the stream was rejected.  libm and CUDA agree on log / cos only to a few ulp, so
// every sample whose value could round differently (within `guard` of a half-integer) is reported for the host
// to recompute (kind 0), and every sample within `guard` of the rejection bound or beyond it marks its whole
// stream for host sampling (kind 1).  With guard = 1e-9 that is about one report in 10^8 samples.
struct NoiseArgs {
  signed char* out;            // [n_streams][per_stream]
  int n_streams;
  long per_stream;             // multiple of 4
  const uint32_t* keys;        // [n_streams][8]
  const unsigned long long* word0;
  double guard, bound_guard;   // widths of the two report bands (equal in production; tests widen them separately)
  unsigned* n_flags;           // reports appended to flags[] (counted even beyond max_flags)
  unsigned long long* flags;   // stream << 40 | kind << 39 | sample index
  unsigned max_flags;
};
__global__ void __launch_bounds__(256) k_noise_sample(const NoiseArgs A) {
  const long groups_per_stream = A.per_stream / 4;
  const long n_groups = groups_per_stream * A.n_streams;
  for (long gi = blockIdx.x * (long)blockDim.x + threadIdx.x; gi < n_groups; gi += (long)gridDim.x * blockDim.x) {
    const int stream = (int)(gi / groups_per_stream);
    const long k0 = 4 * (gi % groups_per_stream);
    uint32_t key[8];
#pragma unroll
    for (int i = 0; i < 8; i++) key[i] = __ldg(A.keys + stream * 8 + i);
    const unsigned long long w = A.word0[stream] + 4ull * k0;
    const int r = (int)(w & 15);
    uint32_t ww[32];
    {
      uint32_t o[16];
      chacha20_block(key, w >> 4, o);
#pragma unroll
      for (int i = 0; i < 16; i++) ww[i] = o[i];
      if (r) {
        chacha20_block(key, (w >> 4) + 1, o);
#pragma unroll
        for (int i = 0; i < 16; i++) ww[16 + i] = o[i];
      }
    }
#pragma unroll
    for (int t = 0; t < 4; t++) {
      const unsigned long long x1 = (unsigned long long)ww[r + 4 * t] | ((unsigned long long)ww[r + 4 * t + 1] << 32);
      const unsigned long long x2 = (unsigned long long)ww[r + 4 * t + 2] | ((unsigned long long)ww[r + 4 * t + 3] << 32);
      const double u1 = ((double)(x1 >> 11) + 1.0) * (1.0 / 9007199254740992.0);
      const double u2 = ((double)(x2 >> 11) + 1.0) * (1.0 / 9007199254740992.0);
      const double z = sqrt(-2.0 * log(u1)) * cos(2.0 * 3.14159265358979323846 * u2) * 3.2;
      const double rz = round(z);  // half away from zero, as llround
      int kind = -1;
      if (!(fabs(z) < 19.2 - A.bound_guard)) kind = 1;
      else if (0.5 - fabs(z - rz) < A.guard) kind = 0;
      if (kind >= 0) {
        const unsigned slot = atomicAdd(A.n_flags, 1u);
        if (slot < A.max_flags)
          A.flags[slot] = ((unsigned long long)stream << 40) | ((unsigned long long)kind << 39) | (unsigned long long)(k0 + t);
      }
      A.out[(size_t)stream * A.per_stream + k0 + t] = (signed char)(int)fmax(-127.0, fmin(127.0, rz));
    }
  }
}

// One CTA per GLWE (grid-stride).  Limbs from the least significant one up, so that the
// normalization carry of each coefficient stays in a register.
__global__ void __launch_bounds__(kThreads, 2) k_glwe_encrypt(const EncArgs A) {
  __shared__ __align__(16) double2 spec[kM];
  __shared__ int a_s[kN];
  const int T = threadIdx.x, w = T >> 5, lane = T & 31;
  const Tw34 tw = load_tw34(A.tw, w, lane);

  for (int j = blockIdx.x; j < A.n_glwe; j += gridDim.x) {
    const int stream = j / A.glwe_per_stream, jl = A.seq ? A.seq[j] : j % A.glwe_per_stream;
    uint32_t key_s[8];
#pragma unroll
    for (int i = 0; i < 8; i++) key_s[i] = __ldg(A.keys + stream * 8 + i);
    int* out = A.out + (size_t)j * A.ct_stride;
    const signed char* noise = A.noise + (size_t)(A.noise_by_seq ? stream * A.glwe_per_stream + jl : j) * kN;
    const signed char* pt = A.pt ? A.pt + (size_t)j * kN : nullptr;
    int m_pos = -1, m_val = 0, m_limb = -1, m_col = 0;
    if (A.mono) {
      const int mm = A.mono[j];
      m_pos = mm & 0xfff; m_val = (mm >> 12) & 1 ? -1 : 1; m_limb = (mm >> 16) & 0xff; m_col = (mm >> 24) & 1;
    }
    const short* poly = nullptr;
    int p_limb = -1;
    if (A.poly) { const int ps = A.poly_sel[j]; poly = A.poly + (size_t)(ps & 0xffff) * kN; p_limb = ps >> 16; }
    const double2* sk_spec = A.sk_spec + (A.sk_sel ? (size_t)A.sk_sel[j] * 2 * kM : 0);  // k_prepare writes two polynomials per secret
    int carry[16];
#pragma unroll
    for (int q = 0; q < 16; q++) carry[q] = 0;

#pragma unroll 1
    for (int l = A.size - 1; l >= 0; l--) {
      // ---- mask limb l: coefficient i = low K bits (sign-extended) of the 64-bit draw whose low word is
      //      stream word base + 2 i  (client.cpp glwe_encrypt: digit(K, xa->next())) ----
      const unsigned long long base = A.word0[stream] + 2ull * ((unsigned long long)(jl * A.size + l) * kN);
      const unsigned long long b0 = base >> 4;
      const int r = (int)(base & 15);
      const int nblk = ((r + 2 * kN - 2) >> 4) + 1;
      for (int blk = T; blk < nblk; blk += kThreads) {
        uint32_t o[16];
        chacha20_block(key_s, b0 + blk, o);
#pragma unroll
        for (int k = 0; k < 16; k++) {
          const int off = blk * 16 + k - r;
          if (off >= 0 && off < 2 * kN && !(off & 1)) a_s[off >> 1] = sext17i((int)(o[k] & 0x1ffffu));
        }
      }
      __syncthreads();
      double2 x[8];
#pragma unroll
      for (int m = 0; m < 8; m++) x[m] = make_double2((double)a_s[T + 256 * m], (double)a_s[T + 256 * m + kM]);
      {
        int* oa = out + ((size_t)l * 2 + 1) * kN;
#pragma unroll
        for (int q = 0; q < 16; q++) {
          const int i = T + 256 * q;
          int v = a_s[i];
          if (m_col == 1 && m_limb == l && i == m_pos) v += m_val;  // plaintext on the mask column: added as is
          oa[i] = v;
        }
      }
      // ---- a_l * s by the negacyclic transform (exact: |a_l * s| < 2^29) ----
      fwd_pass1_store(x, spec, T);
      __syncthreads();
      fwd_warp_passes(spec, w, lane, tw);
      __syncwarp();
#pragma unroll
      for (int jj = 0; jj < 8; jj++) {
        const double2 u = spec[256 * w + 32 * jj + lane];
        const double2 s = __ldg(sk_spec + 256 * w + 32 * jj + lane);
        x[jj] = make_double2(u.x * s.x - u.y * s.y, u.x * s.y + u.y * s.x);
      }
      __syncwarp();
      inv_transform(x, spec, T, w, lane, tw, [] {});
      // ---- body limb l = normalize(-a_l s + pt_l + e_l) with the carry of the limbs below ----
      int* ob = out + (size_t)l * 2 * kN;
#pragma unroll
      for (int q = 0; q < 16; q++) {
        const int i = T + 256 * (q & 7) + (q >> 3) * kM;
        int t = carry[q] - (int)__double2ll_rn((q < 8) ? x[q & 7].x : x[q & 7].y);
        if (l == A.nl) t += (int)noise[i] << A.sh;
        if (pt && l == A.pt_l) t += (int)pt[i] << A.pt_sh;
        if (m_col == 0 && m_limb == l && i == m_pos) t += m_val;
        if (poly && l == p_limb) t += (int)poly[i];
        const int dg = sext17i(t & 0x1ffff);
        carry[q] = (t - dg) >> kK;
        ob[i] = dg;
      }
      __syncthreads();  // a_s and spec are rewritten by the next limb
    }
  }
}

}  // namespace fheram
