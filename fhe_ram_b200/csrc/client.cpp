// client.cpp -- client side of the drop-in API (CPU): secret / evaluation-key generation,
// RAM / address / word encryption, and RAM and word decryption.  These are the calls of
// examples/fhe-ram.rs:34-95,179-237 that run once per key / RAM / address, outside the
// homomorphic hot path (SURVEY.md 8f ranks moving them to the GPU as the next step).
//
// Conventions (Poulpy 0.3.2 is not vendored in the reference; these restate its published
// scheme and are what the device kernels assume):
//   GLWE(k): body b = -a*s + m + e (col 0), mask a uniform per limb (col 1); decrypt = b + a*s.
//   GGSW row r, column c: GLWE encryption of zero with m*2^-(r+1)K added into component c.
//   Automorphism key p: key-switching key from s to phi_{p^-1}(s) (keyswitch, then X -> X^p).
//   GGLWE->GGSW key: rows encrypt s*s*2^-(r+1)K under s.
//   Source: ChaCha20 keystream; uniform limb = sign-extended low 17 bits of next_u64; noise =
//   round(Box-Muller normal * 3.2) truncated at 6 sigma.
#include <cmath>
#include <complex>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "../../include/fheram.h"
#include "client_internal.h"

void fheram_set_error(const char* msg);  // fheram_cuda.cu

namespace {

typedef int64_t i64;
typedef uint64_t u64;
typedef std::complex<double> cd;

int cdiv(int a, int b) { return (a + b - 1) / b; }
inline i64 digit(int k, i64 x) { return (i64)((u64)x << (64 - k)) >> (64 - k); }

// ---------------- ChaCha20 source ----------------
inline uint32_t rotl(uint32_t v, int n) { return (v << n) | (v >> (32 - n)); }
inline void qr(uint32_t* x, int a, int b, int c, int d) {
  x[a] += x[b]; x[d] ^= x[a]; x[d] = rotl(x[d], 16);
  x[c] += x[d]; x[b] ^= x[c]; x[b] = rotl(x[b], 12);
  x[a] += x[b]; x[d] ^= x[a]; x[d] = rotl(x[d], 8);
  x[c] += x[d]; x[b] ^= x[c]; x[b] = rotl(x[b], 7);
}
}  // namespace

struct fheram_source {
  uint32_t key[8];
  u64 counter = 0;
  uint32_t block[16];
  int pos = 16;
  void refill() {
    uint32_t st[16] = {0x61707865, 0x3320646e, 0x79622d32, 0x6b206574};
    for (int i = 0; i < 8; i++) st[4 + i] = key[i];
    st[12] = (uint32_t)counter; st[13] = (uint32_t)(counter >> 32); st[14] = 0; st[15] = 0;
    uint32_t x[16];
    memcpy(x, st, sizeof(x));
    for (int r = 0; r < 10; r++) {
      qr(x, 0, 4, 8, 12); qr(x, 1, 5, 9, 13); qr(x, 2, 6, 10, 14); qr(x, 3, 7, 11, 15);
      qr(x, 0, 5, 10, 15); qr(x, 1, 6, 11, 12); qr(x, 2, 7, 8, 13); qr(x, 3, 4, 9, 14);
    }
    for (int i = 0; i < 16; i++) block[i] = x[i] + st[i];
    counter++;
    pos = 0;
  }
  uint32_t u32() { if (pos >= 16) refill(); return block[pos++]; }
  u64 next() { u64 lo = u32(); u64 hi = u32(); return lo | (hi << 32); }
  double unit() { return ((double)(next() >> 11) + 1.0) * (1.0 / 9007199254740992.0); }
  i64 gauss(double sigma, double bound) {
    for (;;) {
      double u1 = unit(), u2 = unit();
      double z = std::sqrt(-2.0 * std::log(u1)) * std::cos(2.0 * M_PI * u2) * sigma;
      if (std::fabs(z) <= bound) return (i64)std::llround(z);
    }
  }
};

extern "C" fheram_source* fheram_source_new(const uint8_t seed[32]) {
  fheram_source* s = new fheram_source();
  for (int i = 0; i < 8; i++)
    s->key[i] = (uint32_t)seed[4 * i] | ((uint32_t)seed[4 * i + 1] << 8) |
                ((uint32_t)seed[4 * i + 2] << 16) | ((uint32_t)seed[4 * i + 3] << 24);
  return s;
}
extern "C" void fheram_source_free(fheram_source* s) { delete s; }
extern "C" uint32_t fheram_source_next_u32(fheram_source* s) { return s->u32(); }
extern "C" void fheram_source_fill_bytes(fheram_source* s, uint8_t* out, size_t n) {
  size_t i = 0;
  while (i < n) {
    uint32_t w = s->u32();
    for (int b = 0; b < 4 && i < n; b++, i++) out[i] = (uint8_t)(w >> (8 * b));
  }
}

// ---- stream position helpers of the GPU bulk-encryption path (client_internal.h) ----
void fheram_source_tell(const fheram_source* s, uint32_t key[8], uint64_t* word_pos) {
  for (int i = 0; i < 8; i++) key[i] = s->key[i];
  *word_pos = s->counter * 16 + (u64)s->pos - 16;  // counter blocks produced, 16 - pos words of the last unread
}
void fheram_source_skip_words(fheram_source* s, uint64_t n) {
  const u64 wp = s->counter * 16 + (u64)s->pos - 16 + n;
  s->counter = wp / 16;
  s->pos = 16;
  if (wp % 16) { s->refill(); s->pos = (int)(wp % 16); }
}
extern "C" uint64_t fheram_source_position(const fheram_source* s) {
  return s ? s->counter * 16 + (u64)s->pos - 16 : 0;
}
extern "C" void fheram_source_skip(fheram_source* s, uint64_t n_words) {
  if (s) fheram_source_skip_words(s, n_words);
}
int8_t fheram_source_noise_at(const fheram_source* s, uint64_t word_offset) {
  fheram_source t = *s;
  fheram_source_skip_words(&t, word_offset);
  return (int8_t)t.gauss(3.2, 19.2);
}
void fheram_source_noise_i8(fheram_source* s, int8_t* out, size_t n) {
  for (size_t i = 0; i < n; i++) out[i] = (int8_t)s->gauss(3.2, 19.2);
}

namespace {

// ---------------- negacyclic ring arithmetic by a twisted complex FFT ----------------
// Operands here are (17-bit limb) x (small secret): |result| < 2^29, far inside f64 exactness.
class Ring {
 public:
  explicit Ring(int log_n) : n_(1 << log_n), m_(n_ / 2) {
    twist_.resize(m_); roots_.resize(m_);
    const long double PI = 3.14159265358979323846264338327950288L;
    for (int j = 0; j < m_; j++) {
      twist_[j] = cd((double)cosl(PI * j / n_), (double)sinl(PI * j / n_));
      roots_[j] = cd((double)cosl(2 * PI * j / m_), (double)sinl(2 * PI * j / m_));
    }
    rev_.resize(m_);
    int lg = 0;
    while ((1 << lg) < m_) lg++;
    for (int i = 0; i < m_; i++) {
      int r = 0;
      for (int b = 0; b < lg; b++) r |= ((i >> b) & 1) << (lg - 1 - b);
      rev_[i] = r;
    }
  }
  int n() const { return n_; }
  void forward(const i64* a, std::vector<cd>& out) const {
    out.resize(m_);
    for (int j = 0; j < m_; j++) out[rev_[j]] = cd((double)a[j], (double)a[j + m_]) * twist_[j];
    fft(out, false);
  }
  // out = round(inverse(spec))
  void inverse(std::vector<cd>& spec, i64* out) const {
    std::vector<cd> t(m_);
    for (int j = 0; j < m_; j++) t[rev_[j]] = spec[j];
    fft(t, true);
    for (int j = 0; j < m_; j++) {
      cd v = t[j] * std::conj(twist_[j]) / (double)m_;
      out[j] = (i64)std::llround(v.real());
      out[j + m_] = (i64)std::llround(v.imag());
    }
  }
  void mul(const std::vector<cd>& a, const std::vector<cd>& b, std::vector<cd>& out) const {
    out.resize(m_);
    for (int j = 0; j < m_; j++) out[j] = a[j] * b[j];
  }

 private:
  void fft(std::vector<cd>& x, bool inv) const {  // input in bit-reversed order
    for (int len = 2; len <= m_; len <<= 1) {
      const int half = len / 2, step = m_ / len;
      for (int i = 0; i < m_; i += len)
        for (int j = 0; j < half; j++) {
          cd w = roots_[j * step];
          if (inv) w = std::conj(w);
          cd u = x[i + j], v = x[i + j + half] * w;
          x[i + j] = u + v;
          x[i + j + half] = u - v;
        }
    }
  }
  int n_, m_;
  std::vector<cd> twist_, roots_;
  std::vector<int> rev_;
};

struct Dims {
  int n, log_n, K, size_ct, dnum_ct, size_addr, size_evk_trace, dnum_ggsw, size_evk_inv;
  int n_coord, coord_len[8], coord_digits[8][8], n_ggsw, n_glwe;
};
Dims dims(const fheram_params* p) {
  Dims d;
  memset(&d, 0, sizeof(d));
  d.log_n = p->log_n; d.n = 1 << p->log_n; d.K = p->base2k;
  d.size_ct = cdiv(p->k_ct, d.K); d.dnum_ct = d.size_ct;
  d.size_addr = cdiv(p->k_addr, d.K); d.size_evk_trace = cdiv(p->k_evk_trace, d.K);
  d.dnum_ggsw = cdiv(p->k_addr, d.K); d.size_evk_inv = cdiv(p->k_evk_ggsw_inv, d.K);
  int32_t lens[8], digits[64];
  d.n_coord = fheram_base2d(p, lens, digits);
  for (int i = 0; i < d.n_coord; i++) {
    d.coord_len[i] = lens[i];
    for (int j = 0; j < lens[i]; j++) d.coord_digits[i][j] = digits[i * 8 + j];
    d.n_ggsw += lens[i];
  }
  d.n_glwe = (int)((p->max_addr + (u64)d.n - 1) / (u64)d.n);
  return d;
}

// balanced base-2^K digits of sum_l big[l] 2^(K(size-1-l)), top carry dropped
void normalize(int n, int K, int size, const std::vector<i64>& big, i64* out, int out_cols, int out_col) {
  for (int i = 0; i < n; i++) {
    i64 c = 0;
    for (int l = size - 1; l >= 0; l--) {
      i64 t = big[(size_t)l * n + i] + c;
      i64 d = digit(K, t);
      c = (t - d) >> K;
      out[((size_t)l * out_cols + out_col) * n + i] = d;
    }
  }
}

// one GLWE(size limbs) encryption; pt (pt_size limbs, 1 column) goes to component pt_col
void glwe_encrypt(const Ring& R, int K, i64* ct, int size, int k_noise, const i64* pt, int pt_size,
                  int pt_col, const std::vector<cd>& sk_spec, fheram_source* xa, fheram_source* xe) {
  const int n = R.n();
  std::vector<i64> big((size_t)size * n);
  std::vector<cd> spec, prod;
  std::vector<i64> tmp(n);
  for (int l = 0; l < size; l++) {
    i64* a = ct + ((size_t)l * 2 + 1) * n;
    for (int i = 0; i < n; i++) a[i] = digit(K, (i64)xa->next());
    R.forward(a, spec);
    R.mul(spec, sk_spec, prod);
    R.inverse(prod, tmp.data());
    for (int i = 0; i < n; i++) big[(size_t)l * n + i] = -tmp[i];
  }
  if (pt && pt_col == 0)
    for (int l = 0; l < pt_size && l < size; l++)
      for (int i = 0; i < n; i++) big[(size_t)l * n + i] += pt[(size_t)l * n + i];
  const int nl = cdiv(k_noise, K) - 1, sh = (nl + 1) * K - k_noise;
  for (int i = 0; i < n; i++) big[(size_t)nl * n + i] += xe->gauss(3.2, 19.2) << sh;
  normalize(n, K, size, big, ct, 2, 0);
  if (pt && pt_col == 1)
    for (int l = 0; l < pt_size && l < size; l++) {
      i64* a = ct + ((size_t)l * 2 + 1) * n;
      for (int i = 0; i < n; i++) a[i] += pt[(size_t)l * n + i];
    }
}

void automorphism(int n, i64 p, const i64* a, i64* out) {
  const i64 two_n = 2 * (i64)n;
  const i64 pp = ((p % two_n) + two_n) % two_n;
  for (int i = 0; i < n; i++) {
    i64 e = (i64)(((unsigned __int128)(u64)i * (u64)pp) % (u64)two_n);
    if (e >= n) out[e - n] = -a[i]; else out[e] = a[i];
  }
}
i64 inv_mod_2n(i64 p, i64 two_n) {
  i64 b = ((p % two_n) + two_n) % two_n, r = 1;
  u64 e = (u64)(two_n / 2 - 1);
  while (e) {
    if (e & 1) r = (i64)((unsigned __int128)r * b % two_n);
    b = (i64)((unsigned __int128)b * b % two_n);
    e >>= 1;
  }
  return r;
}

// rows of GLWE(size) each encrypting msg * 2^-(r+1)K under sk_out
void gglwe_encrypt(const Ring& R, int K, i64* key, int rows, int size, int k_noise, const i64* msg,
                   const std::vector<cd>& sk_out_spec, fheram_source* xa, fheram_source* xe) {
  const int n = R.n();
  std::vector<i64> pt((size_t)size * n);
  for (int r = 0; r < rows; r++) {
    std::fill(pt.begin(), pt.end(), 0);
    memcpy(pt.data() + (size_t)r * n, msg, sizeof(i64) * n);
    glwe_encrypt(R, K, key + (size_t)r * 2 * size * n, size, k_noise, pt.data(), r + 1, 0, sk_out_spec, xa, xe);
  }
}
void atk_encrypt(const Ring& R, int K, i64* key, int rows, int size, int k_noise, i64 p, const i64* sk,
                 fheram_source* xa, fheram_source* xe) {
  const int n = R.n();
  std::vector<i64> sk_out(n);
  automorphism(n, inv_mod_2n(p, 2 * (i64)n), sk, sk_out.data());
  std::vector<cd> so;
  R.forward(sk_out.data(), so);
  gglwe_encrypt(R, K, key, rows, size, k_noise, sk, so, xa, xe);
}

// seeded: the rows with ci = 1 carry scalar * s in the body instead of scalar in the mask (same phase, raw mask)
void ggsw_encrypt(const Ring& R, const Dims& d, int k_addr, i64* ggsw, const i64* scalar,
                  const std::vector<cd>& sk_spec, fheram_source* xa, fheram_source* xe, bool seeded = false) {
  const int n = d.n, S = d.size_addr;
  const size_t glwe = (size_t)2 * S * n;
  std::vector<i64> pt((size_t)S * n), pt_s, ms;
  if (seeded) {  // scalar * s: a signed rotation of the secret, exact through the transform
    std::vector<cd> spec, prod;
    R.forward(scalar, spec);
    R.mul(spec, sk_spec, prod);
    ms.resize(n);
    R.inverse(prod, ms.data());
    pt_s.resize((size_t)S * n);
  }
  for (int r = 0; r < d.dnum_ct; r++) {
    std::fill(pt.begin(), pt.end(), 0);
    memcpy(pt.data() + (size_t)r * n, scalar, sizeof(i64) * n);
    if (seeded) {
      std::fill(pt_s.begin(), pt_s.end(), 0);
      memcpy(pt_s.data() + (size_t)r * n, ms.data(), sizeof(i64) * n);
    }
    for (int ci = 0; ci < 2; ci++) {
      const bool body = seeded && ci == 1;
      glwe_encrypt(R, d.K, ggsw + ((size_t)r * 2 + ci) * glwe, S, k_addr, body ? pt_s.data() : pt.data(), r + 1,
                   body ? 0 : ci, sk_spec, xa, xe);
    }
  }
}

// body columns of n_glwe GLWEs of `size` limbs: [n_glwe][size][2][N] -> [n_glwe][size][N]
void take_bodies(int n, int size, size_t n_glwe, const i64* ct, i64* bodies) {
  for (size_t t = 0; t < n_glwe * size; t++) memcpy(bodies + t * n, ct + t * 2 * n, sizeof(i64) * n);
}

// value * 2^-k placed in `size` limbs (torus wrap), coefficient idx
void encode_coeff(int n, int K, i64* pt, int size, int idx, i64 v, int k) {
  const int l = cdiv(k, K) - 1, sh = (l + 1) * K - k;
  i64 t = v << sh;
  for (int j = l; j >= 0; j--) {
    i64 dg = digit(K, t);
    if (j < size) pt[(size_t)j * n + idx] = dg;
    t = (t - dg) >> K;
  }
}

int check(const fheram_params* p) {
  if (!p || p->log_n < 4 || p->log_n > 14 || p->base2k < 2 || p->base2k > 30) {
    fheram_set_error("bad parameters");
    return FHERAM_ERR_INVALID;
  }
  return fheram_params_check(p);  // digit tables, max_addr, word_size: shared with fheram_ctx_create
}

}  // namespace

extern "C" int fheram_secret_gen(const fheram_params* p, fheram_source* xs, int64_t* sk) {
  if (check(p) || !xs || !sk) return FHERAM_ERR_INVALID;
  const int n = 1 << p->log_n;
  for (int i = 0; i < n; i++) {  // fill_ternary_prob(0.5): examples/fhe-ram.rs:50
    u64 r = xs->next();
    sk[i] = (r & 1) ? ((r & 2) ? 1 : -1) : 0;
  }
  return 0;
}

extern "C" int fheram_keygen(const fheram_params* p, const int64_t* sk, fheram_source* xa,
                             fheram_source* xe, int64_t* atk_glwe, int64_t* tsk, int64_t* atk_inv) {
  if (check(p) || !sk || !xa || !xe || !atk_glwe || !tsk || !atk_inv) return FHERAM_ERR_INVALID;
  const Dims d = dims(p);
  Ring R(d.log_n);
  const size_t atk_len = fheram_atk_len(p);
  for (int i = 0; i < d.log_n; i++)  // src/keys.rs:158-165
    atk_encrypt(R, d.K, atk_glwe + (size_t)i * atk_len, d.dnum_ct, d.size_evk_trace, p->k_evk_trace,
                fheram_trace_galois_element(p, i), sk, xa, xe);
  {  // src/keys.rs:167-169
    std::vector<cd> s_spec, s2_spec;
    R.forward(sk, s_spec);
    R.mul(s_spec, s_spec, s2_spec);
    std::vector<i64> s2(d.n);
    R.inverse(s2_spec, s2.data());
    gglwe_encrypt(R, d.K, tsk, d.dnum_ggsw, d.size_evk_inv, p->k_evk_ggsw_inv, s2.data(), s_spec, xa, xe);
  }
  // src/keys.rs:171-173
  atk_encrypt(R, d.K, atk_inv, d.dnum_ggsw, d.size_evk_inv, p->k_evk_ggsw_inv, -1, sk, xa, xe);
  return 0;
}

namespace {
// Ram::encrypt_sk: every GLWE into cts, or (cts null) its body column into bodies
int encrypt_ram(const fheram_params* p, const uint8_t* data, const int64_t* sk, fheram_source* xa,
                fheram_source* xe, int64_t* cts, int64_t* bodies) {
  const Dims d = dims(p);
  Ring R(d.log_n);
  std::vector<cd> s_spec;
  R.forward(sk, s_spec);
  const int ws = p->word_size, pt_size = cdiv(p->k_pt, d.K);
  const size_t glwe = fheram_glwe_len(p);
  std::vector<i64> pt((size_t)pt_size * d.n), one(cts ? 0 : glwe);
  for (int i = 0; i < ws; i++)           // src/ram.rs:161-166
    for (int h = 0; h < d.n_glwe; h++) { // src/ram.rs:358-379
      std::fill(pt.begin(), pt.end(), 0);
      for (int j = 0; j < d.n; j++) {
        const u64 addr = (u64)h * d.n + j;
        const i64 v = addr < p->max_addr ? (i64)(int8_t)data[addr * ws + i] : 0;  // :364
        encode_coeff(d.n, d.K, pt.data(), pt_size, j, v, p->k_pt);                // :368
      }
      const size_t g = (size_t)i * d.n_glwe + h;
      i64* ct = cts ? cts + g * glwe : one.data();
      glwe_encrypt(R, d.K, ct, d.size_ct, p->k_ct, pt.data(), pt_size, 0, s_spec, xa, xe);
      if (!cts) take_bodies(d.n, d.size_ct, 1, ct, bodies + g * glwe / 2);
    }
  return 0;
}
}  // namespace

extern "C" int fheram_encrypt_ram(const fheram_params* p, const uint8_t* data, const int64_t* sk,
                                  fheram_source* xa, fheram_source* xe, int64_t* cts) {
  if (check(p) || !data || !sk || !xa || !xe || !cts) return FHERAM_ERR_INVALID;
  return encrypt_ram(p, data, sk, xa, xe, cts, nullptr);
}

int fheram_address_monomials(const fheram_params* p, uint32_t value, int32_t* pos_out, int32_t* sign_out) {
  if (check(p)) return FHERAM_ERR_INVALID;
  const Dims d = dims(p);
  if ((u64)value >= p->max_addr) {
    fheram_set_error("address out of range (src/address.rs:96)");
    return FHERAM_ERR_INVALID;
  }
  u64 remain2d = value;
  int g = 0;
  for (int ci = 0; ci < d.n_coord; ci++) {  // src/address.rs:102-108
    u64 max = 1;
    for (int k = 0; k < d.coord_len[ci]; k++) max <<= d.coord_digits[ci][k];
    const i64 v = -(i64)(remain2d & (max - 1));
    const int sign = v > 0 ? 1 : (v < 0 ? -1 : 0);
    u64 remain = (u64)(v < 0 ? -v : v);
    int tot_base = 0;
    for (int k = 0; k < d.coord_len[ci]; k++) {  // src/coordinate.rs:148-179
      const int base = d.coord_digits[ci][k];
      const u64 chunk = (remain & ((1ull << base) - 1)) << tot_base;
      if (sign < 0 && chunk != 0) { pos_out[g] = (int32_t)(d.n - chunk); sign_out[g] = -1; }
      else { pos_out[g] = (int32_t)chunk; sign_out[g] = 1; }
      remain >>= base;
      tot_base += base;
      g++;
    }
    remain2d /= max;
  }
  return g;
}

namespace {
// Address::encrypt_sk: every GGSW into ggsw, or (ggsw null) the seeded form's body columns into bodies
int encrypt_address(const fheram_params* p, uint32_t value, const int64_t* sk, fheram_source* xa,
                    fheram_source* xe, int64_t* ggsw, int64_t* bodies) {
  const Dims d = dims(p);
  int32_t pos[64], sign[64];
  const int n_ggsw = fheram_address_monomials(p, value, pos, sign);
  if (n_ggsw < 0) return n_ggsw;
  Ring R(d.log_n);
  std::vector<cd> s_spec;
  R.forward(sk, s_spec);
  const size_t ggsw_len = fheram_ggsw_len(p);
  std::vector<i64> scalar(d.n, 0), one(ggsw ? 0 : ggsw_len);
  for (int g = 0; g < n_ggsw; g++) {
    scalar[pos[g]] = sign[g];
    i64* out = ggsw ? ggsw + (size_t)g * ggsw_len : one.data();
    ggsw_encrypt(R, d, p->k_addr, out, scalar.data(), s_spec, xa, xe, !ggsw);
    if (!ggsw) take_bodies(d.n, d.size_addr, (size_t)d.dnum_ct * 2, out, bodies + (size_t)g * ggsw_len / 2);
    scalar[pos[g]] = 0;
  }
  return 0;
}
}  // namespace

extern "C" int fheram_encrypt_address(const fheram_params* p, uint32_t value, const int64_t* sk,
                                      fheram_source* xa, fheram_source* xe, int64_t* ggsw) {
  if (check(p) || !sk || !xa || !xe || !ggsw) return FHERAM_ERR_INVALID;
  return encrypt_address(p, value, sk, xa, xe, ggsw, nullptr);
}

extern "C" int fheram_encrypt_word(const fheram_params* p, uint8_t value, const int64_t* sk,
                                   fheram_source* xa, fheram_source* xe, int64_t* glwe) {
  if (check(p) || !sk || !xa || !xe || !glwe) return FHERAM_ERR_INVALID;
  const Dims d = dims(p);
  Ring R(d.log_n);
  std::vector<cd> s_spec;
  R.forward(sk, s_spec);
  const int pt_size = cdiv(p->k_pt, d.K);
  std::vector<i64> pt((size_t)pt_size * d.n, 0);
  encode_coeff(d.n, d.K, pt.data(), pt_size, 0, (i64)value, p->k_pt);  // examples/fhe-ram.rs:197
  glwe_encrypt(R, d.K, glwe, d.size_ct, p->k_ct, pt.data(), pt_size, 0, s_spec, xa, xe);
  return 0;
}

// ---- seeded ciphertexts (fheram.h): bodies + the mask Source's state ----
extern "C" int fheram_source_seed(const fheram_source* s, fheram_seed* seed) {
  if (!s || !seed) { fheram_set_error("fheram_source_seed: null argument"); return FHERAM_ERR_INVALID; }
  fheram_source_tell(s, seed->key, &seed->word0);
  return 0;
}

namespace {
int check_seeded(const fheram_params* p, const int64_t* sk, const fheram_source* xa, const fheram_source* xe,
                 const void* bodies, const fheram_seed* seed) {
  if (check(p)) return FHERAM_ERR_INVALID;
  if (!sk || !xa || !xe || !bodies || !seed) { fheram_set_error("null argument"); return FHERAM_ERR_INVALID; }
  if (xa == xe) { fheram_set_error("mask and noise need distinct Sources"); return FHERAM_ERR_INVALID; }
  return 0;
}

// n_glwe GLWEs of `size` limbs from their bodies ([n_glwe][size][N]) and the mask stream of seed
void expand(const Dims& d, int size, size_t n_glwe, const i64* bodies, const fheram_seed* seed, i64* out) {
  fheram_source s;
  memcpy(s.key, seed->key, sizeof(s.key));
  fheram_source_skip_words(&s, seed->word0);
  const size_t n = (size_t)d.n;
  for (size_t t = 0; t < n_glwe * size; t++) {  // (GLWE, limb) in stream order, as glwe_encrypt draws them
    memcpy(out + t * 2 * n, bodies + t * n, sizeof(i64) * n);
    i64* a = out + (t * 2 + 1) * n;
    for (size_t i = 0; i < n; i++) a[i] = digit(d.K, (i64)s.next());
  }
}
}  // namespace

extern "C" int fheram_encrypt_ram_seeded(const fheram_params* p, const uint8_t* data, const int64_t* sk,
                                         fheram_source* xa, fheram_source* xe, int64_t* bodies, fheram_seed* seed) {
  if (int rc = check_seeded(p, sk, xa, xe, bodies, seed)) return rc;
  if (!data) { fheram_set_error("null argument"); return FHERAM_ERR_INVALID; }
  fheram_source_tell(xa, seed->key, &seed->word0);
  return encrypt_ram(p, data, sk, xa, xe, nullptr, bodies);
}

extern "C" int fheram_encrypt_address_seeded(const fheram_params* p, uint32_t value, const int64_t* sk,
                                             fheram_source* xa, fheram_source* xe, int64_t* bodies,
                                             fheram_seed* seed) {
  if (int rc = check_seeded(p, sk, xa, xe, bodies, seed)) return rc;
  fheram_source_tell(xa, seed->key, &seed->word0);
  return encrypt_address(p, value, sk, xa, xe, nullptr, bodies);
}

extern "C" int fheram_ram_expand(const fheram_params* p, const int64_t* bodies, const fheram_seed* seed,
                                 int64_t* cts) {
  if (check(p)) return FHERAM_ERR_INVALID;
  if (!bodies || !seed || !cts) { fheram_set_error("fheram_ram_expand: null argument"); return FHERAM_ERR_INVALID; }
  const Dims d = dims(p);
  expand(d, d.size_ct, (size_t)p->word_size * d.n_glwe, bodies, seed, cts);
  return 0;
}

extern "C" int fheram_address_expand(const fheram_params* p, const int64_t* bodies, const fheram_seed* seed,
                                     int64_t* ggsw) {
  if (check(p)) return FHERAM_ERR_INVALID;
  if (!bodies || !seed || !ggsw) { fheram_set_error("fheram_address_expand: null argument"); return FHERAM_ERR_INVALID; }
  const Dims d = dims(p);
  expand(d, d.size_addr, (size_t)d.n_ggsw * d.dnum_ct * 2, bodies, seed, ggsw);
  return 0;
}

namespace {
// pt = normalize(body + mask * s) of one GLWE(S limbs): [S][n] balanced digits; big and tmp are scratch
void decrypt_phase(const Ring& R, int K, int S, const i64* glwe, const std::vector<cd>& s_spec, std::vector<i64>& big,
                   std::vector<i64>& tmp, i64* pt) {
  const int n = R.n();
  std::vector<cd> spec, prod;
  big.resize((size_t)S * n);
  tmp.resize(n);
  for (int l = 0; l < S; l++) {
    R.forward(glwe + ((size_t)l * 2 + 1) * n, spec);
    R.mul(spec, s_spec, prod);
    R.inverse(prod, tmp.data());
    const i64* b = glwe + ((size_t)l * 2) * n;
    for (int i = 0; i < n; i++) big[(size_t)l * n + i] = tmp[i] + b[i];
  }
  normalize(n, K, S, big, pt, 1, 0);
}
}  // namespace

extern "C" int fheram_decrypt_word(const fheram_params* p, const int64_t* glwe, const int64_t* sk,
                                   int64_t want, int64_t* value, double* noise) {
  if (check(p) || !glwe || !sk || !value || !noise) return FHERAM_ERR_INVALID;
  const Dims d = dims(p);
  Ring R(d.log_n);
  std::vector<cd> s_spec;
  R.forward(sk, s_spec);
  const int n = d.n, S = d.size_ct;
  std::vector<i64> big, tmp, pt((size_t)S * n);
  decrypt_phase(R, d.K, S, glwe, s_spec, big, tmp, pt.data());
  // examples/fhe-ram.rs:229-235
  const int k = p->k_ct, log_scale = k - p->k_pt;
  i64 v = 0;
  for (int j = 0; j < S; j++) v += pt[(size_t)j * n] << (d.K * (S - 1 - j));
  v >>= (S * d.K - k);
  const i64 diff = v - want * ((i64)1 << log_scale);
  *noise = std::log2((double)(diff < 0 ? -diff : diff)) - (double)k;
  *value = (i64)std::llround((double)v / std::exp2((double)log_scale));
  return 0;
}

int fheram_decode_shifts(const fheram_params* p, int* vsh, int* ls) {
  const int S = cdiv(p->k_ct, p->base2k);
  if (p->k_ct < 1 || p->k_pt >= p->k_ct || S * p->base2k > 62) {
    fheram_set_error("decryption needs k_pt < k_ct and ceil(k_ct / base2k) * base2k <= 62");
    return FHERAM_ERR_INVALID;
  }
  *vsh = S * p->base2k - p->k_ct;
  *ls = p->k_ct - p->k_pt;
  return 0;
}

// Every byte of a RAM in fheram_encrypt_ram's layout ([word_size][n_glwe] GLWE), each GLWE decrypted as
// fheram_decrypt_word decrypts coefficient 0, on all host threads.  values / err: [max_addr][word_size].
extern "C" int fheram_decrypt_ram(const fheram_params* p, const int64_t* cts, const int64_t* sk, int16_t* values,
                                  int64_t* err) {
  if (check(p)) return FHERAM_ERR_INVALID;
  if (!cts || !sk || !values) { fheram_set_error("fheram_decrypt_ram: null argument"); return FHERAM_ERR_INVALID; }
  int vsh, ls;
  if (int rc = fheram_decode_shifts(p, &vsh, &ls)) return rc;
  const Dims d = dims(p);
  for (int i = 0; i < d.n; i++)
    if (sk[i] < -1 || sk[i] > 1) { fheram_set_error("secret key is not ternary"); return FHERAM_ERR_INVALID; }
  Ring R(d.log_n);
  std::vector<cd> s_spec;
  R.forward(sk, s_spec);
  const int n = d.n, S = d.size_ct, ws = p->word_size, G = d.n_glwe;
  const size_t glwe = fheram_glwe_len(p);
  const int total = ws * G;
  unsigned nt = std::thread::hardware_concurrency();
  nt = nt < 1 ? 1 : nt;
  if ((int)nt > total) nt = total;
  auto work = [&](unsigned t) {
    std::vector<i64> big, tmp, pt((size_t)S * n);
    for (int g = (int)t; g < total; g += (int)nt) {
      const int i = g / G, h = g % G;
      decrypt_phase(R, d.K, S, cts + (size_t)g * glwe, s_spec, big, tmp, pt.data());
      for (int j = 0; j < n; j++) {
        const u64 addr = (u64)h * n + j;
        if (addr >= p->max_addr) break;
        i64 v = 0;
        for (int l = 0; l < S; l++) v += pt[(size_t)l * n + j] * ((i64)1 << (d.K * (S - 1 - l)));
        int64_t e;
        fheram_decode(v >> vsh, ls, p->k_pt, values + addr * ws + i, &e);
        if (err) err[addr * ws + i] = e;
      }
    }
  };
  std::vector<std::thread> th;
  for (unsigned t = 1; t < nt; t++) th.emplace_back(work, t);
  work(0);
  for (auto& t : th) t.join();
  return 0;
}

// ---- packed host format: normalised base-2^17 digits as a little-endian stream of 17-bit two's-complement fields
// (limb i = bits [17 i, 17 i + 17)); 2.125 bytes per limb against 8 in Poulpy's containers.  n a multiple of 32
// (every polynomial is), out = n * 17 / 32 words.
extern "C" int fheram_pack17(const int64_t* limbs, size_t n, uint32_t* out) {
  if (!limbs || !out || n % 32) { fheram_set_error("fheram_pack17: null argument or n not a multiple of 32"); return FHERAM_ERR_INVALID; }
  int bad = 0;
  const size_t groups = n / 32;
#pragma omp parallel for schedule(static) reduction(| : bad)
  for (long long g = 0; g < (long long)groups; g++) {
    const int64_t* in = limbs + (size_t)g * 32;
    uint32_t* o = out + (size_t)g * 17;
    unsigned __int128 acc = 0;
    int bits = 0, w = 0;
    for (int k = 0; k < 32; k++) {
      const int64_t v = in[k];
      if (v < -65536 || v > 65535) bad = 1;
      acc |= (unsigned __int128)((uint64_t)v & 0x1ffffu) << bits;
      bits += 17;
      while (bits >= 32) { o[w++] = (uint32_t)acc; acc >>= 32; bits -= 32; }
    }
  }
  if (bad) { fheram_set_error("fheram_pack17: limb outside [-2^16, 2^16): only normalised digits can be packed"); return FHERAM_ERR_RANGE; }
  return 0;
}
extern "C" int fheram_unpack17(const uint32_t* packed, size_t n, int64_t* limbs) {
  if (!packed || !limbs || n % 32) { fheram_set_error("fheram_unpack17: null argument or n not a multiple of 32"); return FHERAM_ERR_INVALID; }
  for (size_t i = 0; i < n; i++) {
    const size_t bit = 17 * i, w = bit >> 5;
    const unsigned sh = (unsigned)(bit & 31);
    uint64_t two = (uint64_t)packed[w];
    if (sh > 15) two |= (uint64_t)packed[w + 1] << 32;
    const uint32_t f = (uint32_t)(two >> sh) & 0x1ffffu;
    limbs[i] = (int64_t)((int32_t)(f << 15) >> 15);
  }
  return 0;
}
