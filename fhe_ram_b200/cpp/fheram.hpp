// fheram.hpp -- C++17 mirror of the reference's Rust API over the C ABI (include/fheram.h).
// The reference host language is Rust; its toolchain is absent from this image, so the compiled
// host layer is C++ (the Rust shim is shipped as source under rust/).  Type and method names follow
// phantomzone-org/fhe-ram: Parameters (src/parameters.rs:147), EvaluationKeys /
// EvaluationKeysPrepared (src/keys.rs:21-71), Address (src/address.rs:21), Ram (src/ram.rs:25).
// Errors: where the reference panics (assert!), these throw fheram::Panic.
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "fheram.h"

namespace fheram {

struct Panic : std::runtime_error {
  int code;
  Panic(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
inline void check(int rc) {
  if (rc != 0) throw Panic(rc, fheram_last_error());
}

class Source {  // poulpy_hal::source::Source
 public:
  explicit Source(const uint8_t (&seed)[32]) : h_(fheram_source_new(seed)) {}
  static Source filled(uint8_t b) {  // Source::new([b; 32])
    uint8_t s[32];
    for (auto& x : s) x = b;
    return Source(s);
  }
  Source(Source&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
  Source(const Source&) = delete;
  ~Source() { if (h_) fheram_source_free(h_); }
  uint32_t next_u32() { return fheram_source_next_u32(h_); }
  void fill_bytes(std::vector<uint8_t>& v) { fheram_source_fill_bytes(h_, v.data(), v.size()); }
  fheram_source* raw() { return h_; }
  fheram_seed seed() const {  // the state of the stream here (seeded ciphertexts, fheram.h)
    fheram_seed s;
    check(fheram_source_seed(h_, &s));
    return s;
  }

 private:
  fheram_source* h_;
};

class Parameters {  // src/parameters.rs:147-288
 public:
  static Parameters new_() { Parameters p; fheram_params_default(&p.c); return p; }   // Parameters::new()
  static Parameters readme() { Parameters p; fheram_params_readme(&p.c); return p; }  // README.md:17-34
  size_t max_addr() const { return c.max_addr; }
  size_t word_size() const { return (size_t)c.word_size; }
  int k_glwe_pt() const { return c.k_pt; }
  int k_glwe_ct() const { return c.k_ct; }
  int basek() const { return c.base2k; }
  size_t n() const { return (size_t)1 << c.log_n; }
  size_t glwe_len() const { return fheram_glwe_len(&c); }
  size_t ggsw_len() const { return fheram_ggsw_len(&c); }
  size_t n_ggsw() const { return (size_t)fheram_n_ggsw(&c); }
  size_t n_glwe() const { return (size_t)fheram_n_glwe_per_subram(&c); }
  // Module::<B>::new(1 << LOG_N): the device context, created on first use
  fheram_ctx* module(int device = 0) {
    if (!ctx_) check(fheram_ctx_create(&c, device, &ctx_));
    return ctx_;
  }
  ~Parameters() { if (ctx_) fheram_ctx_destroy(ctx_); }
  Parameters(Parameters&& o) noexcept : c(o.c), ctx_(o.ctx_) { o.ctx_ = nullptr; }
  Parameters(const Parameters&) = delete;
  fheram_params c;

 private:
  Parameters() = default;
  fheram_ctx* ctx_ = nullptr;
};

struct GLWESecret {  // GLWESecret::alloc_from_infos + fill_ternary_prob(0.5, xs)
  std::vector<int64_t> data;
  static GLWESecret fill_ternary_prob(const Parameters& p, double prob, Source& xs) {
    if (prob != 0.5) throw Panic(-1, "only prob = 0.5 is used by the reference");
    GLWESecret s;
    s.data.resize(p.n());
    check(fheram_secret_gen(&p.c, xs.raw(), s.data.data()));
    return s;
  }
};

struct EvaluationKeys {  // src/keys.rs:21-25
  std::vector<int64_t> atk_glwe, gglwe_to_ggsw_key, atk_ggsw_inv;
  static EvaluationKeys encrypt_sk(const Parameters& p, const GLWESecret& sk, Source& xa, Source& xe) {  // :135-180
    EvaluationKeys k;
    k.atk_glwe.resize((size_t)fheram_n_trace_keys(&p.c) * fheram_atk_len(&p.c));
    k.gglwe_to_ggsw_key.resize(fheram_evk_inv_len(&p.c));
    k.atk_ggsw_inv.resize(fheram_evk_inv_len(&p.c));
    check(fheram_keygen(&p.c, sk.data.data(), xa.raw(), xe.raw(), k.atk_glwe.data(),
                        k.gglwe_to_ggsw_key.data(), k.atk_ggsw_inv.data()));
    return k;
  }
};

class EvaluationKeysPrepared {  // src/keys.rs:27-71
 public:
  static EvaluationKeysPrepared alloc(Parameters& p) { return EvaluationKeysPrepared(p); }
  // EvaluationKeys::encrypt_sk (:135-180) + prepare on the device: same limbs, keys never leave the GPU
  static EvaluationKeysPrepared encrypt_sk_device(Parameters& p, const GLWESecret& sk, Source& xa, Source& xe) {
    EvaluationKeysPrepared k(p);
    check(fheram_keys_encrypt_sk(p.module(), sk.data.data(), xa.raw(), xe.raw(), &k.h_));
    return k;
  }
  void prepare(const EvaluationKeys& k) {
    check(fheram_keys_prepare(p_.module(), k.atk_glwe.data(), k.gglwe_to_ggsw_key.data(), k.atk_ggsw_inv.data(), &h_));
  }
  ~EvaluationKeysPrepared() { if (h_) fheram_keys_destroy(h_); }
  fheram_keys* raw() const { return h_; }

 private:
  explicit EvaluationKeysPrepared(Parameters& p) : p_(p) {}
  Parameters& p_;
  fheram_keys* h_ = nullptr;
};

class Address {  // src/address.rs:21-24
 public:
  static Address alloc_from_params(Parameters& p) { return Address(p); }  // :58-60
  void encrypt_sk(const Parameters& p, uint32_t value, const GLWESecret& sk, Source& xa, Source& xe) {  // :86-109
    check(fheram_encrypt_address(&p.c, value, sk.data.data(), xa.raw(), xe.raw(), data.data()));
    if (h_) { fheram_address_destroy(h_); h_ = nullptr; }
    seeded_ = false;
    bodies.clear();
  }
  // the seeded form (fheram.h): bodies + the mask Source's seed, half the bytes; data = its expanded limbs (another
  // valid encryption than encrypt_sk's), device() uploads the bodies and regenerates the masks on the GPU
  void encrypt_sk_seeded(const Parameters& p, uint32_t value, const GLWESecret& sk, Source& xa, Source& xe) {
    bodies.resize(data.size() / 2);
    check(fheram_encrypt_address_seeded(&p.c, value, sk.data.data(), xa.raw(), xe.raw(), bodies.data(), &seed));
    check(fheram_address_expand(&p.c, bodies.data(), &seed, data.data()));
    if (h_) { fheram_address_destroy(h_); h_ = nullptr; }
    seeded_ = true;
  }
  fheram_address* device() {  // resident + CoordinatePrepared::prepare
    if (!h_) check(seeded_ ? fheram_address_load_seeded(p_.module(), bodies.data(), &seed, 1, &h_)
                           : fheram_address_load(p_.module(), data.data(), &h_));
    return h_;
  }
  ~Address() { if (h_) fheram_address_destroy(h_); }
  std::vector<int64_t> data;
  std::vector<int64_t> bodies;  // seeded form only
  fheram_seed seed{};

 private:
  explicit Address(Parameters& p) : data(p.n_ggsw() * p.ggsw_len()), p_(p) {}
  Parameters& p_;
  fheram_address* h_ = nullptr;
  bool seeded_ = false;
};

using GLWE = std::vector<int64_t>;

class Ram {  // src/ram.rs:25-29
 public:
  explicit Ram(Parameters& p) : p_(p) { check(fheram_ram_create(p.module(), &h_)); }  // Ram::new()
  // multi-GPU (one process per GPU): rank `rank` of `n_ranks`; id = the 128 bytes of Ram::comm_unique_id() on rank 0,
  // handed to the other ranks by the host program.  read / read_prepare_write / write keep their signatures.
  Ram(Parameters& p, int n_ranks, int rank, const uint8_t (&id)[128]) : p_(p) {
    check(fheram_comm_init(p.module(), n_ranks, rank, id));
    check(fheram_ram_create_sharded(p.module(), rank, n_ranks, &h_));
  }
  static void comm_unique_id(uint8_t (&id)[128]) { check(fheram_comm_unique_id(id)); }
  ~Ram() { if (h_) fheram_ram_destroy(h_); }
  void encrypt_sk(const std::vector<uint8_t>& data, const GLWESecret& sk, Source& xa, Source& xe) {  // :129-167
    if (data.size() % p_.word_size() != 0) throw Panic(-1, "invalid data: data.len()%ram_chunks != 0");
    if (data.size() / p_.word_size() != p_.max_addr()) throw Panic(-1, "invalid data: data.len()/ram_chunks != max_addr");
    // on the device, straight into the resident RAM: the limbs fheram_encrypt_ram + fheram_ram_load would install
    check(fheram_ram_encrypt_sk(h_, data.data(), sk.data.data(), xa.raw(), xe.raw()));
  }
  // Ram::encrypt_sk on the client (CPU) in the seeded form, then load_seeded: bodies + seed are what a separated
  // client ships (half the bytes of the limbs), and they expand to exactly the limbs of fheram_encrypt_ram
  void encrypt_sk_seeded(const std::vector<uint8_t>& data, const GLWESecret& sk, Source& xa, Source& xe,
                         std::vector<int64_t>& bodies, fheram_seed& seed) {
    if (data.size() != p_.max_addr() * p_.word_size()) throw Panic(-1, "invalid data: data.len() != max_addr * ram_chunks");
    bodies.resize(p_.word_size() * p_.n_glwe() * p_.glwe_len() / 2);
    check(fheram_encrypt_ram_seeded(&p_.c, data.data(), sk.data.data(), xa.raw(), xe.raw(), bodies.data(), &seed));
    load_seeded(bodies, seed);
  }
  void load_seeded(const std::vector<int64_t>& bodies, const fheram_seed& seed) {
    if (bodies.size() != p_.word_size() * p_.n_glwe() * p_.glwe_len() / 2) throw Panic(-1, "bodies are not a whole RAM");
    check(fheram_ram_load_seeded(h_, bodies.data(), &seed));
  }
  // n seeded addresses from host buffers: bodies packed by fheram_pack17, one seed each; int32 limbs out
  std::vector<int32_t> read_batch_host_seeded(const std::vector<uint32_t>& bodies_p17, const std::vector<fheram_seed>& seeds,
                                              const EvaluationKeysPrepared& k) {
    const int n = (int)seeds.size();
    if (bodies_p17.size() != (size_t)n * p_.n_ggsw() * p_.ggsw_len() / 2 * 17 / 32)
      throw Panic(-1, "bodies_p17 does not hold one packed address per seed");
    std::vector<int32_t> out((size_t)n * p_.word_size() * p_.glwe_len());
    check(fheram_ram_read_batch_host_seeded(h_, bodies_p17.data(), seeds.data(), n, k.raw(), out.data()));
    return out;
  }
  std::vector<GLWE> read(Address& a, const EvaluationKeysPrepared& k) {  // :172-191
    std::vector<int64_t> out(p_.word_size() * p_.glwe_len());
    check(fheram_ram_read(h_, a.device(), k.raw(), out.data()));
    return split(out);
  }
  std::vector<GLWE> read_prepare_write(Address& a, const EvaluationKeysPrepared& k) {  // :196-222
    std::vector<int64_t> out(p_.word_size() * p_.glwe_len());
    check(fheram_ram_read_prepare_write(h_, a.device(), k.raw(), out.data()));
    return split(out);
  }
  void write(const std::vector<GLWE>& w, Address& a, const EvaluationKeysPrepared& k) {  // :226-294
    if (w.size() != p_.word_size()) throw Panic(-1, "assertion failed: w.len() == self.subrams.len()");
    std::vector<int64_t> flat;
    for (auto& g : w) flat.insert(flat.end(), g.begin(), g.end());
    check(fheram_ram_write(h_, flat.data(), a.device(), k.raw()));
  }
  // reads / writes at plaintext addresses (include/fheram.h): the address is disclosed to the server, the words stay
  // encrypted.  read_plain: one [word_size] GLWE per address
  std::vector<std::vector<GLWE>> read_plain(const std::vector<uint32_t>& addrs, const EvaluationKeysPrepared& k) {
    std::vector<int64_t> out(addrs.size() * p_.word_size() * p_.glwe_len());
    check(fheram_ram_read_plain(h_, addrs.data(), (int)addrs.size(), k.raw(), out.data()));
    std::vector<std::vector<GLWE>> r;
    const size_t per = p_.word_size() * p_.glwe_len();
    for (size_t b = 0; b < addrs.size(); b++) r.push_back(split(std::vector<int64_t>(out.begin() + b * per, out.begin() + (b + 1) * per)));
    return r;
  }
  void write_plain(uint32_t addr, const std::vector<GLWE>& w, const EvaluationKeysPrepared& k) {
    if (w.size() != p_.word_size()) throw Panic(-1, "assertion failed: w.len() == self.subrams.len()");
    std::vector<int64_t> flat;
    for (auto& g : w) flat.insert(flat.end(), g.begin(), g.end());
    check(fheram_ram_write_plain(h_, addr, flat.data(), k.raw()));
  }
  // every byte of the resident RAM decrypted on the device: values / err are [max_addr][word_size] row-major (byte i of
  // word j at j * word_size + i), the numbers of fheram_decrypt_ram on the stored RAM, bit for bit
  void decrypt_sk(const GLWESecret& sk, std::vector<int16_t>& values, std::vector<int64_t>& err) {
    values.assign(p_.max_addr() * p_.word_size(), 0);
    err.assign(values.size(), 0);
    check(fheram_ram_decrypt_sk(h_, sk.data.data(), values.data(), err.data()));
  }

 private:
  std::vector<GLWE> split(const std::vector<int64_t>& o) {
    std::vector<GLWE> r;
    for (size_t i = 0; i < p_.word_size(); i++) r.emplace_back(o.begin() + i * p_.glwe_len(), o.begin() + (i + 1) * p_.glwe_len());
    return r;
  }
  Parameters& p_;
  fheram_ram* h_ = nullptr;
};

// coefficient 0 of n device-resident GLWE(k_ct) (int32 [n][limb][col][N], e.g. a batched read's result arena),
// decrypted on the device
inline void decrypt_words_device(Parameters& p, const int32_t* d_glwe, int n, const GLWESecret& sk,
                                 std::vector<int16_t>& values, std::vector<int64_t>& err) {
  values.assign((size_t)n, 0);
  err.assign((size_t)n, 0);
  check(fheram_decrypt_words_device(p.module(), d_glwe, n, sk.data.data(), values.data(), err.data()));
}

}  // namespace fheram
