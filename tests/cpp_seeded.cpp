// The seeded calls of the C++ host layer (fhe_ram_b200/cpp/fheram.hpp), run by tests/test_gpu_cpp_seeded.py.
// One Address object is reused across accesses, as the reference example does, alternating the seeded and the full
// encryption: every read must return the word of the address the object was last encrypted with.  Then a seeded RAM
// and a batch of seeded addresses from host buffers.  Prints OK and exits 0 when every decryption holds.
#include <cstdio>
#include <vector>

#include "fheram.hpp"

using namespace fheram;

static int64_t cast_u8_to_signed(uint8_t v, int bits) {
  int shift = 8 - bits;
  return (int64_t)((int8_t)(uint8_t)(v << shift)) >> shift;
}

static int failures = 0;
static void expect_word(const Parameters& p, const GLWESecret& sk, const int64_t* glwe_limbs, size_t glwe_len,
                        const std::vector<uint8_t>& data, uint32_t idx, const char* what) {
  const size_t ws = p.word_size();
  for (size_t i = 0; i < ws; i++) {
    const int64_t want = cast_u8_to_signed(data[i + ws * idx], p.k_glwe_pt());
    int64_t v;
    double noise;
    check(fheram_decrypt_word(&p.c, glwe_limbs + i * glwe_len, sk.data.data(), want, &v, &noise));
    if (v != want || !(noise < -(p.k_glwe_pt() + 1.0))) {
      printf("FAIL %s: address %u byte %zu: got %lld want %lld noise %f\n", what, idx, i, (long long)v,
             (long long)want, noise);
      failures++;
    }
  }
}

int main() {
  try {
    Parameters params = Parameters::new_();
    params.c.max_addr = 1ull << 13;
    params.c.word_size = 2;
    params.c.k_pt = 8;
    Source xs = Source::filled(1), xa = Source::filled(2), xe = Source::filled(3);
    GLWESecret sk = GLWESecret::fill_ternary_prob(params, 0.5, xs);
    EvaluationKeys keys = EvaluationKeys::encrypt_sk(params, sk, xa, xe);
    EvaluationKeysPrepared kp = EvaluationKeysPrepared::alloc(params);
    kp.prepare(keys);
    Source src = Source::filled(5);
    const size_t ws = params.word_size(), L = params.glwe_len();
    std::vector<uint8_t> data(params.max_addr() * ws);
    src.fill_bytes(data);
    Ram ram(params);
    std::vector<int64_t> ram_bodies;
    fheram_seed ram_seed;
    Source ya = Source::filled(6), ye = Source::filled(7);
    ram.encrypt_sk_seeded(data, sk, ya, ye, ram_bodies, ram_seed);

    // one Address object, seeded and full encryptions alternating
    Address addr = Address::alloc_from_params(params);
    const uint32_t idxs[4] = {17, 4097, 8000, 3};
    for (int k = 0; k < 4; k++) {
      if (k % 2 == 0) addr.encrypt_sk_seeded(params, idxs[k], sk, xa, xe);
      else addr.encrypt_sk(params, idxs[k], sk, xa, xe);
      std::vector<GLWE> got = ram.read(addr, kp);
      std::vector<int64_t> flat;
      for (auto& g : got) flat.insert(flat.end(), g.begin(), g.end());
      expect_word(params, sk, flat.data(), L, data, idxs[k], k % 2 == 0 ? "read, seeded address" : "read, full address");
    }

    // a batch of seeded addresses from host buffers
    const int n = 5;
    std::vector<int64_t> bodies;
    std::vector<fheram_seed> seeds;
    std::vector<uint32_t> values;
    for (int i = 0; i < n; i++) {
      Address a = Address::alloc_from_params(params);
      values.push_back((uint32_t)((977 * i + 11) % params.max_addr()));
      a.encrypt_sk_seeded(params, values.back(), sk, xa, xe);
      bodies.insert(bodies.end(), a.bodies.begin(), a.bodies.end());
      seeds.push_back(a.seed);
    }
    std::vector<uint32_t> packed(bodies.size() * 17 / 32);
    check(fheram_pack17(bodies.data(), bodies.size(), packed.data()));
    std::vector<int32_t> out = ram.read_batch_host_seeded(packed, seeds, kp);
    std::vector<int64_t> wide(out.begin(), out.end());
    for (int i = 0; i < n; i++) expect_word(params, sk, wide.data() + (size_t)i * ws * L, L, data, values[i], "batch");
  } catch (const std::exception& e) {
    printf("FAIL exception: %s\n", e.what());
    return 1;
  }
  if (failures) return 1;
  printf("OK\n");
  return 0;
}
