// fheram_cuda.cu -- host side of libfheram_cuda.so: device contexts, HBM-resident keys /
// addresses / RAM, and the launch schedules of read / read_prepare_write / write.
// Mirrors (not copies) the control flow of the reference's src/ram.rs; every schedule step
// cites the lines it reproduces.  There is no CPU fallback anywhere in this file.
#include <cuda_runtime.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/fheram.h"
#include "kernels.cuh"
#include "kernels_ks2.cuh"
#include "kernels_ks3.cuh"
#include "kernels_ks4.cuh"
#include "kernels_ks5.cuh"
#include "kernels_ks6.cuh"
#include "kernels_ks7.cuh"
#include "kernels_ext8.cuh"
#include "kernels_ks8.cuh"
#include "kernels_ext9.cuh"
#include "kernels_enc.cuh"
#include "client_internal.h"

using namespace fheram;

// --------------------------------------------------------------------------------------
// errors
// --------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
extern "C" const char* fheram_last_error(void) { return g_err.c_str(); }
extern "C" const char* fheram_version(void) { return "fheram-b200 0.1 (sm_100a)"; }
void fheram_set_error(const char* msg) { g_err = msg; }

#define CU(x)                                                                         \
  do {                                                                                \
    cudaError_t e_ = (x);                                                             \
    if (e_ != cudaSuccess)                                                            \
      return fail(FHERAM_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #x,            \
                  cudaGetErrorString(e_));                                            \
  } while (0)
#define NC(x)                                                                         \
  do {                                                                                \
    ncclResult_t e_ = (x);                                                            \
    if (e_ != ncclSuccess)                                                            \
      return fail(FHERAM_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #x,            \
                  ncclGetErrorString(e_));                                            \
  } while (0)
#define TRY(x)            \
  do {                    \
    int rc_ = (x);        \
    if (rc_) return rc_;  \
  } while (0)

// --------------------------------------------------------------------------------------
// parameters / derived sizes
// --------------------------------------------------------------------------------------
static int cdiv(int a, int b) { return (a + b - 1) / b; }

struct Derived {
  int n, log_n, size_ct, dnum_ct, size_addr, size_evk_trace, dnum_ggsw, size_evk_inv;
  int n_coord, coord_len[8], coord_digits[8][8], n_ggsw, n_glwe;
};

extern "C" void fheram_params_default(fheram_params* p) {  // src/parameters.rs:11-21
  memset(p, 0, sizeof(*p));
  p->log_n = 12; p->base2k = 17; p->k_pt = 3; p->k_ct = 51; p->k_addr = 68;
  p->k_evk_trace = 68; p->k_evk_ggsw_inv = 85; p->word_size = 4; p->n_decomp = 4;
  for (int i = 0; i < 4; i++) p->decomp_n[i] = 3;
  p->max_addr = 1u << 14;
}
extern "C" void fheram_params_readme(fheram_params* p) {  // README.md:17-34
  fheram_params_default(p);
  p->k_pt = 9;
  p->max_addr = 1u << 18;
}

// get_base_2d, src/base.rs:84-108
static int base2d(uint32_t value, const int32_t* base, int n_base, int32_t* lens, int32_t* digits) {
  int n_out = 0;
  uint32_t vm1 = value - 1;
  int bits = vm1 == 0 ? 0 : 32 - __builtin_clz(vm1);
  while (bits != 0 && n_out < 8) {
    int len = 0;
    for (int i = 0; i < n_base; i++) {
      int b = base[i];
      if (b <= bits) { digits[n_out * 8 + len++] = b; bits -= b; }
      else { if (bits != 0) { digits[n_out * 8 + len++] = bits; bits = 0; } break; }
    }
    lens[n_out++] = len;
  }
  return n_out;
}

// one validation for fheram_ctx_create, the size helpers and the client side (client.cpp): the digit tables of
// fheram_params / Derived hold 8 entries per coordinate and 8 coordinates
int fheram_params_check(const fheram_params* p) {
  if (!p) return fail(FHERAM_ERR_INVALID, "null parameters");
  if (p->log_n < 1 || p->log_n > 16 || p->base2k < 1 || p->base2k > 30)
    return fail(FHERAM_ERR_INVALID, "bad log_n / base2k");
  if (p->n_decomp < 1 || p->n_decomp > 8)
    return fail(FHERAM_ERR_INVALID, "n_decomp must be in 1..8 (decomp_n[8])");
  int sum = 0;
  for (int i = 0; i < p->n_decomp; i++) {
    if (p->decomp_n[i] < 1 || p->decomp_n[i] > p->log_n) return fail(FHERAM_ERR_INVALID, "decomp_n[%d] out of range", i);
    sum += p->decomp_n[i];
  }
  if (sum != p->log_n) return fail(FHERAM_ERR_INVALID, "sum(decomp_n) != log_n (src/parameters.rs:168)");
  if (p->max_addr < 1 || p->max_addr > (1ull << (2 * p->log_n)))
    return fail(FHERAM_ERR_INVALID, "max_addr must be in 1..N^2 (the reference's read loop supports two coordinates)");
  if (p->word_size < 1 || p->word_size > 16 || p->k_pt < 1 || p->k_pt > 16)
    return fail(FHERAM_ERR_INVALID, "bad word_size / k_pt");
  return 0;
}

static Derived derive(const fheram_params* p) {
  Derived d;
  memset(&d, 0, sizeof(d));
  d.log_n = p->log_n; d.n = 1 << p->log_n;
  d.size_ct = cdiv(p->k_ct, p->base2k);
  d.dnum_ct = d.size_ct;                       // src/parameters.rs:138-140
  d.size_addr = cdiv(p->k_addr, p->base2k);
  d.size_evk_trace = cdiv(p->k_evk_trace, p->base2k);
  d.dnum_ggsw = cdiv(p->k_addr, p->base2k);    // src/parameters.rs:142-144
  d.size_evk_inv = cdiv(p->k_evk_ggsw_inv, p->base2k);
  int32_t lens[8], digits[64];
  d.n_coord = base2d((uint32_t)p->max_addr, p->decomp_n, p->n_decomp, lens, digits);
  for (int i = 0; i < d.n_coord; i++) {
    d.coord_len[i] = lens[i];
    for (int j = 0; j < lens[i]; j++) d.coord_digits[i][j] = digits[i * 8 + j];
    d.n_ggsw += lens[i];
  }
  d.n_glwe = (int)((p->max_addr + (uint64_t)d.n - 1) / (uint64_t)d.n);
  return d;
}

extern "C" size_t fheram_glwe_len(const fheram_params* p) { if (fheram_params_check(p)) return 0; Derived d = derive(p); return (size_t)2 * d.size_ct * d.n; }
extern "C" size_t fheram_ggsw_len(const fheram_params* p) { if (fheram_params_check(p)) return 0; Derived d = derive(p); return (size_t)d.dnum_ct * 4 * d.size_addr * d.n; }
extern "C" size_t fheram_atk_len(const fheram_params* p) { if (fheram_params_check(p)) return 0; Derived d = derive(p); return (size_t)d.dnum_ct * 2 * d.size_evk_trace * d.n; }
extern "C" size_t fheram_evk_inv_len(const fheram_params* p) { if (fheram_params_check(p)) return 0; Derived d = derive(p); return (size_t)d.dnum_ggsw * 2 * d.size_evk_inv * d.n; }
extern "C" int fheram_n_trace_keys(const fheram_params* p) { return p->log_n; }
extern "C" int fheram_n_ggsw(const fheram_params* p) { return fheram_params_check(p) ? 0 : derive(p).n_ggsw; }
extern "C" int fheram_n_glwe_per_subram(const fheram_params* p) { return fheram_params_check(p) ? 0 : derive(p).n_glwe; }
extern "C" int fheram_base2d(const fheram_params* p, int32_t lens[8], int32_t digits[64]) {
  if (fheram_params_check(p)) return FHERAM_ERR_INVALID;
  return base2d((uint32_t)p->max_addr, p->decomp_n, p->n_decomp, lens, digits);
}
static int64_t galois(int log_n, int i) {  // Poulpy GLWE::trace_galois_elements
  if (i == 0) return -1;
  const uint64_t two_n = 2ull << log_n;
  uint64_t r = 1, b = 5, e = 1ull << (i - 1);
  while (e) { if (e & 1) r = r * b % two_n; b = b * b % two_n; e >>= 1; }
  return (int64_t)r;
}
extern "C" int64_t fheram_trace_galois_element(const fheram_params* p, int i) { return galois(p->log_n, i); }

static uint32_t revbits(uint32_t x, int n) {  // src/lib.rs:23-26
  uint32_t r = 0;
  for (int i = 0; i < n; i++) r |= ((x >> i) & 1u) << (n - 1 - i);
  return r;
}
static int ilog2(int x) { int l = 0; while ((1 << l) < x) l++; return l; }

// --------------------------------------------------------------------------------------
// context
// --------------------------------------------------------------------------------------
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  int ensure(size_t need) {
    if (need <= bytes) return 0;
    // growing while kernels that read the old buffer may still be queued: wait for them explicitly (cudaFree would
    // also synchronise the device, but the guarantee should not hang on an implementation detail of the allocator)
    if (p) { cudaDeviceSynchronize(); cudaFree(p); }
    p = nullptr; bytes = 0;
    cudaError_t e = cudaMalloc(&p, need);
    if (e != cudaSuccess) return fail(FHERAM_ERR_CUDA, "cudaMalloc(%zu): %s", need, cudaGetErrorString(e));
    bytes = need;
    return 0;
  }
  void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
};

constexpr size_t kSmallDownload = (size_t)1 << 19;  // limbs (2 MiB of int32): up to 21 GLWEs at N = 4096, k = 51
struct fheram_ctx {
  fheram_params params;
  Derived d;
  int device = 0, sm_count = 148;
  int ext9_clusters[2] = {0, 0}; // the same for k_ext9
  int ks8_clusters[2] = {0, 0};  // clusters of k_ks8 that can be resident together: [0] eight SMs each, [1] four
  int force_ext = 0, force_ks = 0;  // kernels forced by FHERAM_KERNEL (enum Force), FORCE_NONE: the launch-width rule
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  cudaStream_t copy_stream = nullptr;  // uploads of the asynchronous address path
  // side stream of read_prepare_write: the inverse address of the write that follows (prepare_inv) is built beside
  // the read instead of behind it; its kernels take their per-CTA scratch from scratch_side
  cudaStream_t side = nullptr;
  cudaEvent_t side_fork = nullptr, side_join = nullptr;
  bool on_side = false;
  // multi-GPU (SURVEY.md 8e): one context per rank, NCCL communicator over NVLink (fheram_comm_init)
  ncclComm_t comm = nullptr;
  ncclComm_t comm_prep = nullptr;  // second communicator: all-gather of prepared GGSWs on the upload stream, beside the reads
  int n_ranks = 1, rank = 0;
  double2* d_tw = nullptr;  // tw6 | tw7c | tw8c | tw9 | tw10c
  double2* d_tw16 = nullptr;  // twiddles of the 16-point transform (kernels_ks7.cuh): [16][16] | [128][7]
  Twiddles tw;
  int* d_err = nullptr;
  uint64_t launches = 0;
  DevBuf stage64;   // int64 staging for uploads / downloads
  DevBuf scratch;   // per-CTA scratch of the vmp kernels
  DevBuf scratch_side;
  int* pin32 = nullptr;  // pinned host buffer of small downloads (download_i64)
  DevBuf enc_buf[15];  // operands of the encryption kernels, kept between calls (cudaFree synchronizes the device)
  uint64_t enc_stats[3] = {0, 0, 0};  // noise draws sampled on the device / patched by the host / streams resampled on the host
  DevBuf opbuf[3];  // op-level entry points
  long long* d_phase = nullptr;  // per-CTA phase cycle counters (fheram_debug_phase_cycles)
  // per-kernel-class CUDA-event timing (fheram_ctx_profile)
  bool profile = false;
  std::vector<cudaEvent_t> ev_pool;
  struct EvRec { int cls; size_t e0, e1; uint64_t items, steps; };
  std::vector<EvRec> ev_recs;
  size_t ev_used = 0;
  long ct_stride() const { return (long)2 * d.size_ct * d.n; }          // ints per GLWE(k_ct)
  long ggsw_raw_len() const { return (long)d.dnum_ct * 4 * d.size_addr * d.n; }
  long ggsw_prep_len() const { return (long)d.dnum_ct * 2 * 2 * d.size_addr * kM; }  // double2
  long atk_prep_len() const { return (long)d.dnum_ct * 2 * d.size_evk_trace * kM; }
  long evk_inv_prep_len() const { return (long)d.dnum_ggsw * 2 * d.size_evk_inv * kM; }
};

static size_t smem_bytes(int R) { return (size_t)R * kM * sizeof(double2) + kM * sizeof(double2); }

// kernel instantiations used by the schedules
#define K_AUTO3    k_vmp<3, 4, 3, MODE_AUTO>
#define K_AUTO_INV k_vmp<4, 5, 4, MODE_AUTO>
#define K_EXPAND   k_vmp<4, 5, 4, MODE_EXPAND>

static int set_attrs() {
  CU(cudaFuncSetAttribute(K_AUTO3, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(3)));
  CU(cudaFuncSetAttribute(K_AUTO_INV, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(4)));
  CU(cudaFuncSetAttribute(K_EXPAND, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(4)));
  CU(cudaFuncSetAttribute(k_ks7, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kKs7Smem));
  CU(cudaFuncSetAttribute(k_prepare7, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPrep7Smem));
  CU(cudaFuncSetAttribute(k_ext8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kExt8Smem));
  CU(cudaFuncSetAttribute(k_ext9<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ext9_smem(8)));
  CU(cudaFuncSetAttribute(k_ext9<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ext9_smem(4)));
  CU(cudaFuncSetAttribute(k_ks8<8, MODE_TRACE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ks8_smem(8)));
  CU(cudaFuncSetAttribute(k_ks8<8, MODE_COMBINE2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ks8_smem(8)));
  CU(cudaFuncSetAttribute(k_ks8<4, MODE_TRACE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ks8_smem(4)));
  CU(cudaFuncSetAttribute(k_ks8<4, MODE_COMBINE2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ks8_smem(4)));
  CU(cudaFuncSetAttribute(k_ks6<MODE_TRACE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kKs5Smem));
  CU(cudaFuncSetAttribute(k_ks6<MODE_COMBINE2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kKs5Smem));
  CU(cudaFuncSetAttribute(k_ks5<MODE_TRACE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kKs5Smem));
  CU(cudaFuncSetAttribute(k_ks5<MODE_COMBINE2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kKs5Smem));
  CU(cudaFuncSetAttribute(k_ks4, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kKs4Smem));
  return 0;
}

// FHERAM_KERNEL: a test / A-B timing hook that forces kernels instead of the launch-width rule (DESIGN.md 3.4), a
// comma-separated list of at most one external-product name (ext*) and one key-switch name (ks*)
enum Force { FORCE_NONE, FORCE_EXT8, FORCE_EXT9, FORCE_EXT9C4, FORCE_KS8, FORCE_KS8C4, FORCE_KS7, FORCE_KS6, FORCE_KS5,
             FORCE_KS4, FORCE_COUNT };
static const char* const kForceNames[FORCE_COUNT] = {"", "ext8", "ext9", "ext9c4", "ks8", "ks8c4", "ks7", "ks6", "ks5",
                                                     "ks4"};
static int parse_force(const char* spec, int* force_ext, int* force_ks) {
  *force_ext = *force_ks = FORCE_NONE;
  if (!spec || !*spec) return 0;
  const std::string list(spec);
  for (size_t pos = 0; pos <= list.size();) {
    size_t end = list.find(',', pos);
    if (end == std::string::npos) end = list.size();
    const std::string name = list.substr(pos, end - pos);
    int f = FORCE_NONE;
    for (int i = 1; i < FORCE_COUNT; i++)
      if (name == kForceNames[i]) f = i;
    int* slot = f >= FORCE_KS8 ? force_ks : force_ext;
    if (f == FORCE_NONE || *slot != FORCE_NONE)
      return fail(FHERAM_ERR_INVALID,
                  "FHERAM_KERNEL=%s: expected at most one of ext8 ext9 ext9c4 and one of ks8 ks8c4 ks7 ks6 ks5 ks4, "
                  "comma-separated", spec);
    *slot = f;
    pos = end + 1;
  }
  return 0;
}

static void zeta(int s, int b, double2* out) {
  const long double PI = 3.14159265358979323846264338327950288L;
  long double th = (0.25L + (long double)revbits((uint32_t)b, s)) / (long double)(1ull << s);
  out->x = (double)cosl(PI * th);
  out->y = (double)sinl(PI * th);
}

extern "C" int fheram_ctx_create(const fheram_params* p, int device, fheram_ctx** out) {
  if (!p || !out) return fail(FHERAM_ERR_INVALID, "null argument");
  if (p->log_n != 12 || p->base2k != 17 || p->k_ct != 51 || p->k_addr != 68 ||
      p->k_evk_trace != 68 || p->k_evk_ggsw_inv != 85)
    return fail(FHERAM_ERR_INVALID,
                "unsupported cryptographic parameters: kernels are built for log_n=12 base2k=17 "
                "k_ct=51 k_addr=68 k_evk_trace=68 k_evk_ggsw_inv=85 (src/parameters.rs:11-18)");
  TRY(fheram_params_check(p));
  Derived d = derive(p);
  if (d.n_coord > 2)
    return fail(FHERAM_ERR_INVALID, "max_addr > N^2: the reference's read loop only supports two coordinates");
  if (d.n_glwe & (d.n_glwe - 1))
    return fail(FHERAM_ERR_INVALID, "max_addr / N must be a power of two");
  int force_ext = FORCE_NONE, force_ks = FORCE_NONE;
  TRY(parse_force(getenv("FHERAM_KERNEL"), &force_ext, &force_ks));
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(FHERAM_ERR_CUDA, "no CUDA device: %s (there is no CPU fallback)", cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(FHERAM_ERR_INVALID, "device %d out of range", device);
  CU(cudaSetDevice(device));
  fheram_ctx* c = new fheram_ctx();
  c->params = *p;
  c->d = d;
  c->device = device;
  c->force_ext = force_ext;
  c->force_ks = force_ks;
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  c->sm_count = prop.multiProcessorCount;
  if (prop.major < 10) {
    delete c;
    return fail(FHERAM_ERR_CUDA, "device %s is sm_%d%d; this library is built for sm_100a only",
                prop.name, prop.major, prop.minor);
  }
  CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  TRY(set_attrs());
  // twiddles
  std::vector<double2> lo(64), hi(64 + 64 + 128 + 512 + 512);
  lo[0] = make_double2(0, 0);
  for (int s = 0; s < 6; s++)
    for (int b = 0; b < (1 << s); b++) zeta(s, b, &lo[(1 << s) + b]);
  double2* q = hi.data();
  for (int b = 0; b < 64; b++) zeta(6, b, q++);
  for (int b = 0; b < 64; b++) zeta(7, 2 * b, q++);
  for (int b = 0; b < 128; b++) zeta(8, 2 * b, q++);
  for (int b = 0; b < 512; b++) zeta(9, b, q++);
  // zeta(9, 2k+1) = i zeta(9, 2k): the odd entries (load_tw34 loads them) are set from the even ones, so the
  // identity holds bit for bit
  for (int b = 1; b < 512; b += 2) q[b - 512] = make_double2(-q[b - 513].y, q[b - 513].x);
  for (int b = 0; b < 512; b++) zeta(10, 2 * b, q++);
  // zeta(10, 4k+2) = e^(i pi/4) zeta(10, 4k): same treatment, rounded as ((x - y) r, (x + y) r), r = fl(1/sqrt 2)
  for (int b = 1; b < 512; b += 2) {
    const double2 w = q[b - 513];
    const volatile double dx = w.x - w.y, sx = w.x + w.y;
    const double r = 0.70710678118654757;
    q[b - 512] = make_double2(dx * r, sx * r);
  }
  CU(cudaMemcpyToSymbol(c_tw_lo, lo.data(), sizeof(double2) * 64));
  CU(cudaMalloc(&c->d_tw, sizeof(double2) * hi.size()));
  CU(cudaMemcpy(c->d_tw, hi.data(), sizeof(double2) * hi.size(), cudaMemcpyHostToDevice));
  c->tw.tw6 = c->d_tw;
  c->tw.tw7c = c->d_tw + 64;
  c->tw.tw8c = c->d_tw + 128;
  c->tw.tw9 = c->d_tw + 256;
  c->tw.tw10c = c->d_tw + 768;
  {
    std::vector<double2> t16(kTw16Len);
    t16[0] = make_double2(0, 0);
    for (int a = 0; a < 16; a++)
      for (int k = 1; k < 16; k++) {
        int sl = 0;
        while ((2 << sl) <= k) sl++;
        zeta(4 + sl, (a << sl) + (k - (1 << sl)), &t16[16 * a + k]);
      }
    for (int t = 0; t < 128; t++) {
      double2* p = &t16[256 + 7 * t];
      zeta(8, 2 * t, p); zeta(9, 4 * t, p + 1); zeta(9, 4 * t + 2, p + 2);
      for (int k = 0; k < 4; k++) zeta(10, 8 * t + 2 * k, p + 3 + k);
    }
    CU(cudaMalloc(&c->d_tw16, sizeof(double2) * kTw16Len));
    CU(cudaMemcpy(c->d_tw16, t16.data(), sizeof(double2) * kTw16Len, cudaMemcpyHostToDevice));
  }
  CU(cudaMalloc(&c->d_err, sizeof(int)));
  CU(cudaMemset(c->d_err, 0, sizeof(int)));
  TRY(c->scratch.ensure((size_t)c->sm_count * 2 * c->ct_stride() * sizeof(int)));
  for (int v = 0; v < 2; v++) {
    // how many clusters of k_ks8 fit at once (GPC granularity): the launch rule keeps such launches to one wave
    const int cl = v == 0 ? 8 : 4;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(cl * 64); cfg.blockDim = dim3(512); cfg.dynamicSmemBytes = ks8_smem(cl);
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeClusterDimension;
    at.val.clusterDim.x = cl; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
    cfg.attrs = &at; cfg.numAttrs = 1;
    int n = 0;
    const cudaError_t e = v == 0 ? cudaOccupancyMaxActiveClusters(&n, k_ks8<8, MODE_TRACE>, &cfg)
                                 : cudaOccupancyMaxActiveClusters(&n, k_ks8<4, MODE_TRACE>, &cfg);
    if (e != cudaSuccess) { n = 0; (void)cudaGetLastError(); }
    const int cap = (int)(c->scratch.bytes / (kKs8ScratchWords * sizeof(unsigned long long)));
    c->ks8_clusters[v] = n < cap ? n : cap;
    cfg.dynamicSmemBytes = ext9_smem(cl);
    n = 0;
    const cudaError_t e2 = v == 0 ? cudaOccupancyMaxActiveClusters(&n, k_ext9<8>, &cfg)
                                  : cudaOccupancyMaxActiveClusters(&n, k_ext9<4>, &cfg);
    if (e2 != cudaSuccess) { n = 0; (void)cudaGetLastError(); }
    c->ext9_clusters[v] = n < cap ? n : cap;
  }
  *out = c;
  return 0;
}

static void wipe_secrets(fheram_ctx* c);
extern "C" int fheram_ctx_destroy(fheram_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  wipe_secrets(c);
  cudaStreamSynchronize(c->stream);
  if (c->comm_prep) { ncclCommDestroy(c->comm_prep); c->comm_prep = nullptr; }
  if (c->comm) { ncclCommDestroy(c->comm); c->comm = nullptr; }
  c->stage64.release(); c->scratch.release();
  for (auto& b : c->opbuf) b.release();
  for (auto& b : c->enc_buf) b.release();
  cudaFree(c->d_tw); cudaFree(c->d_tw16); cudaFree(c->d_err);
  if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
  if (c->side) {
    cudaStreamSynchronize(c->side); cudaStreamDestroy(c->side);
    cudaEventDestroy(c->side_fork); cudaEventDestroy(c->side_join);
  }
  c->scratch_side.release();
  if (c->pin32) cudaFreeHost(c->pin32);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
  return 0;
}
extern "C" int fheram_ctx_synchronize(fheram_ctx* c) {
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}
extern "C" void* fheram_ctx_stream(fheram_ctx* c) { return (void*)c->stream; }
extern "C" uint64_t fheram_ctx_launch_count(const fheram_ctx* c) { return c->launches; }

// ---- multi-GPU communicator (one rank per context) --------------------------------------
// Rank 0 draws the id and hands it to the other ranks out of band (MPI_Bcast, a TCP store, a file: 128 bytes);
// every rank then calls fheram_comm_init on its own context.  After that the calls on a RAM created with
// fheram_ram_create_sharded(ctx, rank, n_ranks) do their own exchange steps (all-to-all of packed partials for reads,
// all-gather for read_prepare_write, broadcast of the written word for write), all on the context's stream.
extern "C" int fheram_comm_unique_id(uint8_t id[128]) {
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  if (!id) return fail(FHERAM_ERR_INVALID, "null argument");
  ncclUniqueId u;
  NC(ncclGetUniqueId(&u));
  memcpy(id, &u, sizeof(u));
  return 0;
}
extern "C" int fheram_comm_init(fheram_ctx* c, int n_ranks, int rank, const uint8_t id[128]) {
  if (!c || !id || n_ranks < 1 || rank < 0 || rank >= n_ranks || (n_ranks & (n_ranks - 1)))
    return fail(FHERAM_ERR_INVALID, "n_ranks must be a power of two and 0 <= rank < n_ranks");
  if (c->comm) return fail(FHERAM_ERR_INVALID, "communicator already initialised");
  CU(cudaSetDevice(c->device));
  ncclUniqueId u;
  memcpy(&u, id, sizeof(u));
  NC(ncclCommInitRank(&c->comm, n_ranks, u, rank));
  // collectives of one communicator must not run concurrently: the upload pipeline gets its own
  NC(ncclCommSplit(c->comm, 0, rank, &c->comm_prep, nullptr));
  c->n_ranks = n_ranks; c->rank = rank;
  return 0;
}
extern "C" int fheram_comm_destroy(fheram_ctx* c) {
  if (!c) return 0;
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  if (c->comm_prep) NC(ncclCommDestroy(c->comm_prep));
  if (c->comm) NC(ncclCommDestroy(c->comm));
  c->comm = nullptr; c->comm_prep = nullptr; c->n_ranks = 1; c->rank = 0;
  return 0;
}
extern "C" int fheram_comm_n_ranks(const fheram_ctx* c) { return c ? c->n_ranks : 0; }
extern "C" int fheram_comm_rank(const fheram_ctx* c) { return c ? c->rank : -1; }
// all-to-all of equal blocks (count ints each) on the context stream: block r of `send` goes to rank r, block r of
// `recv` comes from rank r.  Integer limbs only: never a floating-point reduction (SURVEY.md 7, 8e).
static int all_to_all_i32(fheram_ctx* c, const int* send, int* recv, size_t count) {
  NC(ncclGroupStart());
  for (int r = 0; r < c->n_ranks; r++) {
    NC(ncclSend(send + (size_t)r * count, count, ncclInt32, r, c->comm, c->stream));
    NC(ncclRecv(recv + (size_t)r * count, count, ncclInt32, r, c->comm, c->stream));
  }
  NC(ncclGroupEnd());
  return 0;
}
// a sharded RAM can run its own exchange steps when its shard layout is the communicator's
static bool comm_matches(const fheram_ctx* c, int shard, int n_shards) {
  return c->comm && c->n_ranks == n_shards && c->rank == shard;
}

// ---- measurement helpers ----------------------------------------------------------------
extern "C" int fheram_ctx_profile(fheram_ctx* c, int enable) {
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  c->profile = enable != 0;
  c->ev_recs.clear();
  c->ev_used = 0;
  return 0;
}
// per class (0 ext chain, 1 trace/key-switch chain, 2 two-sided combine, 3 other):
// ms[c] = summed device time, launches[c], ops[c] = sum over launches of items*steps
extern "C" int fheram_ctx_profile_get(fheram_ctx* c, double ms[4], uint64_t launches[4], uint64_t ops[4]) {
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  for (int i = 0; i < 4; i++) { ms[i] = 0; launches[i] = 0; ops[i] = 0; }
  for (auto& r : c->ev_recs) {
    float t = 0;
    CU(cudaEventElapsedTime(&t, c->ev_pool[r.e0], c->ev_pool[r.e1]));
    ms[r.cls] += t; launches[r.cls]++; ops[r.cls] += r.items * r.steps;
  }
  return 0;
}

// per-launch records of the profiled region, in launch order; returns the number of records
extern "C" int fheram_ctx_profile_records(fheram_ctx* c, int max_n, int* cls, double* ms, uint64_t* items,
                                          uint64_t* steps) {
  if (cudaSetDevice(c->device) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess) return -1;
  int n = 0;
  for (auto& r : c->ev_recs) {
    if (n >= max_n) break;
    float t = 0;
    cudaEventElapsedTime(&t, c->ev_pool[r.e0], c->ev_pool[r.e1]);
    cls[n] = r.cls; ms[n] = t; items[n] = r.items; steps[n] = r.steps;
    n++;
  }
  return n;
}

__global__ void k_fp64_probe(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, b = 1e-7;
#pragma unroll 1
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < 8; u++) {
      a0 = fma(a0, m, b); a1 = fma(a1, m, b); a2 = fma(a2, m, b); a3 = fma(a3, m, b);
      a4 = fma(a4, m, b); a5 = fma(a5, m, b); a6 = fma(a6, m, b); a7 = fma(a7, m, b);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}
// FP64 FMA-pipe peak of this GPU (MEASURED_PEAKS.json has no FP64 entry): best of `reps`
extern "C" int fheram_fp64_peak_probe(fheram_ctx* c, int reps, double* tflops) {
  CU(cudaSetDevice(c->device));
  const int blocks = c->sm_count * 4, threads = 512, iters = 4096;
  double* d = nullptr;
  CU(cudaMalloc(&d, sizeof(double) * blocks * threads));
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  double best = 0;
  for (int r = 0; r < reps + 1; r++) {
    CU(cudaEventRecord(e0, c->stream));
    k_fp64_probe<<<blocks, threads, 0, c->stream>>>(d, iters);
    CU(cudaEventRecord(e1, c->stream));
    CU(cudaEventSynchronize(e1));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    double tf = (double)blocks * threads * iters * 64 * 2 / (ms * 1e-3) / 1e12;
    if (r > 0 && tf > best) best = tf;
  }
  CU(cudaEventDestroy(e0)); CU(cudaEventDestroy(e1));
  CU(cudaFree(d));
  *tflops = best;
  return 0;
}
// debug: enable (1) / read-and-disable (0) per-phase cycle counters of the vmp kernels; out[8] =
// cycles summed over CTAs for phases {prologue, fwd pass 1, fwd warp passes, contraction, inverse,
// epilogue, rest, unused}
extern "C" int fheram_debug_phase_cycles(fheram_ctx* c, int enable, long long out[8]) {
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  const size_t n = (size_t)c->sm_count * 2 * 8;
  if (enable) {
    if (!c->d_phase) CU(cudaMalloc(&c->d_phase, sizeof(long long) * n));
    CU(cudaMemset(c->d_phase, 0, sizeof(long long) * n));
    return 0;
  }
  if (!c->d_phase) return fail(FHERAM_ERR_INVALID, "phase counters not enabled");
  std::vector<long long> h(n);
  CU(cudaMemcpy(h.data(), c->d_phase, sizeof(long long) * n, cudaMemcpyDeviceToHost));
  for (int i = 0; i < 8; i++) out[i] = 0;
  for (size_t i = 0; i < n; i++) out[i % 8] += h[i];
  CU(cudaFree(c->d_phase));
  c->d_phase = nullptr;
  return 0;
}
extern "C" int fheram_host_register(void* p, size_t bytes) {
  CU(cudaHostRegister(p, bytes, cudaHostRegisterDefault));
  return 0;
}
extern "C" int fheram_host_unregister(void* p) {
  CU(cudaHostUnregister(p));
  return 0;
}

// --------------------------------------------------------------------------------------
// host <-> device limb conversion
// --------------------------------------------------------------------------------------
// packed host format (fheram_pack17): limb i = bits [17 i, 17 i + 17) of a little-endian stream, two's complement
__global__ void k_unpack17(const uint32_t* __restrict__ in, int* __restrict__ out, size_t n) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    const size_t bit = 17 * i, w = bit >> 5;
    const unsigned sh = (unsigned)(bit & 31);
    unsigned long long two = in[w];
    if (sh > 15) two |= (unsigned long long)in[w + 1] << 32;
    const uint32_t f = (uint32_t)(two >> sh) & 0x1ffffu;
    out[i] = (int)(f << 15) >> 15;
  }
}
static int upload_i64(fheram_ctx* c, const int64_t* h, size_t n, int* d_out) {
  const size_t chunk = (size_t)64 << 20;  // limbs per staging pass (512 MiB of int64)
  for (size_t off = 0; off < n; off += chunk) {
    size_t m = n - off < chunk ? n - off : chunk;
    TRY(c->stage64.ensure(m * sizeof(int64_t)));
    CU(cudaMemcpyAsync(c->stage64.p, h + off, m * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    k_i64_to_i32<<<c->sm_count * 8, 256, 0, c->stream>>>((const long long*)c->stage64.p, d_out + off, m, c->d_err);
    c->launches++;
    CU(cudaStreamSynchronize(c->stream));
  }
  int err = 0;
  CU(cudaMemcpy(&err, c->d_err, sizeof(int), cudaMemcpyDeviceToHost));
  if (err) {
    CU(cudaMemset(c->d_err, 0, sizeof(int)));
    return fail(FHERAM_ERR_RANGE, "limb outside +-2^30: ciphertext limbs must be (nearly) normalised");
  }
  return 0;
}
static int download_i64(fheram_ctx* c, const int* d_in, size_t n, int64_t* h) {
  if (n <= kSmallDownload) {
    // results of single operations (word_size GLWEs): int32 limbs by DMA into a pinned buffer of the context, widened by
    // the host -- half the bytes over PCIe, no conversion kernel, no staging copy out of pageable memory by the driver
    if (!c->pin32) CU(cudaMallocHost(&c->pin32, kSmallDownload * sizeof(int)));
    CU(cudaMemcpyAsync(c->pin32, d_in, n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    const int* p = c->pin32;
    for (size_t i = 0; i < n; i++) h[i] = p[i];
    return 0;
  }
  const size_t chunk = (size_t)64 << 20;
  for (size_t off = 0; off < n; off += chunk) {
    size_t m = n - off < chunk ? n - off : chunk;
    TRY(c->stage64.ensure(m * sizeof(int64_t)));
    k_i32_to_i64<<<c->sm_count * 8, 256, 0, c->stream>>>(d_in + off, (long long*)c->stage64.p, m);
    c->launches++;
    CU(cudaMemcpyAsync(h + off, c->stage64.p, m * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
  }
  return 0;
}
extern "C" int fheram_download_glwe(fheram_ctx* c, const int32_t* d_in, int n_glwe, int64_t* out) {
  CU(cudaSetDevice(c->device));
  return download_i64(c, d_in, (size_t)n_glwe * c->ct_stride(), out);
}

// --------------------------------------------------------------------------------------
// launches
// --------------------------------------------------------------------------------------
static VmpArgs base_args(fheram_ctx* c, int n_items, const int* src, int* dst, long ct_stride) {
  VmpArgs a;
  memset(&a, 0, sizeof(a));
  a.n_items = n_items;
  a.src = src; a.dst = dst;
  a.ct_stride = ct_stride;
  a.scratch = (int*)(c->on_side ? c->scratch_side.p : c->scratch.p);
  a.sign = 1;
  for (int i = 0; i < kMaxSteps; i++) { a.gal[i] = 1; a.gal_inv[i] = 1; }
  a.tw = c->tw;
  a.phase_cycles = c->d_phase;
  {
    static int stagger = -1;
    if (stagger < 0) { const char* e = getenv("FHERAM_STAGGER"); stagger = e ? atoi(e) : 0; }
    a.stagger = stagger;
  }
  return a;
}
static size_t prof_event(fheram_ctx* c) {
  if (c->ev_used == c->ev_pool.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    c->ev_pool.push_back(e);
  }
  cudaEventRecord(c->ev_pool[c->ev_used], c->stream);
  return c->ev_used++;
}
enum KClass { KC_EXT = 0, KC_TRACE = 1, KC_COMBINE2 = 2, KC_OTHER = 3, KC_COUNT = 4 };
// one kernel launch on c->stream over a.n_items operations, timed per class `cls` when profiling
template <typename K, typename... X>
static int launch(fheram_ctx* c, int cls, K kernel, int grid, int block, size_t smem, const VmpArgs& a, X... extra) {
  if (a.n_items <= 0) return 0;
  size_t e0 = 0;
  if (c->profile) e0 = prof_event(c);
  kernel<<<grid, block, smem, c->stream>>>(a, extra...);
  if (c->profile) {
    size_t e1 = prof_event(c);
    c->ev_recs.push_back({cls, e0, e1, (uint64_t)a.n_items, (uint64_t)a.n_steps});
  }
  c->launches++;
  CU(cudaGetLastError());
  return 0;
}

// ---- the launch-width rule (DESIGN.md 3.4): the kernel of a launch of n operations -----------------
enum Kernel { KN_EXT9_8, KN_EXT9_4, KN_EXT8, KN_KS8_8, KN_KS8_4, KN_KS7, KN_KS6, KN_KS5, KN_KS4, KN_NONE };
// external-product chains: one chain per cluster of eight (four) SMs while one wave of clusters holds the launch
// (kernels_ext9.cuh), else one ciphertext per SM (kernels_ext8.cuh)
static Kernel select_ext(const fheram_ctx* c, int n) {
  const int e8 = c->ext9_clusters[0], e4 = c->ext9_clusters[1];
  if (c->force_ext == FORCE_EXT8) return KN_EXT8;
  if (c->force_ext == FORCE_EXT9C4 && e4 > 0) return KN_EXT9_4;
  if (c->force_ext == FORCE_EXT9 && n > e8 && e4 > 0) return KN_EXT9_4;
  if (n <= e8) return KN_EXT9_8;
  if (n <= e4) return KN_EXT9_4;
  return KN_EXT8;
}
// the k_ks8 rows, shared by trace and combine launches (one chain per cluster of eight or four SMs, kernels_ks8.cuh)
static Kernel select_ks8(const fheram_ctx* c, int n) {
  const int cap8 = c->ks8_clusters[0], cap4 = c->ks8_clusters[1];
  if (c->force_ks == FORCE_KS8C4 && cap4 > 0) return KN_KS8_4;
  if (n <= cap8) return KN_KS8_8;
  if (n <= cap4) return KN_KS8_4;
  if (c->force_ks == FORCE_KS8 && cap4 > 0) return KN_KS8_4;
  if (c->force_ks == FORCE_KS8 && cap8 > 0) return KN_KS8_8;
  return KN_NONE;
}
// trace chains and one-sided packer levels: wide launches on k_ks7 (two CTAs per SM), narrow ones on the two-SM
// cluster kernel k_ks6 or the one-SM kernel k_ks5
static Kernel select_trace(const fheram_ctx* c, int n) {
  const int S = c->sm_count;
  if (c->force_ks == FORCE_KS7) return KN_KS7;
  if (c->force_ks == FORCE_KS5) return KN_KS5;
  if (c->force_ks == FORCE_KS6 && 2 * n <= S) return KN_KS6;  // k_ks6's per-CTA scratch holds 2 S ciphertexts
  if (const Kernel k = select_ks8(c, n); k != KN_NONE) return k;
  if (n > S) return KN_KS7;
  return 2 * n <= S ? KN_KS6 : KN_KS5;
}
// two-sided combines: as the trace, with k_ks4 (two CTAs per SM) for the wide launches
static Kernel select_combine(const fheram_ctx* c, int n) {
  const int S = c->sm_count;
  if (c->force_ks == FORCE_KS4) return KN_KS4;
  if (c->force_ks == FORCE_KS5) return KN_KS5;
  if (c->force_ks == FORCE_KS6 && 2 * n <= S) return KN_KS6;
  if (const Kernel k = select_ks8(c, n); k != KN_NONE) return k;
  if (2 * n <= S) return KN_KS6;
  return n <= S ? KN_KS5 : KN_KS4;
}
// vmp_prepare of n_mat matrices
static int inv_mod_2n(int g) {  // g odd, modulus 2N = 8192: g^(N-1) since the unit group has exponent N
  long r = 1, b = ((g % (2 * kN)) + 2 * kN) % (2 * kN);
  for (int e = kN - 1; e; e >>= 1) { if (e & 1) r = r * b % (2 * kN); b = b * b % (2 * kN); }
  return (int)r;
}
// vmp_prepare of n_mat matrices; gal != 1 prepares phi_gal(matrix) (key-switch keys, see k_vmp);
// order7: frequency order of the 16-point transform (k_prepare7: consumers k_ks7 / k_ks8 / k_ext8 / k_ext9)
static int prepare(fheram_ctx* c, const int* raw, long raw_stride, double2* out, long out_stride,
                   int n_mat, int rows, int cin, int lout, int gal = 1, bool order7 = false,
                   cudaStream_t stream = nullptr) {
  if (!stream) stream = c->stream;
  PrepArgs a;
  a.raw = raw; a.out = out; a.raw_stride = raw_stride; a.out_stride = out_stride;
  a.rows = rows; a.cin = cin; a.lout = lout; a.tw = c->tw;
  a.gal_inv = inv_mod_2n(gal);
  if (order7) {
    Prep7Args pa;
    pa.p = a; pa.tw16 = c->d_tw16;
    pa.n_polys = n_mat * rows * cin * 2 * lout;
    k_prepare7<<<(pa.n_polys + 1) / 2, 256, kPrep7Smem, stream>>>(pa);
  } else {
    int grid = n_mat * rows * cin * 2 * lout;
    k_prepare<<<grid, kThreads, 0, stream>>>(a);
  }
  c->launches++;
  CU(cudaGetLastError());
  return 0;
}
// CoordinatePrepared::prepare (src/coordinate_prepared.rs:104-116) of n_mat GGSWs, in the frequency order of the
// external-product kernels (k_prepare7)
static int prepare_ggsw(fheram_ctx* c, const int* raw, double2* out, int n_mat) {
  return prepare(c, raw, c->ggsw_raw_len(), out, c->ggsw_prep_len(), n_mat, c->d.dnum_ct, 2, c->d.size_addr, 1, true);
}

// --------------------------------------------------------------------------------------
// keys
// --------------------------------------------------------------------------------------
struct fheram_keys {
  fheram_ctx* c;
  double2* atk = nullptr;      // [log_n] prepared trace keys
  double2* atk7 = nullptr;     // trace keys prepared in the frequency order of k_ks7 / k_ks8 (k_prepare7)
  double2* atk_inv = nullptr;  // prepared atk_ggsw_inv
  double2* tsk = nullptr;      // prepared tsk_ggsw_inv
  int* raw = nullptr;          // fheram_keys_encrypt_sk: the raw keys [atk x log_n | tsk | atk_inv] (fheram_keys_download_raw)
};

// EvaluationKeysPrepared::prepare (src/keys.rs:57-71) from raw int32 keys already on the device:
// d_atk = [log_n] trace keys, d_tsk, d_inv (layouts of include/fheram.h)
static int keys_prepare_device(fheram_ctx* c, const int* d_atk, const int* d_tsk, const int* d_inv, fheram_keys* k) {
  const Derived& d = c->d;
  const size_t atk_raw = (size_t)d.dnum_ct * 2 * d.size_evk_trace * d.n;
  const size_t inv_raw = (size_t)d.dnum_ggsw * 2 * d.size_evk_inv * d.n;
  CU(cudaMalloc(&k->atk, sizeof(double2) * c->atk_prep_len() * d.log_n));
  CU(cudaMalloc(&k->atk7, sizeof(double2) * c->atk_prep_len() * d.log_n));
  CU(cudaMalloc(&k->atk_inv, sizeof(double2) * c->evk_inv_prep_len()));
  CU(cudaMalloc(&k->tsk, sizeof(double2) * c->evk_inv_prep_len()));
  // trace key i is stored as phi_{g_i}(key): the kernels transform phi_g(x) and get phi_g(KS(x)); once per
  // transform family (frequency orders of k_prepare and k_prepare7)
  for (int i = 0; i < d.log_n; i++) {
    const int gal = (int)((galois(d.log_n, i) + 2 * kN) % (2 * kN));
    TRY(prepare(c, d_atk + (size_t)i * atk_raw, (long)atk_raw, k->atk + (size_t)i * c->atk_prep_len(),
                c->atk_prep_len(), 1, d.dnum_ct, 1, d.size_evk_trace, gal));
    TRY(prepare(c, d_atk + (size_t)i * atk_raw, (long)atk_raw, k->atk7 + (size_t)i * c->atk_prep_len(),
                c->atk_prep_len(), 1, d.dnum_ct, 1, d.size_evk_trace, gal, true));
  }
  TRY(prepare(c, d_inv, (long)inv_raw, k->atk_inv, c->evk_inv_prep_len(), 1, d.dnum_ggsw, 1, d.size_evk_inv, 2 * kN - 1));
  TRY(prepare(c, d_tsk, (long)inv_raw, k->tsk, c->evk_inv_prep_len(), 1, d.dnum_ggsw, 1, d.size_evk_inv));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" int fheram_keys_prepare(fheram_ctx* c, const int64_t* atk_glwe, const int64_t* tsk,
                                   const int64_t* atk_inv, fheram_keys** out) {  // src/keys.rs:34-71
  if (!c || !atk_glwe || !tsk || !atk_inv || !out) return fail(FHERAM_ERR_INVALID, "null argument");
  CU(cudaSetDevice(c->device));
  const Derived& d = c->d;
  fheram_keys* k = new fheram_keys();
  k->c = c;
  const size_t atk_raw = (size_t)d.dnum_ct * 2 * d.size_evk_trace * d.n;
  const size_t inv_raw = (size_t)d.dnum_ggsw * 2 * d.size_evk_inv * d.n;
  int* tmp = nullptr;
  CU(cudaMalloc(&tmp, sizeof(int) * (atk_raw * d.log_n + 2 * inv_raw)));
  int *d_atk = tmp, *d_tsk = tmp + atk_raw * d.log_n, *d_inv = d_tsk + inv_raw;
  TRY(upload_i64(c, atk_glwe, atk_raw * d.log_n, d_atk));
  TRY(upload_i64(c, tsk, inv_raw, d_tsk));
  TRY(upload_i64(c, atk_inv, inv_raw, d_inv));
  TRY(keys_prepare_device(c, d_atk, d_tsk, d_inv, k));
  CU(cudaFree(tmp));
  *out = k;
  return 0;
}

extern "C" int fheram_keys_destroy(fheram_keys* k) {
  if (!k) return 0;
  cudaSetDevice(k->c->device);
  cudaFree(k->atk); cudaFree(k->atk7); cudaFree(k->atk_inv); cudaFree(k->tsk); cudaFree(k->raw);
  delete k;
  return 0;
}

// --------------------------------------------------------------------------------------
// addresses
// --------------------------------------------------------------------------------------
struct fheram_address {
  fheram_ctx* c;
  int count = 0;
  int* raw = nullptr;        // [count][n_ggsw] raw GGSW, int32
  double2* prep = nullptr;   // [count][n_ggsw] prepared GGSW
  // split layout of the sharded host pipeline (prep1 != nullptr): prep = [count][coord_len[0]] prepared GGSWs of the
  // first coordinate (every rank needs them for its local stage: all-gathered), prep1 = [own reads][coord_len[1]] of
  // the second coordinate, which only the finishing rank needs (address `prep1_first` of the set is its entry 0)
  double2* prep1 = nullptr;
  int prep1_first = 0;
  // CoordinatePrepared::prepare_inv of every digit (src/ram.rs:260-271,278-289): a cache of the address handle,
  // built by read_prepare_write (off the critical path of the write that follows) or lazily by write
  mutable int* inv_raw = nullptr;    // [n_ggsw] GGSW(X^+digit)
  mutable double2* inv_prep = nullptr;
  mutable bool inv_ready = false;
  // asynchronous slice upload (multi-GPU host-buffer pipeline): int64 staging, copy-stream events
  long long* stage = nullptr;
  size_t stage_cap = 0;
  cudaEvent_t uploaded = nullptr, released = nullptr;
  bool released_valid = false;
};

extern "C" int fheram_address_load_batch(fheram_ctx* c, const int64_t* ggsw, int n, fheram_address** out) {
  if (!c || !ggsw || !out || n < 1) return fail(FHERAM_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  const Derived& d = c->d;
  fheram_address* a = new fheram_address();
  a->c = c; a->count = n;
  const size_t nm = (size_t)n * d.n_ggsw;
  CU(cudaMalloc(&a->raw, sizeof(int) * nm * c->ggsw_raw_len()));
  CU(cudaMalloc(&a->prep, sizeof(double2) * nm * c->ggsw_prep_len()));
  TRY(upload_i64(c, ggsw, nm * c->ggsw_raw_len(), a->raw));
  // CoordinatePrepared::prepare, src/coordinate_prepared.rs:104-116
  TRY(prepare_ggsw(c, a->raw, a->prep, (int)nm));
  CU(cudaStreamSynchronize(c->stream));
  *out = a;
  return 0;
}
// Multi-GPU upload path: allocate n addresses, fill slices of the raw limbs (host upload of this
// rank's share, NVLink all-gather of the rest straight into fheram_address_raw_ptr), then prepare.
extern "C" int fheram_address_alloc(fheram_ctx* c, int n, fheram_address** out) {
  if (!c || !out || n < 1) return fail(FHERAM_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  fheram_address* a = new fheram_address();
  a->c = c; a->count = n;
  const size_t nm = (size_t)n * c->d.n_ggsw;
  CU(cudaMalloc(&a->raw, sizeof(int) * nm * c->ggsw_raw_len()));
  CU(cudaMalloc(&a->prep, sizeof(double2) * nm * c->ggsw_prep_len()));
  *out = a;
  return 0;
}
extern "C" int32_t* fheram_address_raw_ptr(fheram_address* a) { return a ? a->raw : nullptr; }
extern "C" int fheram_address_upload_slice(fheram_address* a, const int64_t* ggsw, int first, int count) {
  if (!a || !ggsw || first < 0 || count < 1 || first + count > a->count) return fail(FHERAM_ERR_INVALID, "bad slice");
  fheram_ctx* c = a->c;
  CU(cudaSetDevice(c->device));
  const size_t per = (size_t)c->d.n_ggsw * c->ggsw_raw_len();
  a->inv_ready = false;
  return upload_i64(c, ggsw, (size_t)count * per, a->raw + (size_t)first * per);
}
// Asynchronous variant for pipelines: host -> device copy and int64 -> int32 conversion run on the
// context's copy stream; fheram_address_wait_upload makes the compute stream wait for them, and
// fheram_address_release (recorded on the compute stream once the reads that use this address set
// have been issued) lets the next upload into the same set start as soon as they are done.
extern "C" int fheram_address_upload_slice_async(fheram_address* a, const int64_t* ggsw, int first, int count) {
  if (!a || !ggsw || first < 0 || count < 1 || first + count > a->count) return fail(FHERAM_ERR_INVALID, "bad slice");
  fheram_ctx* c = a->c;
  CU(cudaSetDevice(c->device));
  if (!c->copy_stream) CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  const size_t per = (size_t)c->d.n_ggsw * c->ggsw_raw_len();
  const size_t n = (size_t)count * per;
  if (a->stage_cap < n) {
    CU(cudaStreamSynchronize(c->copy_stream));
    cudaFree(a->stage);
    a->stage = nullptr; a->stage_cap = 0;
    CU(cudaMalloc(&a->stage, sizeof(long long) * n));
    a->stage_cap = n;
  }
  a->inv_ready = false;
  if (!a->uploaded) CU(cudaEventCreateWithFlags(&a->uploaded, cudaEventDisableTiming));
  if (a->released_valid) CU(cudaStreamWaitEvent(c->copy_stream, a->released, 0));
  CU(cudaMemcpyAsync(a->stage, ggsw, sizeof(long long) * n, cudaMemcpyHostToDevice, c->copy_stream));
  k_i64_to_i32<<<c->sm_count * 8, 256, 0, c->copy_stream>>>(a->stage, a->raw + (size_t)first * per, n, c->d_err);
  c->launches++;
  CU(cudaGetLastError());
  CU(cudaEventRecord(a->uploaded, c->copy_stream));
  return 0;
}
extern "C" int fheram_address_wait_upload(fheram_address* a) {
  if (!a || !a->uploaded) return fail(FHERAM_ERR_INVALID, "no upload in flight");
  CU(cudaSetDevice(a->c->device));
  CU(cudaStreamWaitEvent(a->c->stream, a->uploaded, 0));
  return 0;
}
extern "C" int fheram_address_release(fheram_address* a) {
  if (!a) return fail(FHERAM_ERR_INVALID, "null argument");
  CU(cudaSetDevice(a->c->device));
  if (!a->released) CU(cudaEventCreateWithFlags(&a->released, cudaEventDisableTiming));
  CU(cudaEventRecord(a->released, a->c->stream));
  a->released_valid = true;
  return 0;
}
extern "C" int fheram_address_prepare(fheram_address* a) {  // CoordinatePrepared::prepare for every address
  if (!a) return fail(FHERAM_ERR_INVALID, "null argument");
  fheram_ctx* c = a->c;
  CU(cudaSetDevice(c->device));
  return prepare_ggsw(c, a->raw, a->prep, a->count * c->d.n_ggsw);
}
extern "C" int fheram_address_load(fheram_ctx* c, const int64_t* ggsw, fheram_address** out) {
  return fheram_address_load_batch(c, ggsw, 1, out);
}
extern "C" int fheram_address_count(const fheram_address* a) { return a ? a->count : 0; }
extern "C" int fheram_address_destroy(fheram_address* a) {
  if (!a) return 0;
  cudaSetDevice(a->c->device);
  if (a->c->copy_stream) cudaStreamSynchronize(a->c->copy_stream);
  cudaFree(a->raw); cudaFree(a->prep); cudaFree(a->inv_raw); cudaFree(a->inv_prep); cudaFree(a->stage);
  if (a->uploaded) cudaEventDestroy(a->uploaded);
  if (a->released) cudaEventDestroy(a->released);
  delete a;
  return 0;
}

// --------------------------------------------------------------------------------------
// schedule building blocks (all asynchronous on c->stream, device buffers only)
// --------------------------------------------------------------------------------------
// CoordinatePrepared::product[_inplace] (src/coordinate_prepared.rs:147-177): chain of n_dig
// external products; matrices mats + dig*ggsw_prep_len (+ (item / mat_div) * mat_stride).
static int run_ext_chain(fheram_ctx* c, int n_items, const int* src, const int* src_map, int src_mod,
                         int* dst, const double2* mats, int n_dig, int mat_div, long mat_stride) {
  VmpArgs a = base_args(c, n_items, src, dst, c->ct_stride());
  a.src_map = src_map; a.src_mod = src_mod;
  a.n_steps = n_dig;
  for (int s = 0; s < n_dig; s++) a.mat[s] = mats + (size_t)s * c->ggsw_prep_len();
  a.mat_div = mat_div; a.mat_stride = mat_stride;
  switch (select_ext(c, n_items)) {
    case KN_EXT9_8:
      return launch(c, KC_EXT, k_ext9<8>, 8 * std::min(n_items, c->ext9_clusters[0]), 512, ext9_smem(8), a, c->d_tw16);
    case KN_EXT9_4:
      return launch(c, KC_EXT, k_ext9<4>, 4 * std::min(n_items, c->ext9_clusters[1]), 512, ext9_smem(4), a, c->d_tw16);
    default:
      return launch(c, KC_EXT, k_ext8, std::min(n_items, c->sm_count), kExt8Threads, kExt8Smem, a, c->d_tw16);
  }
}
// a key-switch launch of MODE_TRACE or MODE_COMBINE2: step s uses trace key key0 + s, in the frequency order of the
// selected kernel (k_ks7 and k_ks8 read the keys prepared by k_prepare7, the others those of k_prepare)
template <int MODE>
static int launch_ks(fheram_ctx* c, const fheram_keys* k, int key0, VmpArgs a) {
  const int n = a.n_items, S = c->sm_count, cls = MODE == MODE_TRACE ? KC_TRACE : KC_COMBINE2;
  const Kernel kn = MODE == MODE_TRACE ? select_trace(c, n) : select_combine(c, n);
  const double2* keys = (kn == KN_KS7 || kn == KN_KS8_8 || kn == KN_KS8_4) ? k->atk7 : k->atk;
  for (int s = 0; s < a.n_steps; s++) a.mat[s] = keys + (size_t)(key0 + s) * c->atk_prep_len();
  switch (kn) {
    case KN_KS8_8:
      return launch(c, cls, k_ks8<8, MODE>, 8 * std::min(n, c->ks8_clusters[0]), 512, ks8_smem(8), a, c->d_tw16);
    case KN_KS8_4:
      return launch(c, cls, k_ks8<4, MODE>, 4 * std::min(n, c->ks8_clusters[1]), 512, ks8_smem(4), a, c->d_tw16);
    case KN_KS7: return launch(c, cls, k_ks7, std::min(n, 2 * S), 256, kKs7Smem, a, c->d_tw16);
    case KN_KS6: return launch(c, cls, k_ks6<MODE>, 2 * n, kThreads5, kKs5Smem, a);
    case KN_KS5: return launch(c, cls, k_ks5<MODE>, std::min(n, S), kThreads5, kKs5Smem, a);
    default: return launch(c, cls, k_ks4, std::min(n, 2 * S), kThreads, kKs4Smem, a);
  }
}
// chain of { glwe_rsh(1); automorphism_add with trace key i } for i in [g0, g1)
// (glwe_trace_inplace, and the one-sided levels of GLWEPacker::combine)
static int run_trace_chain(fheram_ctx* c, const fheram_keys* k, int n_items, const int* src,
                           const int* src_map, int src_mod, int src_div, int* dst, int g0, int g1,
                           int rot_mod = 0, int rot_mul = 0, int rot_const = 0, int sign = 1) {
  VmpArgs a = base_args(c, n_items, src, dst, c->ct_stride());
  a.src_map = src_map; a.src_mod = src_mod; a.src_div = src_div;
  a.n_steps = g1 - g0;
  for (int s = 0; s < a.n_steps; s++) {
    a.gal[s] = (int)((galois(c->d.log_n, g0 + s) + 2 * kN) % (2 * kN));
    a.gal_inv[s] = inv_mod_2n(a.gal[s]);
  }
  a.rot_mod = rot_mod; a.rot_mul = rot_mul; a.rot_const = rot_const; a.sign = sign;
  if (a.n_steps == 0) {
    // no level to run (max_addr = N^2: every packer level is two-sided): only the (feed-order) gather remains
    if (!src_map) {
      if (src != dst)
        CU(cudaMemcpyAsync(dst, src, sizeof(int) * (size_t)n_items * c->ct_stride(), cudaMemcpyDeviceToDevice, c->stream));
      return 0;
    }
    k_gather<<<c->sm_count * 8, 256, 0, c->stream>>>(dst, src, src_map, src_mod, n_items, c->ct_stride());
    c->launches++;
    CU(cudaGetLastError());
    return 0;
  }
  return launch_ks<MODE_TRACE>(c, k, g0, a);
}
// GLWEPacker::combine, both operands present, at tree level `level` (0-based absolute):
// in[2i], in[2i+1] -> out[i]
static int run_combine2(fheram_ctx* c, const fheram_keys* k, int n_items, const int* in, int* out, int level) {
  VmpArgs a = base_args(c, n_items, in, out, c->ct_stride());
  a.n_steps = 1;
  a.gal[0] = (int)((galois(c->d.log_n, level) + 2 * kN) % (2 * kN));
  a.gal_inv[0] = inv_mod_2n(a.gal[0]);
  a.rot_const = 1 << (c->d.log_n - level - 1);  // t
  return launch_ks<MODE_COMBINE2>(c, k, level, a);
}

// GLWEPacker over `width` inputs per group (width a power of two), feed order = index order
// of `buf` (caller wrote inputs at m = bitrev(h)).  One-sided levels [0, log_n - log2(width_total))
// must already be applied.  Runs two-sided levels first_level .. first_level + log2(width) - 1,
// ping-ponging between buf and tmp; returns the buffer holding the [groups] results.
static int run_pack_levels(fheram_ctx* c, const fheram_keys* k, int groups, int width, int first_level,
                           int* buf, int* tmp, int** result) {
  int* in = buf;
  int* out = tmp;
  int level = first_level;
  for (int wdt = width; wdt > 1; wdt >>= 1, level++) {
    TRY(run_combine2(c, k, groups * (wdt / 2), in, out, level));
    int* t = in; in = out; out = t;
  }
  *result = in;
  return 0;
}

// --------------------------------------------------------------------------------------
// RAM
// --------------------------------------------------------------------------------------
struct fheram_ram {
  fheram_ctx* c;
  int shard = 0, n_shards = 1;
  int n_local = 0;           // local polynomials per sub-RAM
  int* data = nullptr;       // [word_size][n_local] GLWE   (SubRam::data, src/ram.rs:299)
  int* tree = nullptr;       // [word_size] GLWE            (SubRam::tree[0][0], src/ram.rs:300)
  bool state = false;        // src/ram.rs:302
  bool rotated = false;      // rpw_local_device rotated SubRam::data in place and rpw_finish_device has not completed:
                             // the reference does both inside one call (src/ram.rs:502-533), so no read may see this state
  bool loaded = false;
  int* feed_map = nullptr;   // device: [word_size*n_local] feed position -> data index
  DevBuf bufA, bufB;         // work arenas [B][word_size][n_local] GLWE
  DevBuf partial;            // [B][word_size] packed partials
  DevBuf result;             // [B][word_size] results
  DevBuf wbuf;               // uploaded write words
  DevBuf wstage;             // their int64 staging
  void* wpin = nullptr;      // pinned host copy of the words of the write in flight
  cudaEvent_t wcopied = nullptr;
  DevBuf all;                // results of a chunked batched read
  DevBuf xchg;               // sharded: partials received from the other ranks, [n_shards][reads][word_size]
  DevBuf part_all;           // sharded, device-resident batch: partials of every read before the exchange
  struct HostPipe {          // fheram_ram_read_batch_host: double-buffered upload pipeline
    struct Set { long long* stage = nullptr; fheram_address a; cudaEvent_t copied = nullptr, freed = nullptr; };
    Set sets[2];
    long long* out_stage[2] = {nullptr, nullptr};
    cudaEvent_t out_ready[2] = {nullptr, nullptr}, out_done[2] = {nullptr, nullptr};
    cudaStream_t copy_stream = nullptr, down_stream = nullptr;
    int cap = 0;
  } pipe;
};

static int ram_create(fheram_ctx* c, int shard, int n_shards, fheram_ram** out) {
  if (!c || !out) return fail(FHERAM_ERR_INVALID, "null argument");
  const Derived& d = c->d;
  if (n_shards < 1 || (n_shards & (n_shards - 1)) || n_shards > d.n_glwe || shard < 0 || shard >= n_shards)
    return fail(FHERAM_ERR_INVALID, "n_shards must be a power of two <= max_addr/N and 0 <= shard < n_shards");
  CU(cudaSetDevice(c->device));
  fheram_ram* r = new fheram_ram();
  r->c = c; r->shard = shard; r->n_shards = n_shards;
  r->n_local = d.n_glwe / n_shards;
  const int ws = c->params.word_size;
  CU(cudaMalloc(&r->data, sizeof(int) * (size_t)ws * r->n_local * c->ct_stride()));
  CU(cudaMalloc(&r->tree, sizeof(int) * (size_t)ws * c->ct_stride()));
  CU(cudaMemset(r->tree, 0, sizeof(int) * (size_t)ws * c->ct_stride()));
  // feed order of the packer (src/ram.rs:425-435): position m of the local tree reads local
  // polynomial h' = bitrev(m)
  std::vector<int> map((size_t)ws * r->n_local);
  const int lg = ilog2(r->n_local);
  for (int s = 0; s < ws; s++)
    for (int m = 0; m < r->n_local; m++) map[(size_t)s * r->n_local + m] = s * r->n_local + (int)revbits(m, lg);
  CU(cudaMalloc(&r->feed_map, sizeof(int) * map.size()));
  CU(cudaMemcpy(r->feed_map, map.data(), sizeof(int) * map.size(), cudaMemcpyHostToDevice));
  *out = r;
  return 0;
}
extern "C" int fheram_ram_create(fheram_ctx* c, fheram_ram** out) { return ram_create(c, 0, 1, out); }
extern "C" int fheram_ram_create_sharded(fheram_ctx* c, int shard, int n_shards, fheram_ram** out) {
  return ram_create(c, shard, n_shards, out);
}
extern "C" int fheram_ram_destroy(fheram_ram* r) {
  if (!r) return 0;
  cudaSetDevice(r->c->device);
  cudaFree(r->data); cudaFree(r->tree); cudaFree(r->feed_map);
  if (r->wpin) { cudaStreamSynchronize(r->c->stream); cudaFreeHost(r->wpin); cudaEventDestroy(r->wcopied); }
  r->bufA.release(); r->bufB.release(); r->partial.release(); r->result.release(); r->wbuf.release(); r->wstage.release(); r->all.release(); r->xchg.release(); r->part_all.release();
  for (auto& s : r->pipe.sets) {
    cudaFree(s.stage); cudaFree(s.a.raw); cudaFree(s.a.prep); cudaFree(s.a.prep1);
    s.a.raw = nullptr; s.a.prep = nullptr; s.a.prep1 = nullptr;
    if (s.copied) cudaEventDestroy(s.copied);
    if (s.freed) cudaEventDestroy(s.freed);
  }
  for (int i = 0; i < 2; i++) {
    cudaFree(r->pipe.out_stage[i]);
    if (r->pipe.out_ready[i]) cudaEventDestroy(r->pipe.out_ready[i]);
    if (r->pipe.out_done[i]) cudaEventDestroy(r->pipe.out_done[i]);
  }
  if (r->pipe.copy_stream) cudaStreamDestroy(r->pipe.copy_stream);
  if (r->pipe.down_stream) cudaStreamDestroy(r->pipe.down_stream);
  delete r;
  return 0;
}
// cts: the FULL RAM [word_size][n_glwe]; a sharded RAM keeps h = shard + n_shards*h'
extern "C" int fheram_ram_load(fheram_ram* r, const int64_t* cts) {
  if (!r || !cts) return fail(FHERAM_ERR_INVALID, "null argument");
  fheram_ctx* c = r->c;
  CU(cudaSetDevice(c->device));
  const int ws = c->params.word_size, G = c->d.n_glwe;
  const size_t L = (size_t)c->ct_stride();
  if (r->n_shards == 1) {
    TRY(upload_i64(c, cts, (size_t)ws * G * L, r->data));
  } else {
    // the rank's polynomials (h = shard + n_shards h') of one sub-RAM are gathered on the host and uploaded with one
    // staged copy per sub-RAM (not one synchronous 192 KiB upload per polynomial: 4 096 of them at 2^22 x 4 B)
    std::vector<int64_t> gathered((size_t)r->n_local * L);
    for (int s = 0; s < ws; s++) {
      for (int hp = 0; hp < r->n_local; hp++) {
        const int h = r->shard + r->n_shards * hp;
        memcpy(gathered.data() + (size_t)hp * L, cts + ((size_t)s * G + h) * L, sizeof(int64_t) * L);
      }
      TRY(upload_i64(c, gathered.data(), (size_t)r->n_local * L, r->data + (size_t)s * r->n_local * L));
    }
  }
  r->loaded = true;
  r->state = false;
  r->rotated = false;
  return 0;
}
extern "C" int fheram_ram_store(fheram_ram* r, int64_t* cts) {
  if (!r || !cts) return fail(FHERAM_ERR_INVALID, "null argument");
  fheram_ctx* c = r->c;
  CU(cudaSetDevice(c->device));
  const int ws = c->params.word_size, G = c->d.n_glwe;
  const size_t L = (size_t)c->ct_stride();
  if (r->n_shards == 1) return download_i64(c, r->data, (size_t)ws * G * L, cts);
  for (int s = 0; s < ws; s++)
    for (int hp = 0; hp < r->n_local; hp++) {
      const int h = r->shard + r->n_shards * hp;
      TRY(download_i64(c, r->data + ((size_t)s * r->n_local + hp) * L, L, cts + ((size_t)s * G + h) * L));
    }
  return 0;
}
extern "C" int fheram_ram_tree_store(fheram_ram* r, int64_t* cts) {
  if (!r || !cts) return fail(FHERAM_ERR_INVALID, "null argument");
  CU(cudaSetDevice(r->c->device));
  return download_i64(r->c, r->tree, (size_t)r->c->params.word_size * r->c->ct_stride(), cts);
}
extern "C" int fheram_ram_state(const fheram_ram* r) { return r && r->state ? 1 : 0; }

// --------------------------------------------------------------------------------------
// Bulk secret-key encryption on the device (SURVEY.md 8(f).1): k_glwe_encrypt regenerates the
// mask from the Source's ChaCha20 stream, multiplies by the secret and normalizes; the noise
// is drawn on the host in the order client.cpp draws it.  Limb-for-limb equal to
// fheram_encrypt_ram / fheram_encrypt_address on the same Sources (tests/test_gpu_encrypt.py).
// --------------------------------------------------------------------------------------
struct EncBatch {
  int n_glwe = 0, size = 0, k_noise = 0;
  std::vector<int8_t> pt;                // [n_glwe][N] or empty
  int pt_l = 0, pt_sh = 0;
  std::vector<int> mono;                 // [n_glwe] or empty
  std::vector<short> poly;               // [n_poly][N] or empty (key-switching keys)
  std::vector<int> poly_sel, sk_sel;     // [n_glwe] each, with poly
  std::vector<int> sk_all;               // [n_sk][2 N] secrets the masks are multiplied by (empty: the caller's sk)
  std::vector<int> seq;                  // [n_glwe] position of each GLWE in its stream, or empty (= j % glwe_per_stream)
  std::vector<uint32_t> keys;            // [n_streams][8]
  std::vector<unsigned long long> word0; // [n_streams]
  int glwe_per_stream = 1;
};
// FHERAM_ENC_NOISE=host draws the noise with the host sampler only; default: k_noise_sample + host patches
static bool enc_noise_on_device() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("FHERAM_ENC_NOISE"); v = (e && !strcmp(e, "host")) ? 0 : 1; }
  return v == 1;
}
// widths of the report bands of k_noise_sample (tests widen them to exercise the host paths)
static double enc_guard() {
  static double g = -1.0;
  if (g < 0) { const char* e = getenv("FHERAM_ENC_GUARD"); g = e ? atof(e) : 1e-9; if (!(g >= 1e-12)) g = 1e-12; }
  return g;
}
static double enc_bound_guard() {
  static double g = -1.0;
  if (g < 0) { const char* e = getenv("FHERAM_ENC_BOUND_GUARD"); g = e ? atof(e) : enc_guard(); if (!(g >= 1e-12)) g = 1e-12; }
  return g;
}
// Noise of n_streams Sources (per_stream draws each, stream-major) into d_noise, and every Source advanced as
// that many fheram_source::gauss draws advance it.
static int sample_noise(fheram_ctx* c, fheram_source* const* xe, int n_streams, size_t per_stream, DevBuf& d_noise) {
  TRY(d_noise.ensure((size_t)n_streams * per_stream));
  std::vector<int8_t> host;
  auto host_stream = [&](int s) -> int {
    host.resize(per_stream);
    fheram_source_noise_i8(xe[s], host.data(), per_stream);
    CU(cudaMemcpy((char*)d_noise.p + (size_t)s * per_stream, host.data(), per_stream, cudaMemcpyHostToDevice));
    c->enc_stats[2]++;
    return 0;
  };
  if (!enc_noise_on_device() || per_stream % 4) {  // host sampler only, one thread per stream in flight
    std::vector<int8_t> all((size_t)n_streams * per_stream);
    unsigned nt = std::thread::hardware_concurrency();
    nt = nt < 1 ? 1 : (nt > 32 ? 32 : nt);
    if ((int)nt > n_streams) nt = n_streams;
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; t++)
      th.emplace_back([&, t]() {
        for (int s = t; s < n_streams; s += nt) fheram_source_noise_i8(xe[s], &all[(size_t)s * per_stream], per_stream);
      });
    for (auto& t : th) t.join();
    CU(cudaMemcpy(d_noise.p, all.data(), all.size(), cudaMemcpyHostToDevice));
    c->enc_stats[2] += n_streams;
    return 0;
  }
  const unsigned max_flags = 1u << 16;
  std::vector<uint32_t> keys((size_t)8 * n_streams);
  std::vector<unsigned long long> w0(n_streams);
  for (int s = 0; s < n_streams; s++) fheram_source_tell(xe[s], &keys[8 * s], (uint64_t*)&w0[s]);
  DevBuf &dk = c->enc_buf[0], &dw = c->enc_buf[1], &df = c->enc_buf[2], &dn = c->enc_buf[3];
#define NZ_TRY(x) TRY(x)
#define NZ_CU(x) CU(x)
  NZ_TRY(dk.ensure(keys.size() * sizeof(uint32_t)));
  NZ_TRY(dw.ensure(w0.size() * sizeof(unsigned long long)));
  NZ_TRY(df.ensure((size_t)max_flags * sizeof(unsigned long long)));
  NZ_TRY(dn.ensure(sizeof(unsigned)));
  NZ_CU(cudaMemcpyAsync(dk.p, keys.data(), keys.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
  NZ_CU(cudaMemcpyAsync(dw.p, w0.data(), w0.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, c->stream));
  NZ_CU(cudaMemsetAsync(dn.p, 0, sizeof(unsigned), c->stream));
  NoiseArgs a;
  a.out = (signed char*)d_noise.p; a.n_streams = n_streams; a.per_stream = (long)per_stream;
  a.keys = (const uint32_t*)dk.p; a.word0 = (const unsigned long long*)dw.p; a.guard = enc_guard(); a.bound_guard = enc_bound_guard();
  a.n_flags = (unsigned*)dn.p; a.flags = (unsigned long long*)df.p; a.max_flags = max_flags;
  k_noise_sample<<<c->sm_count * 8, 256, 0, c->stream>>>(a);
  c->launches++;
  NZ_CU(cudaGetLastError());
  unsigned n_flags = 0;
  NZ_CU(cudaMemcpyAsync(&n_flags, dn.p, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
  NZ_CU(cudaStreamSynchronize(c->stream));
  std::vector<char> redo(n_streams, n_flags > max_flags ? 1 : 0);  // more reports than slots: host sampling for all
  if (n_flags && n_flags <= max_flags) {
    std::vector<unsigned long long> flags(n_flags);
    NZ_CU(cudaMemcpy(flags.data(), df.p, (size_t)n_flags * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    for (unsigned long long f : flags)
      if ((f >> 39) & 1) redo[(size_t)(f >> 40)] = 1;
    for (unsigned long long f : flags) {
      const size_t s = (size_t)(f >> 40);
      if (((f >> 39) & 1) || redo[s]) continue;
      const unsigned long long k = f & ((1ull << 39) - 1);
      const int8_t v = fheram_source_noise_at(xe[s], 4ull * k);
      NZ_CU(cudaMemcpy((char*)d_noise.p + s * per_stream + k, &v, 1, cudaMemcpyHostToDevice));
      c->enc_stats[1]++;
    }
  }
  for (int s = 0; s < n_streams; s++) {
    if (redo[s]) NZ_TRY(host_stream(s));
    else { fheram_source_skip_words(xe[s], 4ull * per_stream); c->enc_stats[0] += per_stream; }
  }
#undef NZ_TRY
#undef NZ_CU
  return 0;
}
extern "C" int fheram_debug_encrypt_stats(fheram_ctx* c, uint64_t out[3]) {
  if (!c || !out) return fail(FHERAM_ERR_INVALID, "null argument");
  for (int i = 0; i < 3; i++) out[i] = c->enc_stats[i];
  return 0;
}

static int check_secret(const int64_t* sk, int n) {  // before any Source moves
  for (int i = 0; i < n; i++)
    if (sk[i] < -1 || sk[i] > 1) return fail(FHERAM_ERR_INVALID, "secret key is not ternary");
  return 0;
}
// zero every device buffer that held secret-key material or PRNG state of an encryption call
static void wipe_secrets(fheram_ctx* c) {
  const int idx[] = {0, 1, 4, 5, 9, 10, 11, 12};  // noise Source keys / positions, sk, sk spectrum, mask Source keys / positions, noise, s and s*s
  for (int i : idx)
    if (c->enc_buf[i].p) cudaMemsetAsync(c->enc_buf[i].p, 0, c->enc_buf[i].bytes, c->stream);
}
static int run_encrypt(fheram_ctx* c, const int64_t* sk, const EncBatch& b, const DevBuf& d_noise, bool noise_by_seq,
                       int* d_out, long stride) {
  const int n = c->d.n;
  DevBuf &skraw = c->enc_buf[4], &skspec = c->enc_buf[5], &pt = c->enc_buf[6], &mono = c->enc_buf[7],
         &seq = c->enc_buf[8], &keys = c->enc_buf[9], &word0 = c->enc_buf[10], &poly = c->enc_buf[12],
         &poly_sel = c->enc_buf[13], &sk_sel = c->enc_buf[14];
  // on any failure the secret material already on the device is wiped before returning
#define ENC_TRY(x) do { int rc_ = (x); if (rc_) { wipe_secrets(c); cudaStreamSynchronize(c->stream); return rc_; } } while (0)
#define ENC_CU(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { wipe_secrets(c); cudaStreamSynchronize(c->stream); return fail(FHERAM_ERR_CUDA, "%s: %s", #x, cudaGetErrorString(e_)); } } while (0)
  {
    // the secrets the masks are multiplied by: the caller's sk, or (key generation) the n_sk output secrets of the batch
    std::vector<int> s32;
    if (b.sk_all.empty()) {
      s32.assign((size_t)2 * n, 0);
      for (int i = 0; i < n; i++) s32[i] = (int)sk[i];
    } else {
      s32 = b.sk_all;
    }
    const int n_sk = (int)(s32.size() / (2 * (size_t)n));
    ENC_TRY(skraw.ensure(sizeof(int) * s32.size()));
    ENC_TRY(skspec.ensure(sizeof(double2) * 2 * kM * n_sk));
    ENC_CU(cudaMemcpyAsync(skraw.p, s32.data(), sizeof(int) * s32.size(), cudaMemcpyHostToDevice, c->stream));
    ENC_CU(cudaStreamSynchronize(c->stream));
    volatile int* vs = s32.data();  // host staging copy of the secret
    for (size_t i = 0; i < s32.size(); i++) vs[i] = 0;
    ENC_TRY(prepare(c, (const int*)skraw.p, 2 * n, (double2*)skspec.p, 2 * kM, n_sk, 1, 1, 1));
  }
  auto up = [&](DevBuf& d, const void* h, size_t bytes) -> int {
    if (!bytes) return 0;
    TRY(d.ensure(bytes));
    CU(cudaMemcpyAsync(d.p, h, bytes, cudaMemcpyHostToDevice, c->stream));
    return 0;
  };
  ENC_TRY(up(pt, b.pt.data(), b.pt.size()));
  ENC_TRY(up(mono, b.mono.data(), b.mono.size() * sizeof(int)));
  ENC_TRY(up(seq, b.seq.data(), b.seq.size() * sizeof(int)));
  ENC_TRY(up(keys, b.keys.data(), b.keys.size() * sizeof(uint32_t)));
  ENC_TRY(up(word0, b.word0.data(), b.word0.size() * sizeof(unsigned long long)));
  ENC_TRY(up(poly, b.poly.data(), b.poly.size() * sizeof(short)));
  ENC_TRY(up(poly_sel, b.poly_sel.data(), b.poly_sel.size() * sizeof(int)));
  ENC_TRY(up(sk_sel, b.sk_sel.data(), b.sk_sel.size() * sizeof(int)));
  EncArgs a;
  a.out = d_out; a.ct_stride = stride; a.n_glwe = b.n_glwe; a.size = b.size;
  a.nl = (b.k_noise + kK - 1) / kK - 1; a.sh = (a.nl + 1) * kK - b.k_noise;
  a.sk_spec = (const double2*)skspec.p;
  a.noise = (const signed char*)d_noise.p; a.noise_by_seq = noise_by_seq ? 1 : 0;
  a.pt = b.pt.empty() ? nullptr : (const signed char*)pt.p;
  a.pt_l = b.pt_l; a.pt_sh = b.pt_sh;
  a.mono = b.mono.empty() ? nullptr : (const int*)mono.p;
  a.poly = b.poly.empty() ? nullptr : (const short*)poly.p;
  a.poly_sel = b.poly.empty() ? nullptr : (const int*)poly_sel.p;
  a.sk_sel = b.sk_sel.empty() ? nullptr : (const int*)sk_sel.p;
  a.seq = b.seq.empty() ? nullptr : (const int*)seq.p;
  a.keys = (const uint32_t*)keys.p;
  a.word0 = (const unsigned long long*)word0.p;
  a.glwe_per_stream = b.glwe_per_stream;
  a.tw = c->tw;
  const int grid = b.n_glwe < 2 * c->sm_count ? b.n_glwe : 2 * c->sm_count;
  k_glwe_encrypt<<<grid, kThreads, 0, c->stream>>>(a);
  c->launches++;
  ENC_CU(cudaGetLastError());
  // the secret, its spectrum, the ChaCha20 keys of the Sources and the raw noise do not outlive the call: the
  // context belongs to the evaluator (INTEGRATION.md, colocated client / server mode)
  wipe_secrets(c);
  ENC_CU(cudaStreamSynchronize(c->stream));
#undef ENC_TRY
#undef ENC_CU
  return 0;
}

// Ram::encrypt_sk (src/ram.rs:129-167; SubRam::encrypt_sk :334-380) into the device-resident RAM
extern "C" int fheram_ram_encrypt_sk(fheram_ram* r, const uint8_t* data, const int64_t* sk,
                                     fheram_source* xa, fheram_source* xe) {
  if (!r || !data || !sk || !xa || !xe) return fail(FHERAM_ERR_INVALID, "null argument");
  if (xa == xe) return fail(FHERAM_ERR_INVALID, "mask and noise need distinct Sources");
  fheram_ctx* c = r->c;
  CU(cudaSetDevice(c->device));
  const Derived& d = c->d;
  const fheram_params& p = c->params;
  TRY(check_secret(sk, d.n));
  const int ws = p.word_size, G = d.n_glwe, n = d.n;
  const size_t total = (size_t)ws * G;
  EncBatch b;
  b.n_glwe = ws * r->n_local; b.size = d.size_ct; b.k_noise = p.k_ct;
  b.pt_l = (p.k_pt + kK - 1) / kK - 1; b.pt_sh = (b.pt_l + 1) * kK - p.k_pt;
  if (b.pt_l >= b.size) return fail(FHERAM_ERR_INVALID, "k_pt exceeds k_ct");
  b.keys.resize(8); b.word0.resize(1);
  fheram_source_tell(xa, b.keys.data(), (uint64_t*)&b.word0[0]);
  b.glwe_per_stream = (int)total;
  // noise in the order of src/ram.rs:161-166 (sub-RAM major), every polynomial of every shard: one stream
  DevBuf& d_noise = c->enc_buf[11];
  {
    fheram_source* xes[1] = {xe};
    TRY(sample_noise(c, xes, 1, total * n, d_noise));
  }
  b.pt.resize((size_t)b.n_glwe * n); b.seq.resize(b.n_glwe);
  for (int s = 0; s < ws; s++)
    for (int hp = 0; hp < r->n_local; hp++) {
      const int h = r->shard + r->n_shards * hp;
      const size_t jl = (size_t)s * r->n_local + hp, jg = (size_t)s * G + h;
      b.seq[jl] = (int)jg;
      for (int j = 0; j < n; j++) {
        const uint64_t addr = (uint64_t)h * n + j;
        b.pt[jl * n + j] = addr < p.max_addr ? (int8_t)data[addr * ws + s] : 0;  // src/ram.rs:364
      }
    }
  TRY(run_encrypt(c, sk, b, d_noise, true, r->data, c->ct_stride()));
  fheram_source_skip_words(xa, 2ull * d.size_ct * n * total);
  r->loaded = true;
  r->state = false;
  return 0;
}

// Address::encrypt_sk (src/address.rs:86-109) for addresses [first, first + count) of a device address set.
// n_sources = 1: all addresses draw from (xa[0], xe[0]) one after the other, as `count` calls of
// fheram_encrypt_address would; n_sources = count: address i draws from (xa[i], xe[i]).
// Raw GGSWs only: fheram_address_prepare makes them usable.
extern "C" int fheram_address_encrypt_sk(fheram_address* a, int first, int count, const uint32_t* values,
                                         const int64_t* sk, fheram_source* const* xa, fheram_source* const* xe,
                                         int n_sources) {
  if (!a || !values || !sk || !xa || !xe || first < 0 || count < 1 || first + count > a->count ||
      (n_sources != 1 && n_sources != count))
    return fail(FHERAM_ERR_INVALID, "bad argument");
  fheram_ctx* c = a->c;
  CU(cudaSetDevice(c->device));
  const Derived& d = c->d;
  const int n = d.n, per = d.n_ggsw * d.dnum_ct * 2;
  TRY(check_secret(sk, n));
  for (int i = 0; i < n_sources; i++)
    for (int j = 0; j < n_sources; j++)
      if (xa[i] == xe[j] || (i != j && (xa[i] == xa[j] || xe[i] == xe[j])))
        return fail(FHERAM_ERR_INVALID, "every stream needs its own Source");
  EncBatch b;
  b.n_glwe = count * per; b.size = d.size_addr; b.k_noise = c->params.k_addr;
  b.mono.resize(b.n_glwe);
  for (int i = 0; i < count; i++) {  // every value is checked before a Source is touched
    int32_t pos[64], sign[64];
    const int ng = fheram_address_monomials(&c->params, values[i], pos, sign);
    if (ng < 0) return ng;
    for (int g = 0; g < d.n_ggsw; g++)
      for (int row = 0; row < d.dnum_ct; row++)
        for (int ci = 0; ci < 2; ci++)
          b.mono[(size_t)i * per + (g * d.dnum_ct + row) * 2 + ci] =
              pos[g] | ((sign[g] < 0 ? 1 : 0) << 12) | (row << 16) | (ci << 24);
  }
  b.keys.resize((size_t)8 * n_sources); b.word0.resize(n_sources);
  for (int i = 0; i < n_sources; i++) fheram_source_tell(xa[i], &b.keys[8 * i], (uint64_t*)&b.word0[i]);
  b.glwe_per_stream = n_sources == 1 ? b.n_glwe : per;
  DevBuf& d_noise = c->enc_buf[11];
  TRY(sample_noise(c, xe, n_sources, (size_t)b.n_glwe / n_sources * n, d_noise));
  const long stride = (long)2 * d.size_addr * n;
  TRY(run_encrypt(c, sk, b, d_noise, false, a->raw + (size_t)first * d.n_ggsw * c->ggsw_raw_len(), stride));
  for (int i = 0; i < n_sources; i++)
    fheram_source_skip_words(xa[i], 2ull * d.size_addr * n * (n_sources == 1 ? (uint64_t)b.n_glwe : (uint64_t)per));
  a->inv_ready = false;
  return 0;
}

// EvaluationKeys::encrypt_sk (src/keys.rs:135-180) on the device, followed by EvaluationKeysPrepared::prepare: the 12
// trace keys (GLWEAutomorphismKey, k = k_evk_trace), the GGLWE -> GGSW key and the automorphism key p = -1 (k =
// k_evk_ggsw_inv).  The limbs of fheram_keygen from the same Sources (mask stream regenerated on the device, noise
// sampled on the device, both Sources left where the CPU leaves them); the raw keys stay on the device next to the
// prepared ones (fheram_keys_download_raw).
extern "C" int fheram_keys_encrypt_sk(fheram_ctx* c, const int64_t* sk, fheram_source* xa, fheram_source* xe,
                                      fheram_keys** out) {
  if (!c || !sk || !xa || !xe || !out) return fail(FHERAM_ERR_INVALID, "null argument");
  if (xa == xe) return fail(FHERAM_ERR_INVALID, "mask and noise need distinct Sources");
  CU(cudaSetDevice(c->device));
  const Derived& d = c->d;
  const int n = d.n, log_n = d.log_n;
  TRY(check_secret(sk, n));
  const size_t atk_raw = (size_t)d.dnum_ct * 2 * d.size_evk_trace * n;
  const size_t inv_raw = (size_t)d.dnum_ggsw * 2 * d.size_evk_inv * n;
  fheram_keys* k = new fheram_keys();
  k->c = c;
  CU(cudaMalloc(&k->raw, sizeof(int) * (atk_raw * log_n + 2 * inv_raw)));
  int *d_atk = k->raw, *d_tsk = k->raw + atk_raw * log_n, *d_inv = d_tsk + inv_raw;
  // phi_q(s): coefficient i of s goes to i q mod 2N with the sign of the wrap (client.cpp automorphism)
  auto autom = [&](long q, int* o) {
    for (int i = 0; i < n; i++) {
      const long e = (((long)i * q) % (2L * n) + 2L * n) % (2L * n);
      o[e % n] = e >= n ? -(int)sk[i] : (int)sk[i];
    }
  };
  // plaintext polynomials: 0 = s, 1 = s * s (negacyclic, |coefficient| <= n)
  std::vector<short> poly((size_t)2 * n, 0);
  {
    std::vector<long> s2(n, 0);
    for (int i = 0; i < n; i++) {
      if (!sk[i]) continue;
      for (int j = 0; j < n; j++) {
        if (!sk[j]) continue;
        const int e = i + j;
        s2[e % n] += (e >= n ? -1 : 1) * sk[i] * sk[j];
      }
    }
    for (int i = 0; i < n; i++) { poly[i] = (short)sk[i]; poly[n + i] = (short)s2[i]; }
  }
  struct Part { int n_keys, rows, size, k_noise, poly; int* dst; size_t key_len; };
  const Part parts[3] = {
      {log_n, d.dnum_ct, d.size_evk_trace, c->params.k_evk_trace, 0, d_atk, atk_raw},       // src/keys.rs:158-165
      {1, d.dnum_ggsw, d.size_evk_inv, c->params.k_evk_ggsw_inv, 1, d_tsk, inv_raw},          // :167-169
      {1, d.dnum_ggsw, d.size_evk_inv, c->params.k_evk_ggsw_inv, 0, d_inv, inv_raw}};         // :171-173
  for (int pi = 0; pi < 3; pi++) {
    const Part& P = parts[pi];
    EncBatch b;
    b.n_glwe = P.n_keys * P.rows; b.size = P.size; b.k_noise = P.k_noise;
    b.poly = poly;
    b.sk_all.assign((size_t)P.n_keys * 2 * n, 0);
    for (int ki = 0; ki < P.n_keys; ki++) {
      // output secret of the key: phi_{p^-1}(s) for an automorphism key of p, s itself for the tensor key
      long q = 1;
      if (pi == 0) q = inv_mod_2n((int)((galois(log_n, ki) + 2 * kN) % (2 * kN)));
      if (pi == 2) q = 2 * kN - 1;
      autom(q, &b.sk_all[(size_t)ki * 2 * n]);
      for (int r = 0; r < P.rows; r++) {
        b.poly_sel.push_back(P.poly | (r << 16));
        b.sk_sel.push_back(ki);
      }
    }
    b.keys.resize(8); b.word0.resize(1);
    fheram_source_tell(xa, b.keys.data(), (uint64_t*)&b.word0[0]);
    b.glwe_per_stream = b.n_glwe;
    DevBuf& d_noise = c->enc_buf[11];
    fheram_source* xes[1] = {xe};
    TRY(sample_noise(c, xes, 1, (size_t)b.n_glwe * n, d_noise));
    TRY(run_encrypt(c, sk, b, d_noise, false, P.dst, (long)2 * P.size * n));
    fheram_source_skip_words(xa, 2ull * P.size * n * (uint64_t)b.n_glwe);
    volatile int* vs = b.sk_all.data();
    for (size_t i = 0; i < b.sk_all.size(); i++) vs[i] = 0;
  }
  { volatile short* vp = poly.data(); for (size_t i = 0; i < poly.size(); i++) vp[i] = 0; }
  TRY(keys_prepare_device(c, d_atk, d_tsk, d_inv, k));
  *out = k;
  return 0;
}
// raw limbs of keys made by fheram_keys_encrypt_sk, in the layout fheram_keygen writes (tests; a client that wants to
// keep a copy of the public evaluation keys)
extern "C" int fheram_keys_download_raw(fheram_keys* k, int64_t* atk_glwe, int64_t* tsk, int64_t* atk_inv) {
  if (!k || !atk_glwe || !tsk || !atk_inv) return fail(FHERAM_ERR_INVALID, "null argument");
  if (!k->raw) return fail(FHERAM_ERR_INVALID, "these keys were prepared from host limbs: the caller holds the raw keys");
  fheram_ctx* c = k->c;
  CU(cudaSetDevice(c->device));
  const Derived& d = c->d;
  const size_t atk_raw = (size_t)d.dnum_ct * 2 * d.size_evk_trace * d.n;
  const size_t inv_raw = (size_t)d.dnum_ggsw * 2 * d.size_evk_inv * d.n;
  TRY(download_i64(c, k->raw, atk_raw * d.log_n, atk_glwe));
  TRY(download_i64(c, k->raw + atk_raw * d.log_n, inv_raw, tsk));
  return download_i64(c, k->raw + atk_raw * d.log_n + inv_raw, inv_raw, atk_inv);
}

static int first_coord_ggsw(const Derived& d, int coord) {
  int f = 0;
  for (int i = 0; i < coord; i++) f += d.coord_len[i];
  return f;
}

// Local stage of SubRam::read / read_prepare_write for B addresses (src/ram.rs:411-449 /
// 487-528): rotate every local polynomial by the first coordinate and pack coefficient 0 of
// each into one partial ciphertext per (address, sub-RAM).  inplace = read_prepare_write
// (the rotated polynomials overwrite SubRam::data, src/ram.rs:502-504; B must be 1).
// Result: r->partial = [B][word_size] GLWE.
static int ram_local_stage(fheram_ram* r, const fheram_address* addr, int first_addr, int B,
                           const fheram_keys* k, bool inplace) {
  fheram_ctx* c = r->c;
  const Derived& d = c->d;
  const int ws = c->params.word_size, nl = r->n_local;
  const long L = c->ct_stride();
  const int per_addr = ws * nl;
  const int items = B * per_addr;
  TRY(r->bufA.ensure(sizeof(int) * (size_t)items * L));
  TRY(r->bufB.ensure(sizeof(int) * (size_t)items * L));
  TRY(r->partial.ensure(sizeof(int) * (size_t)B * ws * L));
  int* A = (int*)r->bufA.p;
  int* Bb = (int*)r->bufB.p;
  // matrices of the first coordinate of address first_addr, and the distance to the next address
  const long mat_stride = (long)(addr->prep1 ? d.coord_len[0] : d.n_ggsw) * c->ggsw_prep_len();
  const double2* mats = addr->prep + (size_t)first_addr * mat_stride;
  const int lg_total = ilog2(d.n_glwe);          // two-sided levels of the full tree
  const int one_sided = d.log_n - lg_total;      // levels with a single non-empty child
  if (d.n_coord == 1) {
    // max_addr <= N: product on data[0] only (src/ram.rs:450-452); "partial" = rotated poly
    if (inplace) {
      TRY(run_ext_chain(c, per_addr, r->data, nullptr, 0, r->data, mats, d.coord_len[0], 0, 0));
      CU(cudaMemcpyAsync(r->partial.p, r->data, sizeof(int) * (size_t)ws * L, cudaMemcpyDeviceToDevice, c->stream));
    } else {
      TRY(run_ext_chain(c, items, r->data, nullptr, per_addr, (int*)r->partial.p, mats, d.coord_len[0], per_addr, mat_stride));
    }
    return 0;
  }
  if (inplace) {
    // src/ram.rs:502-504 product_inplace on every polynomial, then pack (src/ram.rs:510-521)
    TRY(run_ext_chain(c, per_addr, r->data, nullptr, 0, r->data, mats, d.coord_len[0], 0, 0));
    TRY(run_trace_chain(c, k, per_addr, r->data, r->feed_map, per_addr, 0, A, 0, one_sided));
  } else {
    // src/ram.rs:429-435: product into tmp_ct then packer.add, in feed order
    TRY(run_ext_chain(c, items, r->data, r->feed_map, per_addr, A, mats, d.coord_len[0], per_addr, mat_stride));
    TRY(run_trace_chain(c, k, items, A, nullptr, 0, 0, A, 0, one_sided));
  }
  int* res = nullptr;
  TRY(run_pack_levels(c, k, B * ws, nl, one_sided, A, Bb, &res));
  CU(cudaMemcpyAsync(r->partial.p, res, sizeof(int) * (size_t)B * ws * L, cudaMemcpyDeviceToDevice, c->stream));
  return 0;
}

// Finishing stage for reads [first, first+count) of a batch of n_total: combine the
// n_shards partials of each (read, sub-RAM) through the top packer levels, rotate by the
// second coordinate (src/ram.rs:453-455) and trace (src/ram.rs:457).  gathered =
// [n_shards][n_total][word_size] GLWE (rank-major).  store_tree: read_prepare_write keeps the
// rotated packed polynomial in SubRam::tree[0][0] (src/ram.rs:525-527,499-504).
static int ram_finish_stage(fheram_ram* r, const int* gathered, int n_total, int first, int count,
                            const fheram_address* addr, int first_addr, const fheram_keys* k,
                            bool store_tree) {
  fheram_ctx* c = r->c;
  const Derived& d = c->d;
  const int ws = c->params.word_size, S = r->n_shards;
  const long L = c->ct_stride();
  TRY(r->result.ensure(sizeof(int) * (size_t)count * ws * L));
  int* res = (int*)r->result.p;
  const int groups = count * ws;
  const int* packed = nullptr;
  if (d.n_coord == 1) {
    packed = gathered + (size_t)first * ws * L;
    if (store_tree) {
      // n2 == 1: result = copy of data[0] (src/ram.rs:536-538); no tree
      CU(cudaMemcpyAsync(res, packed, sizeof(int) * (size_t)groups * L, cudaMemcpyDeviceToDevice, c->stream));
    } else {
      CU(cudaMemcpyAsync(res, packed, sizeof(int) * (size_t)groups * L, cudaMemcpyDeviceToDevice, c->stream));
    }
    TRY(run_trace_chain(c, k, groups, res, nullptr, 0, 0, res, 0, d.log_n));
    return 0;
  }
  if (S > 1) {
    // gather the S partials of each group in tree order: block index bitrev(shard)
    TRY(r->bufA.ensure(sizeof(int) * (size_t)groups * S * L));
    TRY(r->bufB.ensure(sizeof(int) * (size_t)groups * S * L));
    int* A = (int*)r->bufA.p;
    const int lgS = ilog2(S);
    for (int blk = 0; blk < S; blk++) {
      const int shard = (int)revbits(blk, lgS);
      // A[(g*S + blk)] = gathered[shard][first*ws + g]
      CU(cudaMemcpy2DAsync(A + (size_t)blk * L, sizeof(int) * (size_t)S * L,
                           gathered + ((size_t)shard * n_total + first) * ws * L, sizeof(int) * L,
                           sizeof(int) * L, groups, cudaMemcpyDeviceToDevice, c->stream));
    }
    int* out = nullptr;
    const int first_level = d.log_n - lgS;
    TRY(run_pack_levels(c, k, groups, S, first_level, A, (int*)r->bufB.p, &out));
    packed = out;
  } else {
    packed = gathered + (size_t)first * ws * L;
  }
  const int c1 = first_coord_ggsw(d, 1);
  const long mat_stride = (long)(addr->prep1 ? d.coord_len[1] : d.n_ggsw) * c->ggsw_prep_len();
  const double2* mats = addr->prep1
      ? addr->prep1 + (size_t)(first_addr + first - addr->prep1_first) * mat_stride
      : addr->prep + ((size_t)(first_addr + first) * d.n_ggsw + c1) * c->ggsw_prep_len();
  if (store_tree) {
    TRY(run_ext_chain(c, groups, packed, nullptr, 0, r->tree, mats, d.coord_len[1], ws, mat_stride));
    CU(cudaMemcpyAsync(res, r->tree, sizeof(int) * (size_t)groups * L, cudaMemcpyDeviceToDevice, c->stream));  // src/ram.rs:535
  } else {
    TRY(run_ext_chain(c, groups, packed, nullptr, 0, res, mats, d.coord_len[1], ws, mat_stride));
  }
  TRY(run_trace_chain(c, k, groups, res, nullptr, 0, 0, res, 0, d.log_n));  // src/ram.rs:457,540
  return 0;
}

static int check_read_args(fheram_ram* r, const fheram_address* addr, const fheram_keys* k) {
  if (!r || !addr || !k) return fail(FHERAM_ERR_INVALID, "null argument");
  if (addr->c != r->c || k->c != r->c) return fail(FHERAM_ERR_INVALID, "handles belong to different contexts");
  if (!r->loaded) return fail(FHERAM_ERR_UNINIT, "unitialized memory: self.data.len()=0 (src/ram.rs:182-185)");
  if (r->state)
    return fail(FHERAM_ERR_STATE, "invalid call to Memory.read: internal state is true -> requires calling Memory.write (src/ram.rs:393-396)");
  if (r->rotated)
    return fail(FHERAM_ERR_STATE, "read_prepare_write did not complete (rpw_local_device without a successful rpw_finish_device): the RAM is rotated; finish it, then write");
  return 0;
}

// reads per chunk of a batched read: bounds the work arenas (chunk * word_size * n_glwe GLWE)
static int batch_chunk(const fheram_ram* r) {
  const size_t per_read = (size_t)r->c->params.word_size * r->n_local * r->c->ct_stride() * sizeof(int);
  size_t budget = (size_t)3 << 30;  // bytes per arena
  int ch = (int)(budget / (per_read ? per_read : 1));
  if (ch < 1) ch = 1;
  int cap = 64;
  if (const char* e = getenv("FHERAM_CHUNK")) { int v = atoi(e); if (v > 0) cap = v; }
  if (ch > cap) ch = cap;
  return ch;
}

// Sharded RAM with a communicator: addr holds the WHOLE batch (B addresses, the same on every rank, B a multiple of
// n_ranks); rank q finishes reads [q B / G, (q + 1) B / G) and *d_out points at those B / G results.
static int read_batch_device_sharded(fheram_ram* r, const fheram_address* addr, const fheram_keys* k,
                                     const int32_t** d_out) {
  fheram_ctx* c = r->c;
  const int G = r->n_shards, B = addr->count, ws = c->params.word_size;
  const long L = c->ct_stride();
  if (B % G) return fail(FHERAM_ERR_INVALID, "batch must be a multiple of the number of ranks");
  const int mine = B / G;
  const int chunk = batch_chunk(r);
  TRY(r->part_all.ensure(sizeof(int) * (size_t)B * ws * L));
  TRY(r->xchg.ensure(sizeof(int) * (size_t)B * ws * L));
  for (int b0 = 0; b0 < B; b0 += chunk) {          // local stage: rotate + pack the own polynomials for every read
    const int nb = B - b0 < chunk ? B - b0 : chunk;
    TRY(ram_local_stage(r, addr, b0, nb, k, false));
    CU(cudaMemcpyAsync((int*)r->part_all.p + (size_t)b0 * ws * L, r->partial.p, sizeof(int) * (size_t)nb * ws * L,
                       cudaMemcpyDeviceToDevice, c->stream));
  }
  // one exchange step: block q of the partials (reads of rank q) goes to rank q
  TRY(all_to_all_i32(c, (const int*)r->part_all.p, (int*)r->xchg.p, (size_t)mine * ws * L));
  if (mine <= chunk) {
    TRY(ram_finish_stage(r, (const int*)r->xchg.p, mine, 0, mine, addr, r->shard * mine, k, false));
    *d_out = (const int32_t*)r->result.p;
    return 0;
  }
  TRY(r->all.ensure(sizeof(int) * (size_t)mine * ws * L));
  for (int f = 0; f < mine; f += chunk) {
    const int nb = mine - f < chunk ? mine - f : chunk;
    TRY(ram_finish_stage(r, (const int*)r->xchg.p, mine, f, nb, addr, r->shard * mine, k, false));
    CU(cudaMemcpyAsync((int*)r->all.p + (size_t)f * ws * L, r->result.p, sizeof(int) * (size_t)nb * ws * L,
                       cudaMemcpyDeviceToDevice, c->stream));
  }
  *d_out = (const int32_t*)r->all.p;
  return 0;
}

extern "C" int fheram_ram_read_batch_device(fheram_ram* r, const fheram_address* addr,
                                            const fheram_keys* k, const int32_t** d_out) {
  TRY(check_read_args(r, addr, k));
  if (!d_out) return fail(FHERAM_ERR_INVALID, "null argument");
  fheram_ctx* c = r->c;
  CU(cudaSetDevice(c->device));
  if (r->n_shards != 1) {
    if (!comm_matches(c, r->shard, r->n_shards))
      return fail(FHERAM_ERR_INVALID, "sharded RAM: call fheram_comm_init(ctx, n_shards, shard, id) first, or use read_local_device / read_finish_device");
    return read_batch_device_sharded(r, addr, k, d_out);
  }
  const int B = addr->count, ws = c->params.word_size;
  const long L = c->ct_stride();
  const int chunk = batch_chunk(r);
  DevBuf& all = r->all;  // results of every chunk
  if (B <= chunk) {
    TRY(ram_local_stage(r, addr, 0, B, k, false));
    TRY(ram_finish_stage(r, (const int*)r->partial.p, B, 0, B, addr, 0, k, false));
    *d_out = (const int32_t*)r->result.p;
    return 0;
  }
  TRY(all.ensure(sizeof(int) * (size_t)B * ws * L));
  for (int b0 = 0; b0 < B; b0 += chunk) {
    const int nb = B - b0 < chunk ? B - b0 : chunk;
    TRY(ram_local_stage(r, addr, b0, nb, k, false));
    TRY(ram_finish_stage(r, (const int*)r->partial.p, nb, 0, nb, addr, b0, k, false));
    CU(cudaMemcpyAsync((int*)all.p + (size_t)b0 * ws * L, r->result.p, sizeof(int) * (size_t)nb * ws * L,
                       cudaMemcpyDeviceToDevice, c->stream));
  }
  *d_out = (const int32_t*)all.p;
  return 0;
}

extern "C" int fheram_ram_read_batch(fheram_ram* r, const fheram_address* addr, const fheram_keys* k, int64_t* out) {
  if (!out) return fail(FHERAM_ERR_INVALID, "null argument");
  const int32_t* d = nullptr;
  TRY(fheram_ram_read_batch_device(r, addr, k, &d));
  // sharded: this rank's slice of the results (reads [shard B / G, (shard + 1) B / G))
  return download_i64(r->c, d, (size_t)(addr->count / r->n_shards) * r->c->params.word_size * r->c->ct_stride(), out);
}
extern "C" int fheram_ram_read(fheram_ram* r, const fheram_address* addr, const fheram_keys* k, int64_t* out) {
  if (addr && addr->count != 1) return fail(FHERAM_ERR_INVALID, "fheram_ram_read takes a single address");
  return fheram_ram_read_batch(r, addr, k, out);
}

// Pipelined end-to-end batched read from HOST buffers (the reference-facing call for a batch):
// addresses arrive as limbs in host memory, results leave as limbs.  Host formats: int64 limbs (Poulpy's VecZnx,
// elem_bytes 8) or the same limbs as int32 (elem_bytes 4: half the PCIe bytes, no conversion pass).
// Chunks of addresses are double-buffered: the H2D copy of chunk k+1 runs on a copy stream while chunk k is
// prepared (CoordinatePrepared::prepare) and read on the compute stream, and the results of chunk k-1 go back on a
// third stream.
// Sharded RAM (fheram_comm_init done): every rank passes ITS n addresses and receives ITS n results; the global batch
// is the concatenation over ranks.  Per chunk: each rank uploads and prepares only its own addresses, the prepared
// GGSWs are all-gathered over NVLink (NCCL, in place), every rank rotates + packs its own polynomials for all
// n_ranks * nb reads of the chunk, the packed partials are exchanged with one all-to-all, and each rank finishes its
// own nb reads (top log2 n_ranks packer levels, second coordinate, trace).
// in_fmt: 8 (int64 limbs), 4 (int32 limbs) or 17 (packed 17-bit fields, fheram_pack17)
static int read_batch_host_impl(fheram_ram* r, const void* ggsw_host, int in_fmt, int n, const fheram_keys* k,
                                void* out_host, int out_bytes) {
  if (!r || !ggsw_host || !k || !out_host || n < 1) return fail(FHERAM_ERR_INVALID, "bad argument");
  if (k->c != r->c) return fail(FHERAM_ERR_INVALID, "handles belong to different contexts");
  if (!r->loaded) return fail(FHERAM_ERR_UNINIT, "unitialized memory: self.data.len()=0 (src/ram.rs:182-185)");
  if (r->state || r->rotated) return fail(FHERAM_ERR_STATE, "invalid call to Memory.read: internal state is true (src/ram.rs:393-396)");
  fheram_ctx* c = r->c;
  const int G = r->n_shards;
  if (G != 1 && !comm_matches(c, r->shard, G))
    return fail(FHERAM_ERR_INVALID, "sharded RAM: call fheram_comm_init(ctx, n_shards, shard, id) first, or use the *_device halves");
  CU(cudaSetDevice(c->device));
  const Derived& d = c->d;
  const int ws = c->params.word_size;
  const long L = c->ct_stride();
  const size_t per_addr = (size_t)d.n_ggsw * c->ggsw_raw_len();                   // limbs per address
  const size_t glen = (size_t)c->ggsw_prep_len();                                   // double2 per prepared GGSW
  int chunk = batch_chunk(r);   // reads per rank and chunk: the local stage handles G * chunk reads of 1 / G of the RAM
  if (chunk > n) chunk = n;
  // staging buffers, events and the copy stream are created once per RAM handle and reused
  // (cudaMalloc / cudaFree of gigabytes per call cost more than the copies they serve)
  typedef fheram_ram::HostPipe::Set Set;
  fheram_ram::HostPipe& hp = r->pipe;
  int rc = 0;
  auto cleanup = [&]() {
    cudaStreamSynchronize(hp.copy_stream);
    cudaStreamSynchronize(c->stream);
    if (hp.down_stream) cudaStreamSynchronize(hp.down_stream);
  };
#define TRYC(x) do { rc = (x); if (rc) { cleanup(); return rc; } } while (0)
#define CUC(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { cleanup(); return fail(FHERAM_ERR_CUDA, "%s: %s", #x, cudaGetErrorString(e_)); } } while (0)
#define NCC(x) do { ncclResult_t e_ = (x); if (e_ != ncclSuccess) { cleanup(); return fail(FHERAM_ERR_CUDA, "%s: %s", #x, ncclGetErrorString(e_)); } } while (0)
  if (!hp.copy_stream) CU(cudaStreamCreateWithFlags(&hp.copy_stream, cudaStreamNonBlocking));
  if (!hp.down_stream) CU(cudaStreamCreateWithFlags(&hp.down_stream, cudaStreamNonBlocking));
  if (hp.cap < chunk) {
    for (auto& s : hp.sets) {
      cudaFree(s.stage); cudaFree(s.a.raw); cudaFree(s.a.prep); cudaFree(s.a.prep1);
      s.stage = nullptr; s.a.raw = nullptr; s.a.prep = nullptr; s.a.prep1 = nullptr;
      s.a.c = c;
      CU(cudaMalloc(&s.stage, sizeof(long long) * chunk * per_addr));       // int64 staging of the own slice
      CU(cudaMalloc(&s.a.raw, sizeof(int) * chunk * per_addr));             // raw limbs of the own slice
      // prepared GGSWs: first coordinate of every rank's slice (all-gathered), second coordinate of the own slice
      CU(cudaMalloc(&s.a.prep, (size_t)G * chunk * d.coord_len[0] * glen * sizeof(double2)));
      if (d.n_coord > 1) CU(cudaMalloc(&s.a.prep1, (size_t)chunk * d.coord_len[1] * glen * sizeof(double2)));
      if (!s.copied) CU(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
      if (!s.freed) CU(cudaEventCreateWithFlags(&s.freed, cudaEventDisableTiming));
    }
    for (int i = 0; i < 2; i++) {
      cudaFree(hp.out_stage[i]);
      hp.out_stage[i] = nullptr;
      CU(cudaMalloc(&hp.out_stage[i], sizeof(long long) * (size_t)chunk * ws * L));
      if (!hp.out_ready[i]) CU(cudaEventCreateWithFlags(&hp.out_ready[i], cudaEventDisableTiming));
      if (!hp.out_done[i]) CU(cudaEventCreateWithFlags(&hp.out_done[i], cudaEventDisableTiming));
    }
    hp.cap = chunk;
  }
  if (G > 1) TRYC(r->xchg.ensure(sizeof(int) * (size_t)G * chunk * ws * L));
  Set* sets = hp.sets;
  cudaStream_t copy_stream = hp.copy_stream;
  // chunk boundaries: the first chunk is small (its upload overlaps nothing), the sizes then double up to the full
  // chunk, and the schedule is laid out from the END so that no tiny chunk (narrow launches) trails a batch that is
  // not a multiple of the chunk: n = 128 -> 8, 8, 16, 32, 64;  n = 1024 -> 8, 8, 16, 32, 64, 64, ...
  std::vector<int> start;
  {
    std::vector<int> sizes;
    int left = n, sz = chunk;
    while (left > 0) {
      const int take = left < sz ? left : sz;
      sizes.push_back(take);
      left -= take;
      if (left < 2 * sz && sz > 8) sz = sz / 2 > 8 ? sz / 2 : 8;  // ramp down towards the front of the batch
    }
    int b = 0;
    for (size_t i = sizes.size(); i-- > 0;) { start.push_back(b); b += sizes[i]; }
  }
  start.push_back(n);
  const int n_chunks = (int)start.size() - 1;
  const char* in = (const char*)ggsw_host;
  char* out = (char*)out_host;
  // upload side of chunk ci, all on the copy stream: host -> device, limb conversion, CoordinatePrepared::prepare of
  // the OWN addresses, all-gather of the first-coordinate matrices (NVLink, own communicator); it runs beside the reads
  // of chunk ci - 1 on the compute stream
  auto issue_copy = [&](int ci) -> int {
    Set& s = sets[ci & 1];
    const int b0 = start[ci], nb = start[ci + 1] - b0;
    if (ci >= 2) CU(cudaStreamWaitEvent(copy_stream, s.freed, 0));
    void* dst = in_fmt == 4 ? (void*)s.a.raw : (void*)s.stage;  // int32 limbs land where the prepare kernel reads them
    const size_t addr_bytes = in_fmt == 17 ? per_addr * 17 / 8 : per_addr * in_fmt;  // per_addr is a multiple of 4096
    CU(cudaMemcpyAsync(dst, in + (size_t)b0 * addr_bytes, (size_t)nb * addr_bytes, cudaMemcpyHostToDevice, copy_stream));
    if (in_fmt == 8) {
      k_i64_to_i32<<<c->sm_count * 8, 256, 0, copy_stream>>>(s.stage, s.a.raw, (size_t)nb * per_addr, c->d_err);
      c->launches++;
    } else if (in_fmt == 17) {
      k_unpack17<<<c->sm_count * 8, 256, 0, copy_stream>>>((const uint32_t*)s.stage, s.a.raw, (size_t)nb * per_addr);
      c->launches++;
    }
    // one "matrix" of the prepare kernel = the coord_len[.] consecutive GGSWs of one coordinate of one address
    const int n0 = d.coord_len[0], n1 = d.n_coord > 1 ? d.coord_len[1] : 0;
    double2* own = s.a.prep + (size_t)r->shard * nb * n0 * glen;
    TRY(prepare(c, s.a.raw, (long)per_addr, own, (long)(n0 * glen), nb, n0 * d.dnum_ct, 2, d.size_addr, 1, true,
                copy_stream));
    if (n1)
      TRY(prepare(c, s.a.raw + (size_t)n0 * c->ggsw_raw_len(), (long)per_addr, s.a.prep1, (long)(n1 * glen), nb,
                  n1 * d.dnum_ct, 2, d.size_addr, 1, true, copy_stream));
    if (G > 1) NC(ncclAllGather(own, s.a.prep, (size_t)nb * n0 * glen * sizeof(double2), ncclChar, c->comm_prep, copy_stream));
    CU(cudaEventRecord(s.copied, copy_stream));
    return 0;
  };
  TRYC(issue_copy(0));
  for (int ci = 0; ci < n_chunks; ci++) {
    if (ci + 1 < n_chunks) TRYC(issue_copy(ci + 1));
    Set& s = sets[ci & 1];
    const int b0 = start[ci], nb = start[ci + 1] - b0;
    s.a.count = G * nb;
    s.a.prep1_first = r->shard * nb;
    CUC(cudaStreamWaitEvent(c->stream, s.copied, 0));
    TRYC(ram_local_stage(r, &s.a, 0, G * nb, k, false));
    const int* gathered = (const int*)r->partial.p;
    if (G > 1) {
      TRYC(all_to_all_i32(c, (const int*)r->partial.p, (int*)r->xchg.p, (size_t)nb * ws * L));
      gathered = (const int*)r->xchg.p;
    }
    TRYC(ram_finish_stage(r, gathered, nb, 0, nb, &s.a, r->shard * nb, k, false));
    CUC(cudaEventRecord(s.freed, c->stream));
    // results: widened on the compute stream if the host wants int64, downloaded on a third stream (overlaps the
    // next chunk's reads)
    long long* os = hp.out_stage[ci & 1];
    if (ci >= 2) CUC(cudaStreamWaitEvent(c->stream, hp.out_done[ci & 1], 0));
    const size_t n_res = (size_t)nb * ws * L;
    if (out_bytes == 8) {
      k_i32_to_i64<<<c->sm_count * 4, 256, 0, c->stream>>>((const int*)r->result.p, os, n_res);
      c->launches++;
    } else {
      CUC(cudaMemcpyAsync(os, r->result.p, sizeof(int) * n_res, cudaMemcpyDeviceToDevice, c->stream));
    }
    CUC(cudaEventRecord(hp.out_ready[ci & 1], c->stream));
    CUC(cudaStreamWaitEvent(hp.down_stream, hp.out_ready[ci & 1], 0));
    CUC(cudaMemcpyAsync(out + (size_t)b0 * ws * L * out_bytes, os, n_res * out_bytes, cudaMemcpyDeviceToHost, hp.down_stream));
    CUC(cudaEventRecord(hp.out_done[ci & 1], hp.down_stream));
  }
  CUC(cudaStreamSynchronize(c->stream));
  CUC(cudaStreamSynchronize(hp.down_stream));
  int err = 0;
  CUC(cudaMemcpy(&err, c->d_err, sizeof(int), cudaMemcpyDeviceToHost));
  cleanup();
#undef TRYC
#undef CUC
#undef NCC
  if (err) {
    cudaMemset(c->d_err, 0, sizeof(int));
    return fail(FHERAM_ERR_RANGE, "limb outside +-2^30: ciphertext limbs must be (nearly) normalised");
  }
  return 0;
}
extern "C" int fheram_ram_read_batch_host(fheram_ram* r, const int64_t* ggsw_host, int n, const fheram_keys* k,
                                          int64_t* out_host) {
  return read_batch_host_impl(r, ggsw_host, 8, n, k, out_host, 8);
}
// packed host format: addresses as 17-bit fields (fheram_pack17: 2.125 bytes per limb), results as int32 limbs
extern "C" int fheram_ram_read_batch_host_p17(fheram_ram* r, const uint32_t* ggsw_packed, int n, const fheram_keys* k,
                                              int32_t* out_host) {
  return read_batch_host_impl(r, ggsw_packed, 17, n, k, out_host, 4);
}
// compact host format: the same limbs as int32 (normalised digits fit 17 bits), addresses and results
extern "C" int fheram_ram_read_batch_host_i32(fheram_ram* r, const int32_t* ggsw_host, int n, const fheram_keys* k,
                                              int32_t* out_host) {
  return read_batch_host_impl(r, ggsw_host, 4, n, k, out_host, 4);
}

extern "C" int fheram_ram_read_local_device(fheram_ram* r, const fheram_address* addr,
                                            const fheram_keys* k, const int32_t** d_partial) {
  TRY(check_read_args(r, addr, k));
  CU(cudaSetDevice(r->c->device));
  TRY(ram_local_stage(r, addr, 0, addr->count, k, false));
  *d_partial = (const int32_t*)r->partial.p;
  return 0;
}
extern "C" int fheram_ram_read_finish_device(fheram_ram* r, const int32_t* d_gathered, int n_total,
                                             int first, int count, const fheram_address* addr,
                                             int addr_first, const fheram_keys* k, const int32_t** d_out) {
  if (!r || !d_gathered || !addr || !k || !d_out) return fail(FHERAM_ERR_INVALID, "null argument");
  if (first < 0 || count < 0 || first + count > n_total || addr_first < 0 ||
      addr_first + first + count > addr->count)
    return fail(FHERAM_ERR_INVALID, "bad read range");
  TRY(check_read_args(r, addr, k));
  CU(cudaSetDevice(r->c->device));
  TRY(ram_finish_stage(r, d_gathered, n_total, first, count, addr, addr_first, k, false));
  *d_out = (const int32_t*)r->result.p;
  return 0;
}

static int address_prepare_inv(const fheram_address* a, const fheram_keys* k);
// Ram::read_prepare_write (src/ram.rs:196-222, 461-542).  For a sharded RAM the caller runs
// fheram_ram_rpw_local_device, all-gathers the partials and calls fheram_ram_rpw_finish_device
// on every rank (the finishing stage is replicated so every rank holds tree[0][0]).
extern "C" int fheram_ram_rpw_local_device(fheram_ram* r, const fheram_address* addr,
                                           const fheram_keys* k, const int32_t** d_partial) {
  TRY(check_read_args(r, addr, k));
  if (addr->count != 1) return fail(FHERAM_ERR_INVALID, "read_prepare_write takes a single address");
  CU(cudaSetDevice(r->c->device));
  r->rotated = true;  // before the in-place product: a failure below must not leave a readable, rotated RAM
  TRY(ram_local_stage(r, addr, 0, 1, k, true));
  *d_partial = (const int32_t*)r->partial.p;
  return 0;
}
extern "C" int fheram_ram_rpw_finish_device(fheram_ram* r, const int32_t* d_gathered,
                                            const fheram_address* addr, const fheram_keys* k,
                                            const int32_t** d_out) {
  if (!r || !d_gathered || !addr || !k || !d_out) return fail(FHERAM_ERR_INVALID, "null argument");
  if (addr->c != r->c || k->c != r->c) return fail(FHERAM_ERR_INVALID, "handles belong to different contexts");
  if (!r->loaded) return fail(FHERAM_ERR_UNINIT, "unitialized memory: self.data.len()=0 (src/ram.rs:206-209)");
  if (!r->rotated || r->state) return fail(FHERAM_ERR_STATE, "rpw_finish_device without a preceding rpw_local_device");
  if (addr->count != 1) return fail(FHERAM_ERR_INVALID, "read_prepare_write takes a single address");
  CU(cudaSetDevice(r->c->device));
  TRY(ram_finish_stage(r, d_gathered, 1, 0, 1, addr, 0, k, true));
  r->rotated = false;
  r->state = true;  // src/ram.rs:533
  *d_out = (const int32_t*)r->result.p;
  return 0;
}
extern "C" int fheram_ram_read_prepare_write(fheram_ram* r, const fheram_address* addr,
                                             const fheram_keys* k, int64_t* out) {
  if (!out) return fail(FHERAM_ERR_INVALID, "null argument");
  if (r && r->n_shards != 1 && !comm_matches(r->c, r->shard, r->n_shards))
    return fail(FHERAM_ERR_INVALID, "sharded RAM: call fheram_comm_init first, or use rpw_local_device / rpw_finish_device");
  const int32_t *part = nullptr, *res = nullptr;
  if (!r || !addr || !k) return fail(FHERAM_ERR_INVALID, "null argument");
  // the inverse address the write that follows needs (src/ram.rs:260-271,278-289) depends on the address and the keys
  // only: it is built on a side stream beside the read (18 CTAs of key switches + vmp_prepare next to launches that
  // leave most SMs idle in their narrow phases) and joined before this call's last operation
  fheram_ctx* cx = r->c;
  bool forked = false;
  if (addr->c == cx && k->c == cx && addr->count == 1 && !addr->inv_ready && r->loaded && !r->state && !r->rotated) {
    CU(cudaSetDevice(cx->device));
    if (!cx->side) {
      CU(cudaStreamCreateWithFlags(&cx->side, cudaStreamNonBlocking));
      CU(cudaEventCreateWithFlags(&cx->side_fork, cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&cx->side_join, cudaEventDisableTiming));
    }
    const Derived& dd = cx->d;
    TRY(cx->scratch_side.ensure(sizeof(int) * (size_t)dd.n_ggsw * dd.dnum_ct * 8 * dd.size_addr * dd.n));
    CU(cudaEventRecord(cx->side_fork, cx->stream));
    CU(cudaStreamWaitEvent(cx->side, cx->side_fork, 0));
    cudaStream_t main_stream = cx->stream;
    cx->stream = cx->side; cx->on_side = true;
    const int rc = address_prepare_inv(addr, k);
    cx->stream = main_stream; cx->on_side = false;
    CU(cudaEventRecord(cx->side_join, cx->side));
    forked = true;
    if (rc) { cudaStreamWaitEvent(cx->stream, cx->side_join, 0); return rc; }
  }
  const int rc_body = [&]() -> int {
  TRY(fheram_ram_rpw_local_device(r, addr, k, &part));
  if (r->n_shards != 1) {
    // every rank needs tree[0][0] (Ram::write then runs without communication): all-gather the packed partials and
    // finish on every rank (bit-identical by construction: integer limbs, every combine executed with the same operands)
    fheram_ctx* c = r->c;
    const size_t cnt = (size_t)c->params.word_size * c->ct_stride();
    TRY(r->xchg.ensure(sizeof(int) * cnt * r->n_shards));
    NC(ncclAllGather(part, r->xchg.p, cnt, ncclInt32, c->comm, c->stream));
    part = (const int32_t*)r->xchg.p;
  }
  TRY(fheram_ram_rpw_finish_device(r, part, addr, k, &res));
  TRY(download_i64(r->c, res, (size_t)r->c->params.word_size * r->c->ct_stride(), out));
  return 0;
  }();
  if (forked) CU(cudaStreamWaitEvent(cx->stream, cx->side_join, 0));  // whatever follows on the RAM sees the inverse address
  if (rc_body) return rc_body;
  return address_prepare_inv(addr, k);  // (already done on the side stream unless the fork was skipped)
}

// CoordinatePrepared::prepare_inv for every coordinate of the address (src/ram.rs:260-271,
// 278-289 -> src/coordinate_prepared.rs:121-142): GGSW::automorphism(p = -1) of each digit
// (key-switch-automorphism of the column-0 GLWE of every row with atk_ggsw_inv, column 1 rebuilt
// with tsk_ggsw_inv) followed by vmp_prepare.
static int ggsw_invert_device(fheram_ctx* c, const fheram_keys* k, const int* raw, int n_ggsw, int* inv_raw) {
  const Derived& d = c->d;
  const long glwe4 = (long)2 * d.size_addr * d.n;  // one GLWE(k_addr), ints
  const int items = n_ggsw * d.dnum_ct;            // rows
  {
    VmpArgs a = base_args(c, items, raw, inv_raw, 2 * glwe4);
    a.n_steps = 1;
    a.mat[0] = k->atk_inv;
    a.gal[0] = 2 * kN - 1;
    a.gal_inv[0] = 2 * kN - 1;
    TRY(launch(c, KC_OTHER, K_AUTO_INV, std::min(items, c->sm_count), kThreads, smem_bytes(4), a));
  }
  {
    VmpArgs a = base_args(c, items, inv_raw, inv_raw + glwe4, 2 * glwe4);
    a.n_steps = 1;
    a.mat[0] = k->tsk;
    a.gal[0] = 1;
    a.gal_inv[0] = 1;
    TRY(launch(c, KC_OTHER, K_EXPAND, std::min(items, c->sm_count), kThreads, smem_bytes(4), a));
  }
  return 0;
}
static int address_prepare_inv(const fheram_address* a, const fheram_keys* k) {
  fheram_ctx* c = a->c;
  const Derived& d = c->d;
  if (a->count != 1) return fail(FHERAM_ERR_INVALID, "write takes a single address");
  if (a->inv_ready) return 0;
  if (!a->inv_raw) {
    CU(cudaMalloc(&a->inv_raw, sizeof(int) * (size_t)d.n_ggsw * c->ggsw_raw_len()));
    CU(cudaMalloc(&a->inv_prep, sizeof(double2) * (size_t)d.n_ggsw * c->ggsw_prep_len()));
  }
  TRY(ggsw_invert_device(c, k, a->raw, d.n_ggsw, a->inv_raw));
  TRY(prepare_ggsw(c, a->inv_raw, a->inv_prep, d.n_ggsw));
  a->inv_ready = true;
  return 0;
}

// Ram::write (src/ram.rs:226-294).  Works on sharded RAMs without communication: the steps that
// touch tree[0][0] are replicated on every rank, the rest touches only local polynomials.
extern "C" int fheram_ram_write(fheram_ram* r, const int64_t* w, const fheram_address* addr,
                                const fheram_keys* k) {
  if (!r || !addr || !k) return fail(FHERAM_ERR_INVALID, "null argument");
  fheram_ctx* c = r->c;
  const bool bcast = r->n_shards != 1 && comm_matches(c, r->shard, r->n_shards);
  // with a communicator the written word is rank 0's, broadcast over NVLink: the other ranks may pass NULL
  if (!w && !(bcast && r->shard != 0)) return fail(FHERAM_ERR_INVALID, "null argument");
  if (addr->c != c || k->c != c) return fail(FHERAM_ERR_INVALID, "handles belong to different contexts");
  if (!r->state)
    return fail(FHERAM_ERR_NOT_READY, "invalid call to Memory.write: internal state is false -> requires calling Memory.read_prepare_write (src/ram.rs:555-558)");
  CU(cudaSetDevice(c->device));
  const Derived& d = c->d;
  const int ws = c->params.word_size, nl = r->n_local;
  const long L = c->ct_stride();
  const int per = ws * nl;
  TRY(r->wbuf.ensure(sizeof(int) * (size_t)ws * L));
  if (!bcast || r->shard == 0) {
    // staged through a buffer of its own and not waited for: the copy out of pageable memory returns once the
    // host data is staged, the conversion is ordered on the stream
    TRY(r->wstage.ensure(sizeof(long long) * (size_t)ws * L));
    // through a pinned buffer of the RAM handle: the caller's words may be freed as soon as the call returns
    const size_t wbytes = sizeof(long long) * (size_t)ws * L;
    if (!r->wpin) {
      CU(cudaMallocHost(&r->wpin, wbytes));
      CU(cudaEventCreateWithFlags(&r->wcopied, cudaEventDisableTiming));
    } else {
      CU(cudaEventSynchronize(r->wcopied));  // the previous write's copy out of the buffer (long done)
    }
    memcpy(r->wpin, w, wbytes);
    CU(cudaMemcpyAsync(r->wstage.p, r->wpin, wbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaEventRecord(r->wcopied, c->stream));
    k_i64_to_i32<<<c->sm_count, 256, 0, c->stream>>>((const long long*)r->wstage.p, (int*)r->wbuf.p, (size_t)ws * L, c->d_err);
    c->launches++;
  }
  if (bcast) NC(ncclBroadcast(r->wbuf.p, r->wbuf.p, (size_t)ws * L, ncclInt32, 0, c->comm, c->stream));
  TRY(r->bufA.ensure(sizeof(int) * (size_t)per * L));
  TRY(r->bufB.ensure(sizeof(int) * (size_t)per * L));
  int* A = (int*)r->bufA.p;
  int* Bb = (int*)r->bufB.p;
  // GGSW(X^-digit) -> GGSW(X^+digit) for all digits of the address (src/ram.rs:265-271,283-289)
  TRY(address_prepare_inv(addr, k));
  // write_first_step (src/ram.rs:544-577): to = to - TRACE(to) + w, normalised
  int* to = d.n_coord != 1 ? r->tree : r->data;  // n2 == 1: data[0] of every sub-RAM
  if (d.n_coord == 1) {
    // data holds one polynomial per sub-RAM (n_local == 1)
    TRY(run_trace_chain(c, k, ws, r->data, nullptr, 0, 0, A, 0, d.log_n));
    k_sub_add_normalize<<<c->sm_count * 4, 256, 0, c->stream>>>(to, A, (const int*)r->wbuf.p, 0, ws, L);
    c->launches++;
  } else {
    TRY(run_trace_chain(c, k, ws, r->tree, nullptr, 0, 0, A, 0, d.log_n));
    k_sub_add_normalize<<<c->sm_count * 4, 256, 0, c->stream>>>(to, A, (const int*)r->wbuf.p, 0, ws, L);
    c->launches++;
    // write_mid_step (src/ram.rs:579-632), i = 0
    const int c1 = first_coord_ggsw(d, 1);
    const double2* inv1 = addr->inv_prep + (size_t)c1 * c->ggsw_prep_len();
    TRY(run_ext_chain(c, ws, r->tree, nullptr, 0, r->tree, inv1, d.coord_len[1], 0, 0));  // :610
    // T1[h] = TRACE(data[h]) (:616);  T2[h] = TRACE(ct_lo * X^-h) (:621,629), h = shard + S*h'
    TRY(run_trace_chain(c, k, per, r->data, nullptr, 0, 0, A, 0, d.log_n));
    TRY(run_trace_chain(c, k, per, r->tree, nullptr, 0, nl, Bb, 0, d.log_n, nl,
                        2 * kN - r->n_shards, (2 * kN - r->shard) % (2 * kN)));
    // data[h] = normalize(data[h] - T1[h] + T2[h])  (:617,625,626)
    k_sub_add_normalize<<<c->sm_count * 8, 256, 0, c->stream>>>(r->data, A, Bb, 0, per, L);
    c->launches++;
    // the reference leaves ct_lo rotated by X^-1 once per polynomial of the chunk (:629)
    k_rotate<<<c->sm_count, 256, 0, c->stream>>>(A, r->tree, (2 * kN - (d.n_glwe % (2 * kN))) % (2 * kN), ws, L);
    c->launches++;
    CU(cudaMemcpyAsync(r->tree, A, sizeof(int) * (size_t)ws * L, cudaMemcpyDeviceToDevice, c->stream));
  }
  // write_last_step (src/ram.rs:634-649): rotate every polynomial back by the first coordinate
  TRY(run_ext_chain(c, per, r->data, nullptr, 0, r->data, addr->inv_prep, d.coord_len[0], 0, 0));
  CU(cudaGetLastError());
  // no host synchronisation: the call returns with the work queued on the context stream, like every *_device entry
  // point; the next call on this RAM is ordered after it, fheram_ctx_synchronize / any download waits for it
  r->state = false;  // src/ram.rs:648
  return 0;
}

// --------------------------------------------------------------------------------------
// op-level entry points
// --------------------------------------------------------------------------------------
extern "C" int fheram_coordinate_product(fheram_ctx* c, const int64_t* in, int n, const int64_t* ggsws,
                                         int n_ggsw, int64_t* out) {
  if (!c || !in || !ggsws || !out || n < 1 || n_ggsw < 1 || n_ggsw > kMaxSteps)
    return fail(FHERAM_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  const long L = c->ct_stride();
  TRY(c->opbuf[0].ensure(sizeof(int) * (size_t)n * L));
  TRY(c->opbuf[1].ensure(sizeof(int) * (size_t)n_ggsw * c->ggsw_raw_len()));
  TRY(c->opbuf[2].ensure(sizeof(double2) * (size_t)n_ggsw * c->ggsw_prep_len()));
  TRY(upload_i64(c, in, (size_t)n * L, (int*)c->opbuf[0].p));
  TRY(upload_i64(c, ggsws, (size_t)n_ggsw * c->ggsw_raw_len(), (int*)c->opbuf[1].p));
  TRY(prepare_ggsw(c, (int*)c->opbuf[1].p, (double2*)c->opbuf[2].p, n_ggsw));
  TRY(run_ext_chain(c, n, (int*)c->opbuf[0].p, nullptr, 0, (int*)c->opbuf[0].p, (double2*)c->opbuf[2].p,
                    n_ggsw, 0, 0));
  return download_i64(c, (int*)c->opbuf[0].p, (size_t)n * L, out);
}
extern "C" int fheram_external_product_batch(fheram_ctx* c, const int64_t* in, int n, const int64_t* ggsw,
                                             int64_t* out) {
  return fheram_coordinate_product(c, in, n, ggsw, 1, out);
}

extern "C" int fheram_glwe_trace(fheram_ctx* c, const fheram_keys* k, const int64_t* in, int n, int start,
                                 int end, int64_t* out) {
  if (!c || !k || !in || !out || n < 1 || start < 0 || end > c->d.log_n || start > end)
    return fail(FHERAM_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  const long L = c->ct_stride();
  TRY(c->opbuf[0].ensure(sizeof(int) * (size_t)n * L));
  TRY(upload_i64(c, in, (size_t)n * L, (int*)c->opbuf[0].p));
  if (end > start) TRY(run_trace_chain(c, k, n, (int*)c->opbuf[0].p, nullptr, 0, 0, (int*)c->opbuf[0].p, start, end));
  return download_i64(c, (int*)c->opbuf[0].p, (size_t)n * L, out);
}

extern "C" int fheram_glwe_pack(fheram_ctx* c, const fheram_keys* k, const int64_t* in, int n, int64_t* out) {
  if (!c || !k || !in || !out || n < 1 || n > kN || (n & (n - 1))) return fail(FHERAM_ERR_INVALID, "n must be a power of two <= N");
  CU(cudaSetDevice(c->device));
  const long L = c->ct_stride();
  TRY(c->opbuf[0].ensure(sizeof(int) * (size_t)n * L));
  TRY(c->opbuf[1].ensure(sizeof(int) * (size_t)n * L));
  TRY(c->opbuf[2].ensure(sizeof(int) * (size_t)n));
  TRY(upload_i64(c, in, (size_t)n * L, (int*)c->opbuf[1].p));
  const int lg = ilog2(n);
  std::vector<int> map(n);
  for (int m = 0; m < n; m++) map[m] = (int)revbits(m, lg);
  CU(cudaMemcpyAsync(c->opbuf[2].p, map.data(), sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  const int one_sided = c->d.log_n - lg;
  int* A = (int*)c->opbuf[0].p;
  TRY(run_trace_chain(c, k, n, (int*)c->opbuf[1].p, (int*)c->opbuf[2].p, n, 0, A, 0, one_sided));
  int* res = nullptr;
  TRY(run_pack_levels(c, k, 1, n, one_sided, A, (int*)c->opbuf[1].p, &res));
  return download_i64(c, res, (size_t)L, out);
}

extern "C" int fheram_glwe_automorphism(fheram_ctx* c, const fheram_keys* k, int gal_idx, int mode, int rsh,
                                        const int64_t* in, int n, int64_t* out) {
  if (!c || !k || !in || !out || n < 1 || gal_idx < 0 || gal_idx >= c->d.log_n || mode < 0 || mode > 2)
    return fail(FHERAM_ERR_INVALID, "bad argument");
  if ((mode == 0) == (rsh != 0)) return fail(FHERAM_ERR_INVALID, "mode 0 runs without rsh, modes 1/2 with rsh=1 (the fused kernels' shapes)");
  CU(cudaSetDevice(c->device));
  const long L = c->ct_stride();
  TRY(c->opbuf[0].ensure(sizeof(int) * (size_t)n * L));
  TRY(c->opbuf[1].ensure(sizeof(int) * (size_t)n * L));
  TRY(upload_i64(c, in, (size_t)n * L, (int*)c->opbuf[0].p));
  int* res = (int*)c->opbuf[0].p;
  if (mode == 0) {
    VmpArgs a = base_args(c, n, (int*)c->opbuf[0].p, (int*)c->opbuf[1].p, L);
    a.n_steps = 1;
    a.mat[0] = k->atk + (size_t)gal_idx * c->atk_prep_len();
    a.gal[0] = (int)((galois(c->d.log_n, gal_idx) + 2 * kN) % (2 * kN));
    a.gal_inv[0] = inv_mod_2n(a.gal[0]);
    TRY(launch(c, KC_OTHER, K_AUTO3, std::min(n, c->sm_count), kThreads, smem_bytes(3), a));
    res = (int*)c->opbuf[1].p;
  } else {
    TRY(run_trace_chain(c, k, n, res, nullptr, 0, 0, res, gal_idx, gal_idx + 1, 0, 0, 0, mode == 1 ? 1 : -1));
  }
  return download_i64(c, res, (size_t)n * L, out);
}

extern "C" int fheram_ggsw_invert(fheram_ctx* c, const fheram_keys* k, const int64_t* ggsw, int n, int64_t* out) {
  if (!c || !k || !ggsw || !out || n < 1) return fail(FHERAM_ERR_INVALID, "bad argument");
  CU(cudaSetDevice(c->device));
  const size_t len = (size_t)n * c->ggsw_raw_len();
  TRY(c->opbuf[0].ensure(sizeof(int) * len));
  TRY(c->opbuf[1].ensure(sizeof(int) * len));
  TRY(upload_i64(c, ggsw, len, (int*)c->opbuf[0].p));
  TRY(ggsw_invert_device(c, k, (int*)c->opbuf[0].p, n, (int*)c->opbuf[1].p));
  return download_i64(c, (int*)c->opbuf[1].p, len, out);
}
