/*
 * fheram.h -- C ABI of libfheram_cuda.so: the B200-native (sm_100a) FHE-RAM hot path.
 *
 * This is the boundary a maintainer of phantomzone-org/fhe-ram binds from Rust (extern "C",
 * see INTEGRATION.md and rust/src/ffi.rs).  Every entry point names the reference item it
 * replaces (paths relative to the reference tree).  All ciphertext data crosses the boundary
 * as signed 64-bit limbs in Poulpy's own container order:
 *
 *   VecZnx(n, cols, size): index ((limb*cols)+col)*n + coeff, limb 0 most significant
 *   GLWE(k)   : cols = 2 (col 0 body, col 1 mask), size = ceil(k / base2k)
 *   GGSW      : [dnum rows][2 cols_in] GLWE(k_addr)     (MatZnx row-major)
 *   GGLWE key : [dnum rows] GLWE(k_key)
 *
 * Device layout is private (int32 limbs, prepared matrices in the kernel's frequency order).
 * Every function returns 0 on success or a negative fheram_status; fheram_last_error() gives
 * the message (the Rust shim panics on non-zero to keep the reference's assert! behaviour).
 * No function falls back to the CPU: without a CUDA device fheram_ctx_create fails.
 */
#ifndef FHERAM_H
#define FHERAM_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum fheram_status {
  FHERAM_OK = 0,
  FHERAM_ERR_INVALID = -1,    /* bad argument / unsupported parameter set */
  FHERAM_ERR_STATE = -2,      /* read while prepared-for-write (src/ram.rs:393-396,472-475) */
  FHERAM_ERR_NOT_READY = -3,  /* write without read_prepare_write (src/ram.rs:555-558) */
  FHERAM_ERR_UNINIT = -4,     /* uninitialised memory (src/ram.rs:182-185,206-209) */
  FHERAM_ERR_CUDA = -5,       /* CUDA runtime failure or no device */
  FHERAM_ERR_RANGE = -6       /* limb outside the int32 device range */
} fheram_status;

/* src/parameters.rs:11-21 (compile-time consts there; runtime here, SURVEY.md 0.4) */
typedef struct fheram_params {
  int32_t log_n;          /* LOG_N = 12 (only value supported by the kernels) */
  int32_t base2k;         /* BASE2K = 17 */
  int32_t k_pt;           /* K_GLWE_PT: snapshot 3, README 9 */
  int32_t k_ct;           /* K_GLWE_CT = 51 */
  int32_t k_addr;         /* K_GGSW_ADDR = 68 */
  int32_t k_evk_trace;    /* K_EVK_TRACE = 68 */
  int32_t k_evk_ggsw_inv; /* K_EVK_GGSW_INV = 85 */
  int32_t word_size;      /* WORDSIZE */
  int32_t n_decomp;       /* DECOMP_N */
  int32_t decomp_n[8];
  uint64_t max_addr;      /* MAX_ADDR */
} fheram_params;

/* Parameters::new() (src/parameters.rs:167-176): the snapshot's defaults */
void fheram_params_default(fheram_params *p);
/* README.md:17-34 parameter set (MAX_ADDR = 2^18, K_PT = 9): BASELINE.json's workload */
void fheram_params_readme(fheram_params *p);

const char *fheram_last_error(void);
const char *fheram_version(void);

/* ---- sizes, in int64 limbs (GLWE::bytes_of_from_infos & friends) ---- */
size_t fheram_glwe_len(const fheram_params *p);      /* one GLWE(k_ct) */
size_t fheram_ggsw_len(const fheram_params *p);      /* one GGSW(k_addr, dnum_ct) */
size_t fheram_atk_len(const fheram_params *p);       /* one trace automorphism key */
size_t fheram_evk_inv_len(const fheram_params *p);   /* atk_ggsw_inv or tsk_ggsw_inv */
int fheram_n_trace_keys(const fheram_params *p);     /* log_n */
int fheram_n_ggsw(const fheram_params *p);           /* GGSWs per Address (Base2D digits) */
int fheram_n_glwe_per_subram(const fheram_params *p);/* ceil(max_addr / n), src/ram.rs:358-360 */
/* get_base_2d (src/base.rs:84-108): returns #coordinates, lens[c] = digits of coordinate c,
 * digits[c*8 + d] = bit width of digit d */
int fheram_base2d(const fheram_params *p, int32_t lens[8], int32_t digits[64]);
/* GLWE::trace_galois_elements()[i] (keys of EvaluationKeys::atk_glwe, src/keys.rs:158) */
int64_t fheram_trace_galois_element(const fheram_params *p, int i);

/* ---- device context: Module::<B>::new(1 << LOG_N) + ScratchOwned (src/parameters.rs:40,
 * src/ram.rs:61): FFT tables and work arenas on one GPU ---- */
typedef struct fheram_ctx fheram_ctx;
int fheram_ctx_create(const fheram_params *p, int device, fheram_ctx **out);
int fheram_ctx_destroy(fheram_ctx *ctx);
int fheram_ctx_synchronize(fheram_ctx *ctx);
/* CUDA stream the context launches on (cudaStream_t), for event timing by the caller */
void *fheram_ctx_stream(fheram_ctx *ctx);
/* number of kernels launched by this context so far */
uint64_t fheram_ctx_launch_count(const fheram_ctx *ctx);

/* measurement: CUDA-event timing of every vmp-class launch on the context stream.
 * classes: 0 external-product chain, 1 key-switch (trace / one-sided combine) chain,
 * 2 two-sided packer combine, 3 other.  ops = sum over launches of items x chain steps. */
int fheram_ctx_profile(fheram_ctx *ctx, int enable);
int fheram_ctx_profile_get(fheram_ctx *ctx, double ms[4], uint64_t launches[4], uint64_t ops[4]);
/* per-launch records of the profiled region in launch order (class, device ms, items, chain
 * steps); returns the number of records written (<= max_n) */
int fheram_ctx_profile_records(fheram_ctx *ctx, int max_n, int *cls, double *ms, uint64_t *items,
                               uint64_t *steps);
/* FP64 FMA peak of the device in TFLOP/s (dependent-chain DFMA probe, best of reps) */
int fheram_fp64_peak_probe(fheram_ctx *ctx, int reps, double *tflops);
/* debug: per-phase SM-cycle counters of the fused kernels, summed over CTAs.  enable = 1 starts
 * counting, enable = 0 reads {prologue, forward pass 1, forward warp passes, contraction, inverse
 * transform, epilogue, rest, -} into out and stops. */
int fheram_debug_phase_cycles(fheram_ctx *ctx, int enable, long long out[8]);
/* debug: bytes of device memory the library holds right now, over every context, handle and device
 * of the process (a leak check that does not depend on other users of the GPU) */
uint64_t fheram_debug_device_bytes(void);
/* pin / unpin a caller-owned host buffer (cudaHostRegister) so uploads run at PCIe speed */
int fheram_host_register(void *p, size_t bytes);
int fheram_host_unregister(void *p);

/* ---- EvaluationKeysPrepared::alloc + ::prepare (src/keys.rs:34-71): uploads the raw keys and
 * runs vmp_prepare on the device; atk_glwe = the log_n trace keys in
 * fheram_trace_galois_element order, tsk = GGLWEToGGSWKey, atk_inv = automorphism key p=-1 */
typedef struct fheram_keys fheram_keys;
int fheram_keys_prepare(fheram_ctx *ctx, const int64_t *atk_glwe, const int64_t *tsk,
                        const int64_t *atk_inv, fheram_keys **out);
int fheram_keys_destroy(fheram_keys *k);

/* ---- Address (src/address.rs:21-24) resident on the device together with its
 * CoordinatePrepared form (src/coordinate_prepared.rs:104-116; prepared once instead of once per
 * sub-RAM per call as src/ram.rs:416-419 does).  ggsw = fheram_n_ggsw GGSWs, coordinate-major. */
typedef struct fheram_address fheram_address;
int fheram_address_load(fheram_ctx *ctx, const int64_t *ggsw, fheram_address **out);
/* n addresses at once, stored contiguously (batched reads) */
int fheram_address_load_batch(fheram_ctx *ctx, const int64_t *ggsw, int n, fheram_address **out);
/* multi-GPU upload path: allocate n addresses on the device, upload this rank's slice from the
 * host, let the caller all-gather the other slices over NVLink straight into the raw int32 buffer
 * (fheram_address_raw_ptr: [n][n_ggsw][ggsw_len] int32), then prepare all of them on the device */
int fheram_address_alloc(fheram_ctx *ctx, int n, fheram_address **out);
int32_t *fheram_address_raw_ptr(fheram_address *a);
int fheram_address_upload_slice(fheram_address *a, const int64_t *ggsw, int first, int count);
int fheram_address_prepare(fheram_address *a);
/* pipelined variant: the copy (from pinned / registered host memory) and the int64 -> int32 conversion run
 * on a copy stream; _wait_upload orders the compute stream after them; _release is recorded on the compute
 * stream after the last use of this address set so that the next _upload_slice_async into it may start.
 * A limb outside +-2^30 is reported by the next synchronous call (error flag on the device). */
int fheram_address_upload_slice_async(fheram_address *a, const int64_t *ggsw, int first, int count);
int fheram_address_wait_upload(fheram_address *a);
int fheram_address_release(fheram_address *a);
int fheram_address_count(const fheram_address *a);
int fheram_address_destroy(fheram_address *a);

/* ---- Ram (src/ram.rs:25-29) ---- */
typedef struct fheram_ram fheram_ram;
/* Ram::new / Ram::new_from_ram_params (src/ram.rs:59-87): sizes come from the ctx params */
int fheram_ram_create(fheram_ctx *ctx, fheram_ram **out);
int fheram_ram_destroy(fheram_ram *r);
/* installs the result of Ram::encrypt_sk (src/ram.rs:129-167): [word_size][n_glwe] GLWE */
int fheram_ram_load(fheram_ram *r, const int64_t *cts);
/* downloads the current SubRam::data of every sub-RAM in the same order */
int fheram_ram_store(fheram_ram *r, int64_t *cts);
/* downloads tree.last()[0] of every sub-RAM ([word_size] GLWE) */
int fheram_ram_tree_store(fheram_ram *r, int64_t *cts);
int fheram_ram_state(const fheram_ram *r); /* SubRam::state (src/ram.rs:302) */

/* Ram::read (src/ram.rs:172-191): out = [word_size] GLWE on the host */
int fheram_ram_read(fheram_ram *r, const fheram_address *addr, const fheram_keys *k, int64_t *out);
/* Ram::read_prepare_write (src/ram.rs:196-222) */
int fheram_ram_read_prepare_write(fheram_ram *r, const fheram_address *addr, const fheram_keys *k,
                                  int64_t *out);
/* Ram::write (src/ram.rs:226-294): w = [word_size] GLWE encrypting [w_i, 0, ..., 0] */
int fheram_ram_write(fheram_ram *r, const int64_t *w, const fheram_address *addr,
                     const fheram_keys *k);
/* n independent Ram::read calls against the same RAM (BASELINE.json config 3): addr holds n
 * addresses (fheram_address_load_batch); out = [n][word_size] GLWE */
int fheram_ram_read_batch(fheram_ram *r, const fheram_address *addr, const fheram_keys *k,
                          int64_t *out);
/* same, straight from HOST buffers (the reference-facing batch call): ggsw = n addresses as int64
 * limbs (pinned memory recommended, fheram_host_register), out = [n][word_size] GLWE.  Upload,
 * on-device prepare, read and download are pipelined in chunks (copy of chunk k+1 overlaps the
 * reads of chunk k). */
int fheram_ram_read_batch_host(fheram_ram *r, const int64_t *ggsw, int n, const fheram_keys *k,
                               int64_t *out);
/* compact host format: the same limbs as int32 (normalised base-2^17 digits need 17 bits; Poulpy's containers hold
 * them as int64): half the bytes over PCIe in both directions and no conversion pass.  Not range checked. */
int fheram_ram_read_batch_host_i32(fheram_ram *r, const int32_t *ggsw, int n, const fheram_keys *k,
                                   int32_t *out);
/* packed host format: addresses as a little-endian stream of 17-bit two's-complement fields (limb i = bits
 * [17 i, 17 i + 17); fheram_pack17 below), 2.125 bytes per limb: what keeps 8 GPUs fed over one host's PCIe;
 * results as int32 limbs */
int fheram_ram_read_batch_host_p17(fheram_ram *r, const uint32_t *ggsw_packed, int n, const fheram_keys *k,
                                   int32_t *out);
/* host-side packing / unpacking of normalised limbs (n a multiple of 32, packed = n * 17 / 32 words);
 * fheram_pack17 fails with FHERAM_ERR_RANGE on a limb outside [-2^16, 2^16) */
int fheram_pack17(const int64_t *limbs, size_t n, uint32_t *packed);
int fheram_unpack17(const uint32_t *packed, size_t n, int64_t *limbs);
/* device-resident variant: result left in the RAM's result arena (int32 device limbs,
 * [n][word_size][limb][col][N]); returns the device pointer.  No host copies. */
int fheram_ram_read_batch_device(fheram_ram *r, const fheram_address *addr, const fheram_keys *k,
                                 const int32_t **d_out);
/* convert + copy a device result arena to host int64 limbs */
int fheram_download_glwe(fheram_ctx *ctx, const int32_t *d_in, int n_glwe, int64_t *out);

/* ---- reads and writes at plaintext addresses (DESIGN.md 3.8).  The address, and so the polynomial that is read or
 * changed, is disclosed to the server by design: never use these calls for an address that must stay private.  The
 * words stay encrypted and the RAM stays a valid RAM for every oblivious call.  Definitions:
 *   rot(k, x) is glwe_rotate: x X^k, with k taken mod 2N.  It is an exact signed permutation of the limbs, with no
 *     normalisation.
 *   TRACE(x) is glwe_trace(0, log_n), the trace at the end of every read (src/ram.rs:457).
 *   data[s][h] is polynomial h of sub-RAM s as fheram_ram_store lays it out.
 *   For an address a < max_addr: h = a >> log_n and j = a & (N - 1).
 *   read_plain: out[b][s] = TRACE(rot(2N - j_b, data[s][h_b])) for every address b and every sub-RAM s.  It decrypts
 *     to the same value as fheram_ram_read of that address.  The limbs differ, and its noise is one trace's noise.
 *   write_plain with w = [word_size] GLWE, as fheram_ram_write takes it (encrypting [w_s, 0, ..., 0]):
 *     T_s = TRACE(rot(2N - j, data[s][h]))
 *     data[s][h] <- normalize(data[s][h] - rot(j, T_s) + rot(j, w_s))
 *     The sum is exact in integers.  It is normalised once, as k_sub_add_normalize does: balanced base-2^17 digits,
 *     top carry dropped.  This is the reference's write_first_step (to - TRACE(to) + w, src/ram.rs:574-576) applied to
 *     polynomial h seen from coefficient j.  Other polynomials, tree[0][0] and the state flag are untouched; a
 *     write_plain adds one trace's key-switch noise to the N cells of polynomial h in each sub-RAM.
 * Refusals: FHERAM_ERR_INVALID for an address >= max_addr, n < 1, null arguments or handles from another context;
 * FHERAM_ERR_UNINIT for a RAM never loaded; FHERAM_ERR_STATE for a RAM prepared for write or left rotated by
 * fheram_ram_rpw_local_device.  These calls neither need nor consume a read_prepare_write.
 * Sharded RAM (polynomial h lives on shard h mod n_shards).  With a communicator every rank passes the same addresses:
 * read_plain returns all n results on every rank (each computed by the rank that holds its polynomial, exchanged as
 * int32 limbs), write_plain takes rank 0's words (the other ranks may pass NULL) and only the holder updates.  Without
 * one, read_plain fills the entries of the addresses this shard holds and leaves the others as passed (zero in the
 * _device arena); write_plain updates if this shard holds h and otherwise returns 0 having done nothing. ---- */
/* out = [n][word_size] GLWE, as fheram_ram_read_batch; duplicate addresses are allowed */
int fheram_ram_read_plain(fheram_ram *r, const uint32_t *addrs, int n, const fheram_keys *k, int64_t *out);
/* the n results in the RAM's device arena, [n][word_size][limb][col][N] int32, valid until the next call on the RAM */
int fheram_ram_read_plain_device(fheram_ram *r, const uint32_t *addrs, int n, const fheram_keys *k,
                                 const int32_t **d_out);
/* returns with its work queued, like fheram_ram_write; the words are copied out of w before it returns */
int fheram_ram_write_plain(fheram_ram *r, uint32_t addr, const int64_t *w, const fheram_keys *k);

/* ---- multi-GPU (SURVEY.md 8e; the reference's caller makes ONE call per read / read_prepare_write / write,
 * src/ram.rs:172-176,196-200,226-231, and so does the caller here): one context per GPU and rank, an NCCL
 * communicator over NVLink inside the library.  Rank 0 draws the id, the host program hands the 128 bytes to the
 * other ranks (MPI_Bcast, a TCP store, a file), every rank calls fheram_comm_init on its context and creates its RAM
 * with fheram_ram_create_sharded(ctx, rank, n_ranks).  From then on, on such a RAM:
 *   fheram_ram_read_batch_host[_i32]   every rank passes ITS n addresses and receives ITS n results (global batch =
 *                                      concatenation over ranks); prepared GGSWs all-gathered, partials all-to-all
 *   fheram_ram_read_batch[_device]     addr = the WHOLE batch on every rank; rank q receives reads [qB/G, (q+1)B/G)
 *   fheram_ram_read_prepare_write      all-gather of the packed partials, result and tree[0][0] on every rank
 *   fheram_ram_write                   the word of rank 0 is broadcast (other ranks may pass NULL); every rank
 *                                      updates its own polynomials
 * Only integer limbs cross the links (never a floating-point reduction), so results are bit-identical to one GPU. */
int fheram_comm_unique_id(uint8_t id[128]);
int fheram_comm_init(fheram_ctx *ctx, int n_ranks, int rank, const uint8_t id[128]);
int fheram_comm_destroy(fheram_ctx *ctx);
int fheram_comm_n_ranks(const fheram_ctx *ctx);
int fheram_comm_rank(const fheram_ctx *ctx);

/* ---- the halves of the sharded calls, for callers that run the exchange themselves (tests emulate the ranks on one
 * GPU with them; fheram_comm_init is not needed): this RAM holds only the polynomials
 * h == shard (mod n_shards) of every sub-RAM.  Local stage: rotate + pack the local slice;
 * partial results ([n][word_size] GLWE, int32 device limbs) are exchanged by the caller
 * (NCCL all-gather) and finished with fheram_ram_read_finish_sharded on every rank. ---- */
int fheram_ram_create_sharded(fheram_ctx *ctx, int shard, int n_shards, fheram_ram **out);
int fheram_ram_read_local_device(fheram_ram *r, const fheram_address *addr, const fheram_keys *k,
                                 const int32_t **d_partial);
/* d_gathered: [n_shards][n_total][word_size] GLWE partials (rank-major); finishes entries
 * [first, first+count) of it: top log2(n_shards) packer levels, second coordinate, trace.
 * Entry i belongs to address addr_first + i of `addr`.  Result in the result arena,
 * [count][word_size] GLWE. */
int fheram_ram_read_finish_device(fheram_ram *r, const int32_t *d_gathered, int n_total,
                                  int first, int count, const fheram_address *addr,
                                  int addr_first, const fheram_keys *k, const int32_t **d_out);

/* read_prepare_write on a (possibly sharded) RAM, device-resident.  rpw_local rotates the local
 * polynomials in place (src/ram.rs:502-504) and packs them; after the all-gather every rank calls
 * rpw_finish (replicated: every rank keeps tree[0][0], so Ram::write needs no communication).
 * On a single GPU: d_gathered = the pointer rpw_local returned. */
int fheram_ram_rpw_local_device(fheram_ram *r, const fheram_address *addr, const fheram_keys *k,
                                const int32_t **d_partial);
int fheram_ram_rpw_finish_device(fheram_ram *r, const int32_t *d_gathered,
                                 const fheram_address *addr, const fheram_keys *k,
                                 const int32_t **d_out);

/* ---- op-level entry points (BASELINE.json config 2 and kernel parity tests) ---- */
/* n x glwe_external_product(res, a, ggsw) against ONE GGSW (coordinate_prepared.rs:156) */
int fheram_external_product_batch(fheram_ctx *ctx, const int64_t *glwe_in, int n,
                                  const int64_t *ggsw, int64_t *out);
/* CoordinatePrepared::product with n_ggsw digits on n ciphertexts */
int fheram_coordinate_product(fheram_ctx *ctx, const int64_t *glwe_in, int n, const int64_t *ggsws,
                              int n_ggsw, int64_t *out);
/* glwe_trace(start, end) on n ciphertexts (src/ram.rs:457,540,572,616,621) */
int fheram_glwe_trace(fheram_ctx *ctx, const fheram_keys *k, const int64_t *in, int n, int start,
                      int end, int64_t *out);
/* GLWEPacker: add(Some(in[rev(j)])) for rev(j) < n else add(None), then flush
 * (src/ram.rs:424-449); any 1 <= n <= N (the read schedule of a RAM with n polynomials per sub-RAM, including its
 * mixed level when n is not a power of two).  Coefficient h of out = coefficient 0 of in[h] */
int fheram_glwe_pack(fheram_ctx *ctx, const fheram_keys *k, const int64_t *in, int n, int64_t *out);
/* glwe_automorphism (mode 0) / _add (1) / _sub_negate (2) with trace key gal_idx, after an
 * optional glwe_rsh(1) (rsh != 0): n ciphertexts */
int fheram_glwe_automorphism(fheram_ctx *ctx, const fheram_keys *k, int gal_idx, int mode, int rsh,
                             const int64_t *in, int n, int64_t *out);
/* CoordinatePrepared::prepare_inv raw result: GGSW(X^i) -> GGSW(X^-i) (coordinate_prepared.rs:
 * 121-142) on n GGSWs */
int fheram_ggsw_invert(fheram_ctx *ctx, const fheram_keys *k, const int64_t *ggsw, int n,
                       int64_t *out);

/* ---- client side (CPU, src/keys.rs:135-180, src/ram.rs:129-167, src/address.rs:86-109,
 * examples/fhe-ram.rs:179-237).  fheram_source stands in for poulpy_hal::source::Source. ---- */
typedef struct fheram_source fheram_source;
fheram_source *fheram_source_new(const uint8_t seed[32]);
void fheram_source_free(fheram_source *s);
uint32_t fheram_source_next_u32(fheram_source *s);
void fheram_source_fill_bytes(fheram_source *s, uint8_t *out, size_t n);
/* position in the stream, in 32-bit words drawn so far, and a seek forward (the stream is counter based): what lets
 * the device regenerate a Source's draws (fheram_ram_encrypt_sk) and a rank skip the draws of another rank */
uint64_t fheram_source_position(const fheram_source *s);
void fheram_source_skip(fheram_source *s, uint64_t n_words);
/* GLWESecret::fill_ternary_prob(0.5): sk = n coefficients in {-1,0,1} */
int fheram_secret_gen(const fheram_params *p, fheram_source *xs, int64_t *sk);
/* EvaluationKeys::encrypt_sk (src/keys.rs:135-180) */
int fheram_keygen(const fheram_params *p, const int64_t *sk, fheram_source *xa, fheram_source *xe,
                  int64_t *atk_glwe, int64_t *tsk, int64_t *atk_inv);
/* Ram::encrypt_sk (src/ram.rs:129-167): data = max_addr*word_size bytes */
int fheram_encrypt_ram(const fheram_params *p, const uint8_t *data, const int64_t *sk,
                       fheram_source *xa, fheram_source *xe, int64_t *cts);
/* Address::encrypt_sk (src/address.rs:86-109) */
int fheram_encrypt_address(const fheram_params *p, uint32_t value, const int64_t *sk,
                           fheram_source *xa, fheram_source *xe, int64_t *ggsw);
/* examples/fhe-ram.rs:179-210 encrypt_glwe: GLWE of [value, 0, ..., 0] at precision k_pt */
int fheram_encrypt_word(const fheram_params *p, uint8_t value, const int64_t *sk,
                        fheram_source *xa, fheram_source *xe, int64_t *glwe);
/* examples/fhe-ram.rs:212-237 decrypt_glwe: coefficient 0, rounded to k_pt bits, and the
 * log2 noise relative to `want` */
int fheram_decrypt_word(const fheram_params *p, const int64_t *glwe, const int64_t *sk,
                        int64_t want, int64_t *value, double *noise);

/* ---- bulk encryption on the device (SURVEY.md 8(f).1).  For colocated client / server set-ups (tests,
 * benchmarks, loaders that hold the secret): the mask comes from the Source's ChaCha20 stream regenerated on
 * the GPU (k_glwe_encrypt), the product with the secret and the normalization run on the GPU; the noise is
 * sampled on the GPU too (k_noise_sample) and the host re-draws the rare samples whose rounding or rejection
 * could depend on libm's last bit (about one in 10^8).
 * Limb for limb what fheram_encrypt_ram / fheram_encrypt_address produce from the same Sources, and both
 * Sources are left where those calls would leave them. ---- */
/* Ram::encrypt_sk (src/ram.rs:129-167, SubRam::encrypt_sk :334-380) straight into the device RAM (a
 * sharded RAM encrypts its own polynomials); data = max_addr*word_size bytes */
int fheram_ram_encrypt_sk(fheram_ram *r, const uint8_t *data, const int64_t *sk, fheram_source *xa,
                          fheram_source *xe);
/* Address::encrypt_sk (src/address.rs:86-109, Coordinate::encrypt_sk src/coordinate.rs:121-180) for
 * addresses [first, first + count) of a set from fheram_address_alloc; follow with fheram_address_prepare.
 * n_sources = 1: every address draws from (xa[0], xe[0]) in turn; n_sources = count: one pair per address */
int fheram_address_encrypt_sk(fheram_address *a, int first, int count, const uint32_t *values,
                              const int64_t *sk, fheram_source *const *xa, fheram_source *const *xe,
                              int n_sources);
/* EvaluationKeys::encrypt_sk (src/keys.rs:135-180) + EvaluationKeysPrepared::prepare (:57-71) on the device: the
 * limbs of fheram_keygen from the same Sources, prepared and resident; fheram_keys_download_raw gives the raw keys
 * back in fheram_keygen's layout */
int fheram_keys_encrypt_sk(fheram_ctx *ctx, const int64_t *sk, fheram_source *xa, fheram_source *xe,
                           fheram_keys **out);
int fheram_keys_download_raw(fheram_keys *k, int64_t *atk_glwe, int64_t *tsk, int64_t *atk_inv);
/* out = {noise draws sampled on the device, draws re-drawn by the host, streams sampled by the host} so far */
int fheram_debug_encrypt_stats(fheram_ctx *ctx, uint64_t out[3]);

/* ---- bulk decryption (DESIGN.md 3.7).  One definition for every entry point, per GLWE(k_ct) of S limbs:
 *   pt = normalize(body + mask * s)  (balanced base-2^K digits, top carry dropped, as fheram_decrypt_word)
 *   v = (sum_j pt_j 2^(K(S-1-j))) >> (S K - k_ct),  ls = k_ct - k_pt
 *   value_raw = round_half_away(v / 2^ls)   (fheram_decrypt_word's value)
 *   value = value_raw reduced into [-2^(k_pt-1), 2^(k_pt-1)),  err = v - value_raw 2^ls  (exact)
 * fheram_decrypt_word's noise against want = value_raw is log2|err| - k_ct.  For a stored byte b,
 * value == cast_u8_to_signed(b, min(8, k_pt)).  err may be NULL; sk must be ternary. ---- */
/* CPU, all host threads: every byte of a RAM in fheram_encrypt_ram / fheram_ram_store's layout.  values / err =
 * [max_addr][word_size] (byte i of word j at j * word_size + i, the inverse of Ram::encrypt_sk's data) */
int fheram_decrypt_ram(const fheram_params *p, const int64_t *cts, const int64_t *sk, int16_t *values, int64_t *err);
/* the same numbers from the resident RAM on the device, bit for bit.  A sharded RAM fills the entries of its own
 * polynomials (h == shard mod n_shards) and leaves the others as passed.  FHERAM_ERR_UNINIT: never loaded or
 * encrypted; FHERAM_ERR_STATE: prepared for write (read_prepare_write without its write) */
int fheram_ram_decrypt_sk(fheram_ram *r, const int64_t *sk, int16_t *values, int64_t *err);
/* coefficient 0 of n device-resident GLWE(k_ct) in the int32 layout [n][limb][col][N] (e.g. the arena of
 * fheram_ram_read_batch_device, n = reads x word_size); values / err = [n] */
int fheram_decrypt_words_device(fheram_ctx *ctx, const int32_t *d_glwe, int n, const int64_t *sk, int16_t *values,
                                int64_t *err);

/* ---- seeded ciphertexts (DESIGN.md 3.6): the body columns plus the state of the mask Source, half the bytes of the
 * limbs.  A seed is the mask Source before the first mask draw of the object.  Mask coefficient i of limb l of GLWE j
 * of the object is the low base2k bits, sign-extended, of stream word word0 + 2 ((j S + l) N + i) (S = the GLWE's
 * limb count): what fheram_encrypt_ram / fheram_encrypt_address draw.  Bodies are the body columns in Poulpy's order
 * with the column dropped:
 *   RAM      [word_size][n_glwe][size_ct][N], GLWE j = s n_glwe + h, one seed for the whole RAM;
 *   address  [n_ggsw][dnum_ct][2 ci][size_addr][N], GLWE j = (g dnum_ct + r) 2 + ci, one seed per address.
 * A seeded RAM expands to exactly the limbs of fheram_encrypt_ram from the same Sources.  A seeded address is a
 * different, equally valid encryption: the plaintext +/-X^pos of the rows with ci = 1, which fheram_encrypt_address
 * adds to the mask, is moved into the body (body = normalize(-a s + e + X^pos s), mask = a), so that the mask is the
 * raw stream.  Every row has the phase and the noise of fheram_encrypt_address's row, bit for bit, but reads with a
 * seeded address give other limbs than reads with the full one; they decrypt to the same values.
 * A seed discloses every draw of its Source: the mask Source of a seeded object must serve mask draws only. ---- */
typedef struct fheram_seed {
  uint32_t key[8];
  uint64_t word0;
} fheram_seed;
/* the seed of a Source's current position */
int fheram_source_seed(const fheram_source *s, fheram_seed *seed);
/* Ram::encrypt_sk as bodies + seed: bodies = the body columns of fheram_encrypt_ram from the same Sources, which are
 * left where it leaves them.  xa != xe */
int fheram_encrypt_ram_seeded(const fheram_params *p, const uint8_t *data, const int64_t *sk, fheram_source *xa,
                              fheram_source *xe, int64_t *bodies, fheram_seed *seed);
/* Address::encrypt_sk as bodies + seed (the ci = 1 rows carry their plaintext in the body, see above); both Sources
 * are left where fheram_encrypt_address leaves them.  xa != xe */
int fheram_encrypt_address_seeded(const fheram_params *p, uint32_t value, const int64_t *sk, fheram_source *xa,
                                  fheram_source *xe, int64_t *bodies, fheram_seed *seed);
/* CPU expansion to full limbs (the reference of the device expansion): cts in fheram_encrypt_ram's layout, ggsw in
 * fheram_encrypt_address's */
int fheram_ram_expand(const fheram_params *p, const int64_t *bodies, const fheram_seed *seed, int64_t *cts);
int fheram_address_expand(const fheram_params *p, const int64_t *bodies, const fheram_seed *seed, int64_t *ggsw);
/* n seeded addresses made resident and prepared, as fheram_address_load_batch: bodies = n addresses' bodies one
 * after the other, seeds = [n]; the masks are regenerated on the device (k_glwe_expand) */
int fheram_address_load_seeded(fheram_ctx *ctx, const int64_t *bodies, const fheram_seed *seeds, int n,
                               fheram_address **out);
/* fheram_ram_read_batch_host_p17 with seeded addresses: bodies_p17 = the n addresses' bodies packed as fheram_pack17
 * packs limbs (half the bytes of the _p17 format), seeds = [n]; results as int32 limbs.  A sharded RAM follows the
 * contract of the _p17 call: every rank passes its own addresses and receives its own results */
int fheram_ram_read_batch_host_seeded(fheram_ram *r, const uint32_t *bodies_p17, const fheram_seed *seeds, int n,
                                      const fheram_keys *k, int32_t *out);
/* fheram_ram_load of a seeded RAM (bodies in the RAM layout above); a sharded RAM loads its own polynomials */
int fheram_ram_load_seeded(fheram_ram *r, const int64_t *bodies, const fheram_seed *seed);

#ifdef __cplusplus
}
#endif
#endif /* FHERAM_H */
