//! Raw bindings to include/fheram.h (hand-written; one line per C entry point the shim uses).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_double, c_int};

#[repr(C)]
#[derive(Clone, Copy)]
pub struct fheram_params {
    pub log_n: i32,
    pub base2k: i32,
    pub k_pt: i32,
    pub k_ct: i32,
    pub k_addr: i32,
    pub k_evk_trace: i32,
    pub k_evk_ggsw_inv: i32,
    pub word_size: i32,
    pub n_decomp: i32,
    pub decomp_n: [i32; 8],
    pub max_addr: u64,
}
/// state of a mask Source: the seed of a seeded ciphertext (include/fheram.h)
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct fheram_seed {
    pub key: [u32; 8],
    pub word0: u64,
}
macro_rules! opaque { ($($n:ident),*) => { $(#[repr(C)] pub struct $n { _p: [u8; 0] })* } }
opaque!(fheram_ctx, fheram_keys, fheram_address, fheram_ram, fheram_source);

extern "C" {
    pub fn fheram_params_default(p: *mut fheram_params);
    pub fn fheram_params_readme(p: *mut fheram_params);
    pub fn fheram_last_error() -> *const c_char;
    pub fn fheram_glwe_len(p: *const fheram_params) -> usize;
    pub fn fheram_ggsw_len(p: *const fheram_params) -> usize;
    pub fn fheram_atk_len(p: *const fheram_params) -> usize;
    pub fn fheram_evk_inv_len(p: *const fheram_params) -> usize;
    pub fn fheram_n_trace_keys(p: *const fheram_params) -> c_int;
    pub fn fheram_n_ggsw(p: *const fheram_params) -> c_int;
    pub fn fheram_n_glwe_per_subram(p: *const fheram_params) -> c_int;
    pub fn fheram_ctx_create(p: *const fheram_params, device: c_int, out: *mut *mut fheram_ctx) -> c_int;
    pub fn fheram_ctx_destroy(c: *mut fheram_ctx) -> c_int;
    pub fn fheram_keys_prepare(c: *mut fheram_ctx, atk: *const i64, tsk: *const i64, inv: *const i64,
                               out: *mut *mut fheram_keys) -> c_int;
    pub fn fheram_keys_destroy(k: *mut fheram_keys) -> c_int;
    // EvaluationKeys::encrypt_sk + prepare on the device (colocated client / server mode), raw keys back on request
    pub fn fheram_keys_encrypt_sk(c: *mut fheram_ctx, sk: *const i64, xa: *mut fheram_source, xe: *mut fheram_source,
                                  out: *mut *mut fheram_keys) -> c_int;
    pub fn fheram_keys_download_raw(k: *mut fheram_keys, atk: *mut i64, tsk: *mut i64, inv: *mut i64) -> c_int;
    // packed host format of normalised limbs (17-bit fields)
    pub fn fheram_pack17(limbs: *const i64, n: usize, packed: *mut u32) -> c_int;
    pub fn fheram_unpack17(packed: *const u32, n: usize, limbs: *mut i64) -> c_int;
    pub fn fheram_ram_read_batch_host_p17(r: *mut fheram_ram, ggsw_packed: *const u32, n: c_int, k: *const fheram_keys,
                                          out_host: *mut i32) -> c_int;
    pub fn fheram_address_load(c: *mut fheram_ctx, ggsw: *const i64, out: *mut *mut fheram_address) -> c_int;
    pub fn fheram_address_load_batch(c: *mut fheram_ctx, ggsw: *const i64, n: c_int, out: *mut *mut fheram_address) -> c_int;
    pub fn fheram_address_destroy(a: *mut fheram_address) -> c_int;
    // batched reads on one resident RAM (BASELINE config 3); `_host` pipelines upload / prepare / read / download
    pub fn fheram_ram_read_batch(r: *mut fheram_ram, a: *const fheram_address, k: *const fheram_keys, out: *mut i64) -> c_int;
    pub fn fheram_ram_read_batch_host(r: *mut fheram_ram, ggsw_host: *const i64, n: c_int, k: *const fheram_keys,
                                      out_host: *mut i64) -> c_int;
    // compact host format (int32 limbs in and out)
    pub fn fheram_ram_read_batch_host_i32(r: *mut fheram_ram, ggsw_host: *const i32, n: c_int, k: *const fheram_keys,
                                          out_host: *mut i32) -> c_int;
    // multi-GPU: NCCL communicator inside the library (one rank per context); on a RAM from
    // fheram_ram_create_sharded(ctx, rank, n_ranks) the read / read_prepare_write / write calls above then do their own
    // exchange steps (see include/fheram.h)
    pub fn fheram_comm_unique_id(id: *mut u8) -> c_int;
    pub fn fheram_comm_init(c: *mut fheram_ctx, n_ranks: c_int, rank: c_int, id: *const u8) -> c_int;
    pub fn fheram_comm_destroy(c: *mut fheram_ctx) -> c_int;
    pub fn fheram_comm_n_ranks(c: *const fheram_ctx) -> c_int;
    pub fn fheram_comm_rank(c: *const fheram_ctx) -> c_int;
    pub fn fheram_ram_create_sharded(c: *mut fheram_ctx, shard: c_int, n_shards: c_int, out: *mut *mut fheram_ram) -> c_int;
    // multi-GPU building blocks (one process per GPU): each rank uploads 1/G of a batch and all-gathers the rest
    pub fn fheram_address_alloc(c: *mut fheram_ctx, n: c_int, out: *mut *mut fheram_address) -> c_int;
    pub fn fheram_address_upload_slice_async(a: *mut fheram_address, ggsw: *const i64, first: c_int, count: c_int) -> c_int;
    pub fn fheram_address_wait_upload(a: *mut fheram_address) -> c_int;
    pub fn fheram_address_release(a: *mut fheram_address) -> c_int;
    pub fn fheram_address_prepare(a: *mut fheram_address) -> c_int;
    pub fn fheram_ram_create(c: *mut fheram_ctx, out: *mut *mut fheram_ram) -> c_int;
    pub fn fheram_ram_destroy(r: *mut fheram_ram) -> c_int;
    pub fn fheram_ram_load(r: *mut fheram_ram, cts: *const i64) -> c_int;
    pub fn fheram_ram_read(r: *mut fheram_ram, a: *const fheram_address, k: *const fheram_keys, out: *mut i64) -> c_int;
    pub fn fheram_ram_read_prepare_write(r: *mut fheram_ram, a: *const fheram_address, k: *const fheram_keys,
                                         out: *mut i64) -> c_int;
    pub fn fheram_ram_write(r: *mut fheram_ram, w: *const i64, a: *const fheram_address, k: *const fheram_keys) -> c_int;
    pub fn fheram_ram_read_plain(r: *mut fheram_ram, addrs: *const u32, n: c_int, k: *const fheram_keys,
                                 out: *mut i64) -> c_int;
    pub fn fheram_ram_read_plain_device(r: *mut fheram_ram, addrs: *const u32, n: c_int, k: *const fheram_keys,
                                        d_out: *mut *const i32) -> c_int;
    pub fn fheram_ram_write_plain(r: *mut fheram_ram, addr: u32, w: *const i64, k: *const fheram_keys) -> c_int;
    pub fn fheram_source_new(seed: *const u8) -> *mut fheram_source;
    pub fn fheram_source_free(s: *mut fheram_source);
    pub fn fheram_source_position(s: *const fheram_source) -> u64;
    pub fn fheram_source_skip(s: *mut fheram_source, n_words: u64);
    pub fn fheram_secret_gen(p: *const fheram_params, xs: *mut fheram_source, sk: *mut i64) -> c_int;
    pub fn fheram_keygen(p: *const fheram_params, sk: *const i64, xa: *mut fheram_source, xe: *mut fheram_source,
                         atk: *mut i64, tsk: *mut i64, inv: *mut i64) -> c_int;
    pub fn fheram_encrypt_ram(p: *const fheram_params, data: *const u8, sk: *const i64, xa: *mut fheram_source,
                              xe: *mut fheram_source, cts: *mut i64) -> c_int;
    pub fn fheram_ram_encrypt_sk(r: *mut fheram_ram, data: *const u8, sk: *const i64, xa: *mut fheram_source,
                                 xe: *mut fheram_source) -> c_int;
    pub fn fheram_address_encrypt_sk(a: *mut fheram_address, first: c_int, count: c_int, values: *const u32,
                                     sk: *const i64, xa: *const *mut fheram_source, xe: *const *mut fheram_source,
                                     n_sources: c_int) -> c_int;
    pub fn fheram_encrypt_address(p: *const fheram_params, value: u32, sk: *const i64, xa: *mut fheram_source,
                                  xe: *mut fheram_source, ggsw: *mut i64) -> c_int;
    pub fn fheram_encrypt_word(p: *const fheram_params, value: u8, sk: *const i64, xa: *mut fheram_source,
                               xe: *mut fheram_source, glwe: *mut i64) -> c_int;
    pub fn fheram_decrypt_word(p: *const fheram_params, glwe: *const i64, sk: *const i64, want: i64,
                               value: *mut i64, noise: *mut c_double) -> c_int;
    // bulk decryption (DESIGN.md 3.7): a whole RAM on the CPU / on the device, coefficient 0 of device-resident GLWEs
    pub fn fheram_decrypt_ram(p: *const fheram_params, cts: *const i64, sk: *const i64, values: *mut i16,
                              err: *mut i64) -> c_int;
    pub fn fheram_ram_decrypt_sk(r: *mut fheram_ram, sk: *const i64, values: *mut i16, err: *mut i64) -> c_int;
    pub fn fheram_decrypt_words_device(c: *mut fheram_ctx, d_glwe: *const i32, n: c_int, sk: *const i64,
                                       values: *mut i16, err: *mut i64) -> c_int;
    // seeded ciphertexts (DESIGN.md 3.6): bodies + the mask Source's seed, masks regenerated on the device
    pub fn fheram_source_seed(s: *const fheram_source, seed: *mut fheram_seed) -> c_int;
    pub fn fheram_encrypt_ram_seeded(p: *const fheram_params, data: *const u8, sk: *const i64, xa: *mut fheram_source,
                                     xe: *mut fheram_source, bodies: *mut i64, seed: *mut fheram_seed) -> c_int;
    pub fn fheram_encrypt_address_seeded(p: *const fheram_params, value: u32, sk: *const i64, xa: *mut fheram_source,
                                         xe: *mut fheram_source, bodies: *mut i64, seed: *mut fheram_seed) -> c_int;
    pub fn fheram_ram_expand(p: *const fheram_params, bodies: *const i64, seed: *const fheram_seed, cts: *mut i64) -> c_int;
    pub fn fheram_address_expand(p: *const fheram_params, bodies: *const i64, seed: *const fheram_seed,
                                 ggsw: *mut i64) -> c_int;
    pub fn fheram_address_load_seeded(c: *mut fheram_ctx, bodies: *const i64, seeds: *const fheram_seed, n: c_int,
                                      out: *mut *mut fheram_address) -> c_int;
    pub fn fheram_ram_read_batch_host_seeded(r: *mut fheram_ram, bodies_p17: *const u32, seeds: *const fheram_seed,
                                             n: c_int, k: *const fheram_keys, out: *mut i32) -> c_int;
    pub fn fheram_ram_load_seeded(r: *mut fheram_ram, bodies: *const i64, seed: *const fheram_seed) -> c_int;
}
