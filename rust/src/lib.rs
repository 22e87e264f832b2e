//! `fhe-ram` drop-in over the B200 library: same public names as the reference
//! (`Parameters`, `EvaluationKeys[Prepared]`, `Address`, `Ram`, README's `gen_keys`).
//! SOURCE ONLY -- not compiled in this environment (no Rust toolchain).  Failed calls panic with the
//! library's message, which keeps the reference's `assert!` behaviour (src/ram.rs:144-155,182-185,
//! 243,393-396,555-558).
pub mod ffi;
use ffi::*;
use std::ffi::CStr;

fn check(rc: i32) {
    if rc != 0 {
        let msg = unsafe { CStr::from_ptr(fheram_last_error()) }.to_string_lossy().into_owned();
        panic!("{msg}");
    }
}

/// poulpy_hal::source::Source
pub struct Source(*mut fheram_source);
impl Source {
    pub fn new(seed: [u8; 32]) -> Self { Source(unsafe { fheram_source_new(seed.as_ptr()) }) }
}
impl Drop for Source { fn drop(&mut self) { unsafe { fheram_source_free(self.0) } } }

/// src/parameters.rs:147-288 (runtime instead of const parameters)
pub struct Parameters { pub c: fheram_params, ctx: *mut fheram_ctx }
impl Parameters {
    pub fn new() -> Self {
        let mut c = unsafe { std::mem::zeroed() };
        unsafe { fheram_params_default(&mut c) };
        Parameters { c, ctx: std::ptr::null_mut() }
    }
    /// README.md:17-34 parameter set (MAX_ADDR = 2^18, K_PT = 9): BASELINE.json's workload
    pub fn readme() -> Self {
        let mut c = unsafe { std::mem::zeroed() };
        unsafe { fheram_params_readme(&mut c) };
        Parameters { c, ctx: std::ptr::null_mut() }
    }
    /// the runtime overrides of src/ram.rs:72-87 (word_size, decomp_n, max_addr) on top of `new()`
    pub fn with_ram_params(word_size: usize, decomp_n: Vec<u8>, max_addr: usize) -> Self {
        let mut p = Self::new();
        assert!(decomp_n.len() <= 8, "at most 8 digits per coordinate");
        p.c.word_size = word_size as i32;
        p.c.max_addr = max_addr as u64;
        p.c.n_decomp = decomp_n.len() as i32;
        for (i, d) in decomp_n.iter().enumerate() { p.c.decomp_n[i] = *d as i32; }
        p
    }
    pub fn max_addr(&self) -> usize { self.c.max_addr as usize }
    pub fn word_size(&self) -> usize { self.c.word_size as usize }
    pub fn k_glwe_pt(&self) -> u32 { self.c.k_pt as u32 }
    pub fn glwe_len(&self) -> usize { unsafe { fheram_glwe_len(&self.c) } }
    /// Module::<B>::new(1 << LOG_N): the device context
    pub fn module(&mut self) -> *mut fheram_ctx {
        if self.ctx.is_null() { check(unsafe { fheram_ctx_create(&self.c, 0, &mut self.ctx) }); }
        self.ctx
    }
}
impl Drop for Parameters { fn drop(&mut self) { if !self.ctx.is_null() { unsafe { fheram_ctx_destroy(self.ctx); } } } }

pub struct GLWESecret(pub Vec<i64>);
impl GLWESecret {
    pub fn fill_ternary_prob(params: &Parameters, _prob: f64, xs: &mut Source) -> Self {
        let mut sk = vec![0i64; 1 << params.c.log_n];
        check(unsafe { fheram_secret_gen(&params.c, xs.0, sk.as_mut_ptr()) });
        GLWESecret(sk)
    }
}

/// src/keys.rs:21-25
pub struct EvaluationKeys { pub atk_glwe: Vec<i64>, pub gglwe_to_ggsw_key: Vec<i64>, pub atk_ggsw_inv: Vec<i64> }
impl EvaluationKeys {
    /// src/keys.rs:135-180
    pub fn encrypt_sk(params: &Parameters, sk: &GLWESecret, xa: &mut Source, xe: &mut Source) -> Self {
        let p = &params.c;
        let mut k = unsafe {
            EvaluationKeys {
                atk_glwe: vec![0; fheram_n_trace_keys(p) as usize * fheram_atk_len(p)],
                gglwe_to_ggsw_key: vec![0; fheram_evk_inv_len(p)],
                atk_ggsw_inv: vec![0; fheram_evk_inv_len(p)],
            }
        };
        check(unsafe { fheram_keygen(p, sk.0.as_ptr(), xa.0, xe.0, k.atk_glwe.as_mut_ptr(),
                                     k.gglwe_to_ggsw_key.as_mut_ptr(), k.atk_ggsw_inv.as_mut_ptr()) });
        k
    }
}
/// README.md:131
pub fn gen_keys(params: &Parameters) -> (GLWESecret, EvaluationKeys) {
    let (mut xs, mut xa, mut xe) = (Source::new([0; 32]), Source::new([0; 32]), Source::new([0; 32]));
    let sk = GLWESecret::fill_ternary_prob(params, 0.5, &mut xs);
    let evk = EvaluationKeys::encrypt_sk(params, &sk, &mut xa, &mut xe);
    (sk, evk)
}

/// src/keys.rs:27-71
pub struct EvaluationKeysPrepared(*mut fheram_keys);
impl EvaluationKeysPrepared {
    pub fn alloc(_params: &Parameters) -> Self { EvaluationKeysPrepared(std::ptr::null_mut()) }
    /// keygen + prepare on the device (src/keys.rs:135-180, 57-71): same limbs as `EvaluationKeys::encrypt_sk`
    pub fn encrypt_sk_device(params: &mut Parameters, sk: &GLWESecret, xa: &mut Source, xe: &mut Source) -> Self {
        let mut h = std::ptr::null_mut();
        check(unsafe { fheram_keys_encrypt_sk(params.module(), sk.0.as_ptr(), xa.0, xe.0, &mut h) });
        EvaluationKeysPrepared(h)
    }
    pub fn prepare(&mut self, params: &mut Parameters, other: &EvaluationKeys) {
        check(unsafe { fheram_keys_prepare(params.module(), other.atk_glwe.as_ptr(),
                                           other.gglwe_to_ggsw_key.as_ptr(), other.atk_ggsw_inv.as_ptr(), &mut self.0) });
    }
}
impl Drop for EvaluationKeysPrepared { fn drop(&mut self) { if !self.0.is_null() { unsafe { fheram_keys_destroy(self.0); } } } }

/// src/address.rs:21-24.  `seeded`: the bodies and seed of `encrypt_sk_seeded`, uploaded in place of `data`
pub struct Address { pub data: Vec<i64>, pub seeded: Option<(Vec<i64>, fheram_seed)>, dev: *mut fheram_address }
impl Address {
    pub fn alloc_from_params(params: &Parameters) -> Self {
        let n = unsafe { fheram_n_ggsw(&params.c) as usize * fheram_ggsw_len(&params.c) };
        Address { data: vec![0; n], seeded: None, dev: std::ptr::null_mut() }
    }
    pub fn alloc(params: &Parameters) -> Self { Self::alloc_from_params(params) }
    /// src/address.rs:86-109
    pub fn encrypt_sk(&mut self, params: &Parameters, value: u32, sk: &GLWESecret, xa: &mut Source, xe: &mut Source) {
        check(unsafe { fheram_encrypt_address(&params.c, value, sk.0.as_ptr(), xa.0, xe.0, self.data.as_mut_ptr()) });
        self.seeded = None;
        self.drop_device();
    }
    /// the seeded form (include/fheram.h): bodies + the mask Source's seed, half the bytes.  `data` becomes its
    /// expanded limbs, another valid encryption of the same address than `encrypt_sk`'s
    pub fn encrypt_sk_seeded(&mut self, params: &Parameters, value: u32, sk: &GLWESecret, xa: &mut Source,
                             xe: &mut Source) {
        let mut bodies = vec![0i64; self.data.len() / 2];
        let mut seed = fheram_seed::default();
        check(unsafe { fheram_encrypt_address_seeded(&params.c, value, sk.0.as_ptr(), xa.0, xe.0, bodies.as_mut_ptr(),
                                                     &mut seed) });
        check(unsafe { fheram_address_expand(&params.c, bodies.as_ptr(), &seed, self.data.as_mut_ptr()) });
        self.seeded = Some((bodies, seed));
        self.drop_device();
    }
    fn device(&mut self, params: &mut Parameters) -> *const fheram_address {
        if self.dev.is_null() {
            match &self.seeded {
                Some((b, s)) => check(unsafe { fheram_address_load_seeded(params.module(), b.as_ptr(), s, 1, &mut self.dev) }),
                None => check(unsafe { fheram_address_load(params.module(), self.data.as_ptr(), &mut self.dev) }),
            }
        }
        self.dev
    }
    fn drop_device(&mut self) { if !self.dev.is_null() { unsafe { fheram_address_destroy(self.dev); } self.dev = std::ptr::null_mut(); } }
}
impl Drop for Address { fn drop(&mut self) { self.drop_device() } }

/// one GLWE ciphertext as raw limbs (VecZnx order)
pub type GLWE = Vec<i64>;

/// src/ram.rs:25-29
pub struct Ram { pub params: Parameters, h: *mut fheram_ram }
impl Ram {
    /// src/ram.rs:59-69
    pub fn new() -> Self { Self::from_params(Parameters::new()) }
    /// src/ram.rs:72-87
    pub fn new_from_ram_params(word_size: usize, decomp_n: Vec<u8>, max_addr: usize) -> Self {
        Self::from_params(Parameters::with_ram_params(word_size, decomp_n, max_addr))
    }
    /// README.md:116-155 parameter set
    pub fn new_readme() -> Self { Self::from_params(Parameters::readme()) }
    pub fn from_params(mut params: Parameters) -> Self {
        let mut h = std::ptr::null_mut();
        check(unsafe { fheram_ram_create(params.module(), &mut h) });
        Ram { params, h }
    }
    /// multi-GPU: rank `rank` of `n_ranks` (one process per GPU).  `id` = the 128 bytes rank 0 got from
    /// `Ram::comm_unique_id()` and handed to the other ranks (MPI, a TCP store, ...).  read / read_prepare_write /
    /// write keep their signatures; batched reads split the batch over the ranks (include/fheram.h).
    pub fn new_sharded(mut params: Parameters, n_ranks: usize, rank: usize, id: &[u8; 128]) -> Self {
        check(unsafe { fheram_comm_init(params.module(), n_ranks as i32, rank as i32, id.as_ptr()) });
        let mut h = std::ptr::null_mut();
        check(unsafe { fheram_ram_create_sharded(params.module(), rank as i32, n_ranks as i32, &mut h) });
        Ram { params, h }
    }
    pub fn comm_unique_id() -> [u8; 128] {
        let mut id = [0u8; 128];
        check(unsafe { fheram_comm_unique_id(id.as_mut_ptr()) });
        id
    }
    /// src/ram.rs:129-167
    pub fn encrypt_sk(&mut self, data: &[u8], sk: &GLWESecret, xa: &mut Source, xe: &mut Source) {
        let p = &self.params;
        assert!(data.len() % p.word_size() == 0, "invalid data: data.len()%ram_chunks != 0");
        assert!(data.len() / p.word_size() == p.max_addr(), "invalid data: data.len()/ram_chunks != max_addr");
        // on the device, straight into the resident RAM (the limbs fheram_encrypt_ram + fheram_ram_load would install)
        check(unsafe { fheram_ram_encrypt_sk(self.h, data.as_ptr(), sk.0.as_ptr(), xa.0, xe.0) });
    }
    /// `encrypt_sk` on the client (CPU) in the seeded form, then `load_seeded`; returns (bodies, seed), what a
    /// separated client ships: they expand to exactly the limbs of `fheram_encrypt_ram`
    pub fn encrypt_sk_seeded(&mut self, data: &[u8], sk: &GLWESecret, xa: &mut Source, xe: &mut Source)
                             -> (Vec<i64>, fheram_seed) {
        let p = &self.params;
        assert!(data.len() == p.max_addr() * p.word_size(), "invalid data: data.len() != max_addr * ram_chunks");
        let n_glwe = unsafe { fheram_n_glwe_per_subram(&p.c) } as usize;
        let mut bodies = vec![0i64; p.word_size() * n_glwe * p.glwe_len() / 2];
        let mut seed = fheram_seed::default();
        check(unsafe { fheram_encrypt_ram_seeded(&p.c, data.as_ptr(), sk.0.as_ptr(), xa.0, xe.0, bodies.as_mut_ptr(),
                                                 &mut seed) });
        self.load_seeded(&bodies, &seed);
        (bodies, seed)
    }
    /// `fheram_ram_load` of a seeded RAM (a sharded RAM expands its own polynomials)
    pub fn load_seeded(&mut self, bodies: &[i64], seed: &fheram_seed) {
        check(unsafe { fheram_ram_load_seeded(self.h, bodies.as_ptr(), seed) });
    }
    /// n = seeds.len() seeded addresses from host buffers (bodies packed by `fheram_pack17`); int32 limbs out
    pub fn read_batch_host_seeded(&mut self, bodies_p17: &[u32], seeds: &[fheram_seed], keys: &EvaluationKeysPrepared)
                                  -> Vec<i32> {
        let mut out = vec![0i32; seeds.len() * self.params.word_size() * self.params.glwe_len()];
        check(unsafe { fheram_ram_read_batch_host_seeded(self.h, bodies_p17.as_ptr(), seeds.as_ptr(), seeds.len() as i32,
                                                         keys.0, out.as_mut_ptr()) });
        out
    }
    fn split(&self, flat: Vec<i64>) -> Vec<GLWE> { flat.chunks(self.params.glwe_len()).map(|c| c.to_vec()).collect() }
    /// src/ram.rs:172-191
    pub fn read(&mut self, address: &mut Address, keys: &EvaluationKeysPrepared) -> Vec<GLWE> {
        let mut out = vec![0i64; self.params.word_size() * self.params.glwe_len()];
        let a = address.device(&mut self.params);
        check(unsafe { fheram_ram_read(self.h, a, keys.0, out.as_mut_ptr()) });
        self.split(out)
    }
    /// src/ram.rs:196-222
    pub fn read_prepare_write(&mut self, address: &mut Address, keys: &EvaluationKeysPrepared) -> Vec<GLWE> {
        let mut out = vec![0i64; self.params.word_size() * self.params.glwe_len()];
        let a = address.device(&mut self.params);
        check(unsafe { fheram_ram_read_prepare_write(self.h, a, keys.0, out.as_mut_ptr()) });
        self.split(out)
    }
    /// src/ram.rs:226-294
    pub fn write(&mut self, w: &[GLWE], address: &mut Address, keys: &EvaluationKeysPrepared) {
        assert!(w.len() == self.params.word_size());
        let flat: Vec<i64> = w.iter().flatten().copied().collect();
        let a = address.device(&mut self.params);
        check(unsafe { fheram_ram_write(self.h, flat.as_ptr(), a, keys.0) });
    }
    /// reads at plaintext addresses (include/fheram.h): TRACE(data[s][h] X^-j) for a = h N + j, one [word_size] GLWE
    /// per address.  The addresses are disclosed to the server; the words stay encrypted.
    pub fn read_plain(&mut self, addrs: &[u32], keys: &EvaluationKeysPrepared) -> Vec<Vec<GLWE>> {
        let per = self.params.word_size() * self.params.glwe_len();
        let mut out = vec![0i64; addrs.len() * per];
        check(unsafe { fheram_ram_read_plain(self.h, addrs.as_ptr(), addrs.len() as i32, keys.0, out.as_mut_ptr()) });
        out.chunks(per).map(|c| self.split(c.to_vec())).collect()
    }
    /// write at a plaintext address: the write_first_step of Ram::write on polynomial h seen from coefficient j
    pub fn write_plain(&mut self, addr: u32, w: &[GLWE], keys: &EvaluationKeysPrepared) {
        assert!(w.len() == self.params.word_size());
        let flat: Vec<i64> = w.iter().flatten().copied().collect();
        check(unsafe { fheram_ram_write_plain(self.h, addr, flat.as_ptr(), keys.0) });
    }
    /// every byte of the resident RAM decrypted on the device: (values, err), [max_addr][word_size] row-major (byte i of
    /// word j at j * word_size + i); the numbers of `decrypt_ram` on the stored RAM, bit for bit
    pub fn decrypt_sk(&mut self, sk: &GLWESecret) -> (Vec<i16>, Vec<i64>) {
        let len = self.params.max_addr() * self.params.word_size();
        let (mut values, mut err) = (vec![0i16; len], vec![0i64; len]);
        check(unsafe { fheram_ram_decrypt_sk(self.h, sk.0.as_ptr(), values.as_mut_ptr(), err.as_mut_ptr()) });
        (values, err)
    }
}

/// every byte of a RAM in `fheram_encrypt_ram`'s layout ([word_size][n_glwe] GLWE), decrypted on the CPU: (values, err)
/// as `Ram::decrypt_sk` returns them
pub fn decrypt_ram(params: &Parameters, cts: &[i64], sk: &GLWESecret) -> (Vec<i16>, Vec<i64>) {
    let len = params.max_addr() * params.word_size();
    let (mut values, mut err) = (vec![0i16; len], vec![0i64; len]);
    check(unsafe { fheram_decrypt_ram(&params.c, cts.as_ptr(), sk.0.as_ptr(), values.as_mut_ptr(), err.as_mut_ptr()) });
    (values, err)
}

/// coefficient 0 of `n` device-resident GLWE(k_ct) (int32 `[n][limb][col][N]`, e.g. a batched read's result arena),
/// decrypted on the device: (values, err), `n` each
pub fn decrypt_words_device(params: &mut Parameters, d_glwe: *const i32, n: usize, sk: &GLWESecret) -> (Vec<i16>, Vec<i64>) {
    let (mut values, mut err) = (vec![0i16; n], vec![0i64; n]);
    check(unsafe { fheram_decrypt_words_device(params.module(), d_glwe, n as i32, sk.0.as_ptr(), values.as_mut_ptr(),
                                               err.as_mut_ptr()) });
    (values, err)
}
impl Drop for Ram { fn drop(&mut self) { unsafe { fheram_ram_destroy(self.h); } } }
