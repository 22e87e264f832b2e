"""Host-side mirror of the reference's public API over the C ABI (include/fheram.h).

Names, argument meaning and error behaviour follow phantomzone-org/fhe-ram:
  Parameters            src/parameters.rs:147-288
  Source                poulpy_hal::source::Source (examples/fhe-ram.rs:37-43)
  GLWESecret            examples/fhe-ram.rs:49-50
  EvaluationKeys        src/keys.rs:21-25,135-180
  EvaluationKeysPrepared src/keys.rs:27-71
  Address               src/address.rs:21-24,58-109
  Ram                   src/ram.rs:25-29,59-87,129-294
  gen_keys              README.md:131 (older spelling of the same keygen)
The reference is Rust; its toolchain is absent from this image, so the compiled host layer is
C++ (fhe_ram_b200/cpp/fheram.hpp) and this module is the ctypes binding the tests and bench
use.  All arithmetic of read / read_prepare_write / write happens in libfheram_cuda.so on the
GPU; this file never computes on ciphertexts and there is no CPU fallback: a missing library
or GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
_LIB_PATH = Path(os.environ.get("FHERAM_LIB", _PKG / "libfheram_cuda.so"))  # FHERAM_LIB: dev builds (tools/ablate.sh)


class FheRamError(RuntimeError):
    """Raised where the reference would panic (assert!) or on CUDA failures."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"[{code}] {msg}")
        self.code = code


class CParams(C.Structure):
    _fields_ = [
        ("log_n", C.c_int32), ("base2k", C.c_int32), ("k_pt", C.c_int32), ("k_ct", C.c_int32),
        ("k_addr", C.c_int32), ("k_evk_trace", C.c_int32), ("k_evk_ggsw_inv", C.c_int32),
        ("word_size", C.c_int32), ("n_decomp", C.c_int32), ("decomp_n", C.c_int32 * 8),
        ("max_addr", C.c_uint64),
    ]


class CSeed(C.Structure):
    """fheram_seed: the state of a mask Source (ChaCha20 key, stream position in 32-bit words)"""
    _fields_ = [("key", C.c_uint32 * 8), ("word0", C.c_uint64)]


# seeds as numpy records (one per address of a batch), laid out as fheram_seed
SEED_DTYPE = np.dtype([("key", "<u4", (8,)), ("word0", "<u8")], align=True)
assert SEED_DTYPE.itemsize == C.sizeof(CSeed)

_P64 = C.POINTER(C.c_int64)
_PU8 = C.POINTER(C.c_uint8)
_V = C.c_void_p
_PV = C.POINTER(C.c_void_p)
_PP = C.POINTER(CParams)
_PS = C.POINTER(CSeed)

# every symbol include/fheram.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "fheram_params_default": (None, [_PP]),
    "fheram_params_readme": (None, [_PP]),
    "fheram_last_error": (C.c_char_p, []),
    "fheram_version": (C.c_char_p, []),
    "fheram_glwe_len": (C.c_size_t, [_PP]),
    "fheram_ggsw_len": (C.c_size_t, [_PP]),
    "fheram_atk_len": (C.c_size_t, [_PP]),
    "fheram_evk_inv_len": (C.c_size_t, [_PP]),
    "fheram_n_trace_keys": (C.c_int, [_PP]),
    "fheram_n_ggsw": (C.c_int, [_PP]),
    "fheram_n_glwe_per_subram": (C.c_int, [_PP]),
    "fheram_base2d": (C.c_int, [_PP, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "fheram_trace_galois_element": (C.c_int64, [_PP, C.c_int]),
    "fheram_ctx_create": (C.c_int, [_PP, C.c_int, _PV]),
    "fheram_ctx_destroy": (C.c_int, [_V]),
    "fheram_ctx_synchronize": (C.c_int, [_V]),
    "fheram_ctx_stream": (_V, [_V]),
    "fheram_ctx_launch_count": (C.c_uint64, [_V]),
    "fheram_ctx_profile": (C.c_int, [_V, C.c_int]),
    "fheram_ctx_profile_get": (C.c_int, [_V, C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "fheram_ctx_profile_records": (C.c_int, [_V, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_double),
                                             C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "fheram_fp64_peak_probe": (C.c_int, [_V, C.c_int, C.POINTER(C.c_double)]),
    "fheram_debug_phase_cycles": (C.c_int, [_V, C.c_int, C.POINTER(C.c_longlong)]),
    "fheram_debug_device_bytes": (C.c_uint64, []),
    "fheram_host_register": (C.c_int, [_V, C.c_size_t]),
    "fheram_host_unregister": (C.c_int, [_V]),
    "fheram_keys_prepare": (C.c_int, [_V, _P64, _P64, _P64, _PV]),
    "fheram_keys_destroy": (C.c_int, [_V]),
    "fheram_keys_encrypt_sk": (C.c_int, [_V, _P64, _V, _V, _PV]),
    "fheram_keys_download_raw": (C.c_int, [_V, _P64, _P64, _P64]),
    "fheram_address_load": (C.c_int, [_V, _P64, _PV]),
    "fheram_address_load_batch": (C.c_int, [_V, _P64, C.c_int, _PV]),
    "fheram_address_alloc": (C.c_int, [_V, C.c_int, _PV]),
    "fheram_address_raw_ptr": (_V, [_V]),
    "fheram_address_upload_slice": (C.c_int, [_V, _P64, C.c_int, C.c_int]),
    "fheram_address_upload_slice_async": (C.c_int, [_V, _P64, C.c_int, C.c_int]),
    "fheram_address_wait_upload": (C.c_int, [_V]),
    "fheram_address_release": (C.c_int, [_V]),
    "fheram_address_prepare": (C.c_int, [_V]),
    "fheram_address_count": (C.c_int, [_V]),
    "fheram_address_destroy": (C.c_int, [_V]),
    "fheram_ram_create": (C.c_int, [_V, _PV]),
    "fheram_ram_create_sharded": (C.c_int, [_V, C.c_int, C.c_int, _PV]),
    "fheram_ram_destroy": (C.c_int, [_V]),
    "fheram_ram_load": (C.c_int, [_V, _P64]),
    "fheram_ram_store": (C.c_int, [_V, _P64]),
    "fheram_ram_tree_store": (C.c_int, [_V, _P64]),
    "fheram_ram_state": (C.c_int, [_V]),
    "fheram_ram_read": (C.c_int, [_V, _V, _V, _P64]),
    "fheram_ram_read_prepare_write": (C.c_int, [_V, _V, _V, _P64]),
    "fheram_ram_write": (C.c_int, [_V, _P64, _V, _V]),
    "fheram_ram_read_batch": (C.c_int, [_V, _V, _V, _P64]),
    "fheram_ram_read_batch_host": (C.c_int, [_V, _P64, C.c_int, _V, _P64]),
    "fheram_ram_read_batch_host_i32": (C.c_int, [_V, C.POINTER(C.c_int32), C.c_int, _V, C.POINTER(C.c_int32)]),
    "fheram_ram_read_batch_host_p17": (C.c_int, [_V, C.POINTER(C.c_uint32), C.c_int, _V, C.POINTER(C.c_int32)]),
    "fheram_pack17": (C.c_int, [_P64, C.c_size_t, C.POINTER(C.c_uint32)]),
    "fheram_unpack17": (C.c_int, [C.POINTER(C.c_uint32), C.c_size_t, _P64]),
    "fheram_ram_read_batch_device": (C.c_int, [_V, _V, _V, _PV]),
    "fheram_comm_unique_id": (C.c_int, [_PU8]),
    "fheram_comm_init": (C.c_int, [_V, C.c_int, C.c_int, _PU8]),
    "fheram_comm_destroy": (C.c_int, [_V]),
    "fheram_comm_n_ranks": (C.c_int, [_V]),
    "fheram_comm_rank": (C.c_int, [_V]),
    "fheram_download_glwe": (C.c_int, [_V, _V, C.c_int, _P64]),
    "fheram_ram_read_local_device": (C.c_int, [_V, _V, _V, _PV]),
    "fheram_ram_read_finish_device": (C.c_int, [_V, _V, C.c_int, C.c_int, C.c_int, _V, C.c_int, _V, _PV]),
    "fheram_ram_rpw_local_device": (C.c_int, [_V, _V, _V, _PV]),
    "fheram_ram_rpw_finish_device": (C.c_int, [_V, _V, _V, _V, _PV]),
    "fheram_external_product_batch": (C.c_int, [_V, _P64, C.c_int, _P64, _P64]),
    "fheram_coordinate_product": (C.c_int, [_V, _P64, C.c_int, _P64, C.c_int, _P64]),
    "fheram_glwe_trace": (C.c_int, [_V, _V, _P64, C.c_int, C.c_int, C.c_int, _P64]),
    "fheram_glwe_pack": (C.c_int, [_V, _V, _P64, C.c_int, _P64]),
    "fheram_glwe_automorphism": (C.c_int, [_V, _V, C.c_int, C.c_int, C.c_int, _P64, C.c_int, _P64]),
    "fheram_ggsw_invert": (C.c_int, [_V, _V, _P64, C.c_int, _P64]),
    "fheram_source_new": (_V, [_PU8]),
    "fheram_source_free": (None, [_V]),
    "fheram_source_next_u32": (C.c_uint32, [_V]),
    "fheram_source_fill_bytes": (None, [_V, _PU8, C.c_size_t]),
    "fheram_source_position": (C.c_uint64, [_V]),
    "fheram_source_skip": (None, [_V, C.c_uint64]),
    "fheram_secret_gen": (C.c_int, [_PP, _V, _P64]),
    "fheram_keygen": (C.c_int, [_PP, _P64, _V, _V, _P64, _P64, _P64]),
    "fheram_encrypt_ram": (C.c_int, [_PP, _PU8, _P64, _V, _V, _P64]),
    "fheram_encrypt_address": (C.c_int, [_PP, C.c_uint32, _P64, _V, _V, _P64]),
    "fheram_encrypt_word": (C.c_int, [_PP, C.c_uint8, _P64, _V, _V, _P64]),
    "fheram_decrypt_word": (C.c_int, [_PP, _P64, _P64, C.c_int64, _P64, C.POINTER(C.c_double)]),
    "fheram_ram_encrypt_sk": (C.c_int, [_V, _PU8, _P64, _V, _V]),
    "fheram_debug_encrypt_stats": (C.c_int, [_V, C.POINTER(C.c_uint64)]),
    "fheram_address_encrypt_sk": (C.c_int, [_V, C.c_int, C.c_int, C.POINTER(C.c_uint32), _P64,
                                            C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int]),
    "fheram_decrypt_ram": (C.c_int, [_PP, _P64, _P64, C.POINTER(C.c_int16), _P64]),
    "fheram_ram_decrypt_sk": (C.c_int, [_V, _P64, C.POINTER(C.c_int16), _P64]),
    "fheram_decrypt_words_device": (C.c_int, [_V, _V, C.c_int, _P64, C.POINTER(C.c_int16), _P64]),
    "fheram_source_seed": (C.c_int, [_V, _PS]),
    "fheram_encrypt_ram_seeded": (C.c_int, [_PP, _PU8, _P64, _V, _V, _P64, _PS]),
    "fheram_encrypt_address_seeded": (C.c_int, [_PP, C.c_uint32, _P64, _V, _V, _P64, _PS]),
    "fheram_ram_expand": (C.c_int, [_PP, _P64, _PS, _P64]),
    "fheram_address_expand": (C.c_int, [_PP, _P64, _PS, _P64]),
    "fheram_address_load_seeded": (C.c_int, [_V, _P64, _PS, C.c_int, _PV]),
    "fheram_ram_read_batch_host_seeded": (C.c_int, [_V, C.POINTER(C.c_uint32), _PS, C.c_int, _V,
                                                    C.POINTER(C.c_int32)]),
    "fheram_ram_load_seeded": (C.c_int, [_V, _P64, _PS]),
    "fheram_ram_read_plain": (C.c_int, [_V, C.POINTER(C.c_uint32), C.c_int, _V, _P64]),
    "fheram_ram_read_plain_device": (C.c_int, [_V, C.POINTER(C.c_uint32), C.c_int, _V, _PV]),
    "fheram_ram_write_plain": (C.c_int, [_V, C.c_uint32, _P64, _V]),
}

_lib = None


def lib() -> C.CDLL:
    """Loads libfheram_cuda.so (built by __graft_entry__.build()); fails loudly if absent."""
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise FheRamError(-5, f"{_LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; "
                                  "g.build()'` (there is no CPU fallback)")
        _lib = C.CDLL(str(_LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            f = getattr(_lib, name)
            f.restype, f.argtypes = res, args
    return _lib


def _check(rc: int) -> None:
    if rc != 0:
        raise FheRamError(rc, lib().fheram_last_error().decode())


def _p(a: np.ndarray):
    assert a.dtype == np.int64 and a.flags["C_CONTIGUOUS"], "int64 contiguous limbs expected"
    return a.ctypes.data_as(_P64)


class Parameters:
    """src/parameters.rs:147-288.  `Parameters.new()` = the snapshot's constants; the README /
    BASELINE parameter set is `Parameters.readme()`.  max_addr / word_size / decomp_n / k_pt are
    runtime values (Ram::new_from_ram_params, src/ram.rs:72-87)."""

    def __init__(self, c: CParams, device: int = 0):
        self.c = c
        self.device = device
        self._ctx = None

    @classmethod
    def new(cls, device: int = 0, **over) -> "Parameters":
        c = CParams()
        lib().fheram_params_default(C.byref(c))
        return cls(c, device)._override(over)

    @classmethod
    def readme(cls, device: int = 0, **over) -> "Parameters":
        c = CParams()
        lib().fheram_params_readme(C.byref(c))
        return cls(c, device)._override(over)

    def _override(self, over):
        for k, v in over.items():
            if k == "decomp_n":
                self.c.n_decomp = len(v)
                for i, d in enumerate(v):
                    self.c.decomp_n[i] = d
            else:
                setattr(self.c, k, v)
        return self

    # accessors, src/parameters.rs:233-287
    def max_addr(self): return int(self.c.max_addr)
    def word_size(self): return int(self.c.word_size)
    def basek(self): return int(self.c.base2k)
    def k_glwe_ct(self): return int(self.c.k_ct)
    def k_glwe_pt(self): return int(self.c.k_pt)
    def k_ggsw_addr(self): return int(self.c.k_addr)
    def k_evk_trace(self): return int(self.c.k_evk_trace)
    def k_evk_ggsw_inv(self): return int(self.c.k_evk_ggsw_inv)
    def rank(self): return 1
    def n(self): return 1 << int(self.c.log_n)
    def log_n(self): return int(self.c.log_n)
    def decomp_n(self): return [int(self.c.decomp_n[i]) for i in range(self.c.n_decomp)]
    def dnum_ct(self): return -(-self.k_glwe_ct() // self.basek())
    def dnum_ggsw(self): return -(-self.k_ggsw_addr() // self.basek())

    def base2d(self):
        lens = (C.c_int32 * 8)()
        digits = (C.c_int32 * 64)()
        n = lib().fheram_base2d(C.byref(self.c), lens, digits)
        return [[int(digits[i * 8 + j]) for j in range(lens[i])] for i in range(n)]

    # sizes in int64 limbs
    def glwe_len(self): return lib().fheram_glwe_len(C.byref(self.c))
    def ggsw_len(self): return lib().fheram_ggsw_len(C.byref(self.c))
    def atk_len(self): return lib().fheram_atk_len(C.byref(self.c))
    def evk_inv_len(self): return lib().fheram_evk_inv_len(C.byref(self.c))
    def n_trace_keys(self): return lib().fheram_n_trace_keys(C.byref(self.c))
    def n_ggsw(self): return lib().fheram_n_ggsw(C.byref(self.c))
    def n_glwe(self): return lib().fheram_n_glwe_per_subram(C.byref(self.c))
    def trace_galois_elements(self):
        return [int(lib().fheram_trace_galois_element(C.byref(self.c), i)) for i in range(self.n_trace_keys())]

    def module(self):
        """Module::<B>::new(1 << LOG_N): here, the device context (created on first use)."""
        if self._ctx is None:
            h = C.c_void_p()
            _check(lib().fheram_ctx_create(C.byref(self.c), self.device, C.byref(h)))
            self._ctx = h
        return self._ctx

    def synchronize(self):
        _check(lib().fheram_ctx_synchronize(self.module()))

    def launch_count(self) -> int:
        return int(lib().fheram_ctx_launch_count(self.module()))

    def stream(self) -> int:
        return int(lib().fheram_ctx_stream(self.module()) or 0)

    def encrypt_stats(self) -> dict:
        """noise draws of the device encryption path so far: sampled on the device / re-drawn by the host /
        streams sampled by the host"""
        out = (C.c_uint64 * 3)()
        _check(lib().fheram_debug_encrypt_stats(self.module(), out))
        return {"device_draws": int(out[0]), "host_redraws": int(out[1]), "host_streams": int(out[2])}

    def profile(self, enable: bool):
        _check(lib().fheram_ctx_profile(self.module(), 1 if enable else 0))

    def profile_get(self):
        """per kernel class (ext, trace, combine2, other): (ms, launches, ops)"""
        ms = (C.c_double * 4)()
        ln = (C.c_uint64 * 4)()
        ops = (C.c_uint64 * 4)()
        _check(lib().fheram_ctx_profile_get(self.module(), ms, ln, ops))
        names = ("ext", "trace", "combine2", "other")
        return {n: {"ms": ms[i], "launches": int(ln[i]), "ops": int(ops[i])} for i, n in enumerate(names)}

    def profile_records(self, max_n: int = 256):
        """[(class, ms, items, steps)] per launch of the profiled region"""
        cls = (C.c_int * max_n)()
        ms = (C.c_double * max_n)()
        it = (C.c_uint64 * max_n)()
        st = (C.c_uint64 * max_n)()
        n = lib().fheram_ctx_profile_records(self.module(), max_n, cls, ms, it, st)
        names = ("ext", "trace", "combine2", "other")
        return [(names[cls[i]], ms[i], int(it[i]), int(st[i])) for i in range(max(n, 0))]

    # ---- multi-GPU communicator (fheram_comm_*): NCCL inside the library, one rank per context ----
    @staticmethod
    def comm_unique_id() -> np.ndarray:
        """rank 0: the 128-byte id the other ranks need (hand it over with MPI / a store / torch.distributed)"""
        out = np.zeros(128, dtype=np.uint8)
        _check(lib().fheram_comm_unique_id(out.ctypes.data_as(_PU8)))
        return out

    def comm_init(self, n_ranks: int, rank: int, uid: np.ndarray):
        uid = np.ascontiguousarray(uid, dtype=np.uint8)
        assert uid.size == 128
        _check(lib().fheram_comm_init(self.module(), n_ranks, rank, uid.ctypes.data_as(_PU8)))

    def comm_destroy(self):
        _check(lib().fheram_comm_destroy(self.module()))

    def fp64_peak_tflops(self, reps: int = 5) -> float:
        v = C.c_double()
        _check(lib().fheram_fp64_peak_probe(self.module(), reps, C.byref(v)))
        return float(v.value)

    def close(self):
        if self._ctx is not None:
            lib().fheram_ctx_destroy(self._ctx)
            self._ctx = None


def pack17(limbs: np.ndarray) -> np.ndarray:
    """normalised int64 limbs -> the packed host format (17-bit fields, uint32 words)"""
    a = np.ascontiguousarray(limbs, dtype=np.int64).reshape(-1)
    out = np.zeros(a.size * 17 // 32, dtype=np.uint32)
    _check(lib().fheram_pack17(_p(a), a.size, out.ctypes.data_as(C.POINTER(C.c_uint32))))
    return out


def unpack17(packed: np.ndarray, n: int) -> np.ndarray:
    p = np.ascontiguousarray(packed, dtype=np.uint32).reshape(-1)
    out = np.zeros(n, dtype=np.int64)
    _check(lib().fheram_unpack17(p.ctypes.data_as(C.POINTER(C.c_uint32)), n, _p(out)))
    return out


def _ps(seeds: np.ndarray, n: int):
    assert seeds.dtype == SEED_DTYPE and seeds.flags["C_CONTIGUOUS"] and seeds.size == n, \
        f"{n} seed(s) of SEED_DTYPE expected"
    return seeds.ctypes.data_as(_PS)


def _seeds(seeds) -> np.ndarray:
    """one SEED_DTYPE array from an array of seeds or a list of them"""
    if isinstance(seeds, (list, tuple)):
        seeds = np.concatenate([np.asarray(x, dtype=SEED_DTYPE).reshape(-1) for x in seeds])
    return np.ascontiguousarray(np.asarray(seeds, dtype=SEED_DTYPE).reshape(-1))


def host_register(a: np.ndarray):
    _check(lib().fheram_host_register(a.ctypes.data_as(C.c_void_p), a.nbytes))


def host_unregister(a: np.ndarray):
    _check(lib().fheram_host_unregister(a.ctypes.data_as(C.c_void_p)))


class Source:
    """poulpy_hal::source::Source::new(seed) (examples/fhe-ram.rs:41-43)."""

    def __init__(self, seed):
        if isinstance(seed, int):  # [x; 32] as the example's seeds, or a 256-bit integer
            seed = bytes([seed] * 32) if 0 <= seed < 256 else int(seed).to_bytes(32, "little")
        self.h = lib().fheram_source_new((C.c_uint8 * 32)(*seed))

    def next_u32(self) -> int:
        return int(lib().fheram_source_next_u32(self.h))

    def position(self) -> int:
        """32-bit words drawn so far"""
        return int(lib().fheram_source_position(self.h))

    def skip(self, n_words: int):
        lib().fheram_source_skip(self.h, int(n_words))

    def fill_bytes(self, n: int) -> np.ndarray:
        out = np.zeros(n, dtype=np.uint8)
        lib().fheram_source_fill_bytes(self.h, out.ctypes.data_as(_PU8), n)
        return out

    def seed(self) -> np.ndarray:
        """the seed of the current position (one SEED_DTYPE record, shape (1,))"""
        out = np.zeros(1, dtype=SEED_DTYPE)
        _check(lib().fheram_source_seed(self.h, _ps(out, 1)))
        return out

    def __del__(self):
        try:
            lib().fheram_source_free(self.h)
        except Exception:
            pass


class GLWESecret:
    """GLWESecret::alloc_from_infos + fill_ternary_prob(0.5, xs) (examples/fhe-ram.rs:49-50)."""

    def __init__(self, params: Parameters, data: np.ndarray):
        self.params, self.data = params, data

    @classmethod
    def fill_ternary_prob(cls, params: Parameters, prob: float, source_xs: Source) -> "GLWESecret":
        assert prob == 0.5, "the reference only uses prob = 0.5"
        sk = np.zeros(params.n(), dtype=np.int64)
        _check(lib().fheram_secret_gen(C.byref(params.c), source_xs.h, _p(sk)))
        return cls(params, sk)


class EvaluationKeys:
    """src/keys.rs:21-25: atk_glwe (one automorphism key per trace Galois element),
    atk_ggsw_inv (p = -1) and the GGLWE->GGSW key, as raw int64 limbs."""

    def __init__(self, params, atk_glwe, tsk, atk_inv):
        self.params, self.atk_glwe, self.gglwe_to_ggsw_key, self.atk_ggsw_inv = params, atk_glwe, tsk, atk_inv

    @classmethod
    def encrypt_sk(cls, params: Parameters, sk: GLWESecret, source_xa: Source, source_xe: Source):
        """src/keys.rs:135-180"""
        atk = np.zeros(params.n_trace_keys() * params.atk_len(), dtype=np.int64)
        tsk = np.zeros(params.evk_inv_len(), dtype=np.int64)
        inv = np.zeros(params.evk_inv_len(), dtype=np.int64)
        _check(lib().fheram_keygen(C.byref(params.c), _p(sk.data), source_xa.h, source_xe.h,
                                   _p(atk), _p(tsk), _p(inv)))
        return cls(params, atk, tsk, inv)


class EvaluationKeysPrepared:
    """src/keys.rs:27-71: alloc(params) then prepare(module, keys, scratch); the prepared keys
    live in HBM."""

    def __init__(self, params: Parameters):
        self.params, self.h = params, None

    @classmethod
    def alloc(cls, params: Parameters) -> "EvaluationKeysPrepared":
        return cls(params)

    def prepare(self, keys: EvaluationKeys) -> "EvaluationKeysPrepared":
        h = C.c_void_p()
        _check(lib().fheram_keys_prepare(self.params.module(), _p(keys.atk_glwe),
                                         _p(keys.gglwe_to_ggsw_key), _p(keys.atk_ggsw_inv), C.byref(h)))
        self.h = h
        return self

    @classmethod
    def encrypt_sk_gpu(cls, params: Parameters, sk: "GLWESecret", source_xa: "Source", source_xe: "Source") -> "EvaluationKeysPrepared":
        """EvaluationKeys::encrypt_sk (src/keys.rs:135-180) + prepare on the device: the limbs of
        `EvaluationKeys.encrypt_sk` from the same Sources, resident and prepared"""
        k = cls(params)
        h = C.c_void_p()
        _check(lib().fheram_keys_encrypt_sk(params.module(), _p(sk.data), source_xa.h, source_xe.h, C.byref(h)))
        k.h = h
        return k

    def download_raw(self) -> "EvaluationKeys":
        """raw limbs of keys made by encrypt_sk_gpu (fheram_keygen's layout)"""
        p = self.params
        atk = np.zeros(p.n_trace_keys() * p.atk_len(), dtype=np.int64)
        tsk = np.zeros(p.evk_inv_len(), dtype=np.int64)
        inv = np.zeros(p.evk_inv_len(), dtype=np.int64)
        _check(lib().fheram_keys_download_raw(self.h, _p(atk), _p(tsk), _p(inv)))
        return EvaluationKeys(p, atk, tsk, inv)

    def close(self):
        if self.h is not None:
            lib().fheram_keys_destroy(self.h)
            self.h = None


def gen_keys(params: Parameters, seed_xs=0, seed_xa=0, seed_xe=0):
    """README.md:131 `let (sk, evk) = gen_keys(&params)`; seeds as in examples/fhe-ram.rs:37-39."""
    sk = GLWESecret.fill_ternary_prob(params, 0.5, Source(seed_xs))
    evk = EvaluationKeys.encrypt_sk(params, sk, Source(seed_xa), Source(seed_xe))
    return sk, evk


class Address:
    """src/address.rs:21-24.  `encrypt_sk` is client side (CPU); the encrypted address is then
    made resident on the device together with its prepared form."""

    def __init__(self, params: Parameters):
        self.params = params
        self.data = np.zeros(params.n_ggsw() * params.ggsw_len(), dtype=np.int64)
        self.h = None
        self.count = 1

    @classmethod
    def alloc_from_params(cls, params: Parameters) -> "Address":   # src/address.rs:58-60
        return cls(params)

    alloc = alloc_from_params                                       # README.md:141

    def encrypt_sk(self, params: Parameters, value: int, sk: GLWESecret, source_xa: Source,
                   source_xe: Source) -> "Address":                 # src/address.rs:86-109
        _check(lib().fheram_encrypt_address(C.byref(params.c), int(value), _p(sk.data), source_xa.h,
                                            source_xe.h, _p(self.data)))
        self._drop()
        return self

    @staticmethod
    def encrypt_sk_seeded(params: Parameters, value: int, sk: GLWESecret, source_xa: Source, source_xe: Source):
        """Address::encrypt_sk in the seeded form (include/fheram.h): (bodies int64 [n_ggsw][dnum][2][size][N]
        flattened, seed).  The rows with ci = 1 carry their plaintext in the body, so the limbs differ from
        `encrypt_sk`'s (same phase, same noise); both Sources end where `encrypt_sk` leaves them."""
        bodies = np.zeros(params.n_ggsw() * params.ggsw_len() // 2, dtype=np.int64)
        seed = np.zeros(1, dtype=SEED_DTYPE)
        _check(lib().fheram_encrypt_address_seeded(C.byref(params.c), int(value), _p(sk.data), source_xa.h,
                                                   source_xe.h, _p(bodies), _ps(seed, 1)))
        return bodies, seed

    @classmethod
    def expand(cls, params: Parameters, bodies: np.ndarray, seeds, count: int = 1) -> "Address":
        """full limbs of `count` seeded addresses (CPU): what the device expansion builds"""
        seeds = _seeds(seeds)
        bodies = np.ascontiguousarray(bodies, dtype=np.int64).reshape(count, -1)
        per = params.n_ggsw() * params.ggsw_len()
        if bodies.shape[1] != per // 2 or seeds.size != count:
            raise FheRamError(-1, "bodies / seeds do not hold `count` addresses")
        out = np.zeros((count, per), dtype=np.int64)
        for i in range(count):
            _check(lib().fheram_address_expand(C.byref(params.c), _p(bodies[i]), _ps(seeds[i:i + 1], 1), _p(out[i])))
        return cls.from_limbs(params, out, count)

    @classmethod
    def load_seeded(cls, params: Parameters, bodies: np.ndarray, seeds, count: int = 1) -> "Address":
        """`count` seeded addresses made resident and prepared; the masks are regenerated on the device"""
        seeds = _seeds(seeds)
        bodies = np.ascontiguousarray(bodies, dtype=np.int64).reshape(-1)
        if bodies.size != count * params.n_ggsw() * params.ggsw_len() // 2:
            raise FheRamError(-1, "bodies do not hold `count` addresses")
        a = cls.__new__(cls)
        a.params, a.data, a.count = params, None, count
        h = C.c_void_p()
        _check(lib().fheram_address_load_seeded(params.module(), _p(bodies), _ps(seeds, count), count, C.byref(h)))
        a.h = h
        return a

    @classmethod
    def from_limbs(cls, params: Parameters, limbs: np.ndarray, count: int = 1) -> "Address":
        a = cls(params)
        a.data = np.ascontiguousarray(limbs, dtype=np.int64).reshape(-1)
        a.count = count
        assert a.data.size == count * params.n_ggsw() * params.ggsw_len()
        return a

    @classmethod
    def device_alloc(cls, params: Parameters, count: int) -> "Address":
        """n addresses allocated on the device only (multi-GPU path: upload_slice + all-gather into
        raw_ptr() + prepare())."""
        a = cls.__new__(cls)
        a.params, a.data, a.count = params, None, count
        h = C.c_void_p()
        _check(lib().fheram_address_alloc(params.module(), count, C.byref(h)))
        a.h = h
        return a

    @classmethod
    def encrypt_sk_gpu(cls, params: Parameters, values, sk: GLWESecret, sources_xa, sources_xe,
                       prepare: bool = True) -> "Address":
        """src/address.rs:86-109 for every value, on the device (k_glwe_encrypt): the same limbs as
        `encrypt_sk` from the same Sources.  One (xa, xe) pair for all addresses in turn, or one pair
        per address.  Returns the device-resident address set, prepared."""
        values = np.ascontiguousarray(values, dtype=np.uint32).reshape(-1)
        xas = list(sources_xa) if isinstance(sources_xa, (list, tuple)) else [sources_xa]
        xes = list(sources_xe) if isinstance(sources_xe, (list, tuple)) else [sources_xe]
        if len(xas) != len(xes) or len(xas) not in (1, values.size):
            raise FheRamError(-1, "one Source pair, or one pair per address")
        a = cls.device_alloc(params, int(values.size))
        ha = (C.c_void_p * len(xas))(*[x.h for x in xas])
        he = (C.c_void_p * len(xes))(*[x.h for x in xes])
        _check(lib().fheram_address_encrypt_sk(a.h, 0, int(values.size), values.ctypes.data_as(C.POINTER(C.c_uint32)),
                                               _p(sk.data), ha, he, len(xas)))
        return a.prepare() if prepare else a

    def download_raw(self) -> np.ndarray:
        """raw GGSW limbs of a device address set as int64 (tests)"""
        per = self.params.n_ggsw() * self.params.ggsw_len()
        out = np.zeros(self.count * per, dtype=np.int64)
        n_glwe_units = out.size // self.params.glwe_len()
        assert n_glwe_units * self.params.glwe_len() == out.size
        _check(lib().fheram_download_glwe(self.params.module(), C.c_void_p(self.raw_ptr()), n_glwe_units, _p(out)))
        return out

    def upload_slice(self, limbs: np.ndarray, first: int, count: int):
        _check(lib().fheram_address_upload_slice(self.h, _p(np.ascontiguousarray(limbs, dtype=np.int64).reshape(-1)),
                                                 first, count))

    def upload_slice_async(self, limbs: np.ndarray, first: int, count: int):
        """limbs must stay alive (and should be pinned: host_register) until wait_upload's stream work ran"""
        assert limbs.dtype == np.int64 and limbs.flags.c_contiguous
        _check(lib().fheram_address_upload_slice_async(self.h, _p(limbs.reshape(-1)), first, count))

    def wait_upload(self):
        _check(lib().fheram_address_wait_upload(self.h))

    def release(self):
        _check(lib().fheram_address_release(self.h))

    def raw_ptr(self) -> int:
        return int(lib().fheram_address_raw_ptr(self.h))

    def prepare(self):
        _check(lib().fheram_address_prepare(self.h))
        return self

    @classmethod
    def batch(cls, params: Parameters, addresses) -> "Address":
        return cls.from_limbs(params, np.concatenate([a.data for a in addresses]), len(addresses))

    def n2(self): return len(self.params.base2d())                  # src/address.rs:113-115

    def device(self):
        if self.h is None:
            h = C.c_void_p()
            _check(lib().fheram_address_load_batch(self.params.module(), _p(self.data), self.count, C.byref(h)))
            self.h = h
        return self.h

    def _drop(self):
        if self.h is not None:
            lib().fheram_address_destroy(self.h)
            self.h = None

    close = _drop


class Ram:
    """src/ram.rs:25-29.  `Ram.new(params)` allocates the device-resident RAM; `encrypt_sk`
    encrypts on the client side and uploads; read / read_prepare_write / write run on the GPU."""

    def __init__(self, params: Parameters, shard: int = 0, n_shards: int = 1):
        self.params = params
        h = C.c_void_p()
        if n_shards == 1:
            _check(lib().fheram_ram_create(params.module(), C.byref(h)))
        else:
            _check(lib().fheram_ram_create_sharded(params.module(), shard, n_shards, C.byref(h)))
        self.h = h
        self.shard, self.n_shards = shard, n_shards

    @classmethod
    def new(cls, params: Parameters | None = None) -> "Ram":                      # src/ram.rs:59-69
        return cls(params if params is not None else Parameters.new())

    @classmethod
    def new_from_ram_params(cls, word_size: int, decomp_n, max_addr: int, **over) -> "Ram":  # :72-87
        return cls(Parameters.new(word_size=word_size, decomp_n=list(decomp_n), max_addr=max_addr, **over))

    def glwe_count(self): return self.params.word_size() * self.params.n_glwe()

    def encrypt_sk(self, data, sk: GLWESecret, source_xa: Source, source_xe: Source) -> np.ndarray:
        """src/ram.rs:129-167 (asserts :144-155)."""
        p = self.params
        data = np.ascontiguousarray(data, dtype=np.uint8)
        ws = p.word_size()
        if data.size % ws != 0:
            raise FheRamError(-1, f"invalid data: data.len()%ram_chunks={data.size % ws} != 0")
        if data.size // ws != p.max_addr():
            raise FheRamError(-1, f"invalid data: data.len()/ram_chunks={data.size // ws} != max_addr={p.max_addr()}")
        cts = np.zeros(self.glwe_count() * p.glwe_len(), dtype=np.int64)
        _check(lib().fheram_encrypt_ram(C.byref(p.c), data.ctypes.data_as(_PU8), _p(sk.data),
                                        source_xa.h, source_xe.h, _p(cts)))
        self.load(cts)
        return cts

    def encrypt_sk_seeded(self, data, sk: GLWESecret, source_xa: Source, source_xe: Source):
        """Ram::encrypt_sk in the seeded form (CPU), then `load_seeded`: returns (bodies, seed).  Expanded, they are
        exactly the limbs `encrypt_sk` returns from the same Sources."""
        p = self.params
        data = np.ascontiguousarray(data, dtype=np.uint8)
        if data.size != p.max_addr() * p.word_size():
            raise FheRamError(-1, f"invalid data: {data.size} bytes != max_addr * word_size")
        bodies = np.zeros(self.glwe_count() * p.glwe_len() // 2, dtype=np.int64)
        seed = np.zeros(1, dtype=SEED_DTYPE)
        _check(lib().fheram_encrypt_ram_seeded(C.byref(p.c), data.ctypes.data_as(_PU8), _p(sk.data), source_xa.h,
                                               source_xe.h, _p(bodies), _ps(seed, 1)))
        self.load_seeded(bodies, seed)
        return bodies, seed

    @staticmethod
    def expand(params: Parameters, bodies: np.ndarray, seed) -> np.ndarray:
        """full limbs of a seeded RAM (CPU), in `encrypt_sk` / `store` layout"""
        bodies = np.ascontiguousarray(bodies, dtype=np.int64).reshape(-1)
        cts = np.zeros(2 * bodies.size, dtype=np.int64)
        if cts.size != params.word_size() * params.n_glwe() * params.glwe_len():
            raise FheRamError(-1, "bodies are not a whole RAM")
        _check(lib().fheram_ram_expand(C.byref(params.c), _p(bodies), _ps(_seeds(seed), 1), _p(cts)))
        return cts

    def load_seeded(self, bodies: np.ndarray, seed):
        """`load` of a seeded RAM (bodies of the whole RAM; a sharded RAM expands its own polynomials)"""
        bodies = np.ascontiguousarray(bodies, dtype=np.int64).reshape(-1)
        if 2 * bodies.size != self.glwe_count() * self.params.glwe_len():
            raise FheRamError(-1, "bodies are not a whole RAM")
        _check(lib().fheram_ram_load_seeded(self.h, _p(bodies), _ps(_seeds(seed), 1)))

    def encrypt_sk_gpu(self, data, sk: GLWESecret, source_xa: Source, source_xe: Source) -> None:
        """src/ram.rs:129-167 on the device (k_glwe_encrypt), straight into the resident RAM: the same
        limbs as `encrypt_sk` from the same Sources, without the host round trip."""
        p = self.params
        data = np.ascontiguousarray(data, dtype=np.uint8)
        ws = p.word_size()
        if data.size % ws != 0:
            raise FheRamError(-1, f"invalid data: data.len()%ram_chunks={data.size % ws} != 0")
        if data.size // ws != p.max_addr():
            raise FheRamError(-1, f"invalid data: data.len()/ram_chunks={data.size // ws} != max_addr={p.max_addr()}")
        _check(lib().fheram_ram_encrypt_sk(self.h, data.ctypes.data_as(_PU8), _p(sk.data), source_xa.h, source_xe.h))

    def decrypt_sk(self, sk: GLWESecret, values=None, err=None):
        """Every byte of the resident RAM, decrypted on the device: (values, err), both [max_addr][word_size]
        (int16 / int64; `decrypt_ram` on `store()`, bit for bit).  A sharded RAM fills the entries of its own
        polynomials and leaves the rest of `values` / `err` (zeros when not passed) as they are."""
        values, err = _dec_out(self.params, values, err)
        _check(lib().fheram_ram_decrypt_sk(self.h, _p(_sk_limbs(sk)), values.ctypes.data_as(C.POINTER(C.c_int16)),
                                           _p(err)))
        return values, err

    def load(self, cts: np.ndarray):
        _check(lib().fheram_ram_load(self.h, _p(np.ascontiguousarray(cts, dtype=np.int64))))

    def store(self) -> np.ndarray:
        out = np.zeros(self.glwe_count() * self.params.glwe_len(), dtype=np.int64)
        _check(lib().fheram_ram_store(self.h, _p(out)))
        return out

    def tree_store(self) -> np.ndarray:
        out = np.zeros(self.params.word_size() * self.params.glwe_len(), dtype=np.int64)
        _check(lib().fheram_ram_tree_store(self.h, _p(out)))
        return out

    def state(self) -> bool: return bool(lib().fheram_ram_state(self.h))

    def _out(self, n=1):
        return np.zeros((n, self.params.word_size(), self.params.glwe_len()), dtype=np.int64)

    def read(self, address: Address, keys: EvaluationKeysPrepared) -> np.ndarray:
        """Ram::read (src/ram.rs:172-191): returns [word_size] GLWE (int64 limbs)."""
        out = self._out()
        _check(lib().fheram_ram_read(self.h, address.device(), keys.h, _p(out)))
        return out[0]

    def read_prepare_write(self, address: Address, keys: EvaluationKeysPrepared) -> np.ndarray:
        """Ram::read_prepare_write (src/ram.rs:196-222)."""
        out = self._out()
        _check(lib().fheram_ram_read_prepare_write(self.h, address.device(), keys.h, _p(out)))
        return out[0]

    def write(self, w, address: Address, keys: EvaluationKeysPrepared) -> None:
        """Ram::write (src/ram.rs:226-294); w = word_size GLWE (assert :243).  Sharded RAM with a communicator:
        rank 0's word is broadcast, the other ranks may pass None."""
        if w is None:
            _check(lib().fheram_ram_write(self.h, None, address.device(), keys.h))
            return
        w = np.ascontiguousarray(w, dtype=np.int64).reshape(-1)
        if w.size != self.params.word_size() * self.params.glwe_len():
            raise FheRamError(-1, "assertion failed: w.len() == self.subrams.len()")
        _check(lib().fheram_ram_write(self.h, _p(w), address.device(), keys.h))

    def read_batch(self, addresses: Address, keys: EvaluationKeysPrepared) -> np.ndarray:
        """n independent reads (BASELINE.json config 3): [n][word_size] GLWE (sharded RAM with a communicator: this
        rank's n / n_shards reads of the batch)."""
        out = self._out(addresses.count // self.n_shards)
        _check(lib().fheram_ram_read_batch(self.h, addresses.device(), keys.h, _p(out)))
        return out

    def read_batch_host(self, addr_limbs: np.ndarray, n: int, keys: EvaluationKeysPrepared, out=None) -> np.ndarray:
        """n reads straight from host int64 address limbs (pipelined upload / prepare / read / download)."""
        out = self._out(n) if out is None else out
        _check(lib().fheram_ram_read_batch_host(self.h, _p(np.ascontiguousarray(addr_limbs, dtype=np.int64).reshape(-1)),
                                                n, keys.h, _p(out.reshape(-1))))
        return out

    def read_batch_host_i32(self, addr_limbs: np.ndarray, n: int, keys: EvaluationKeysPrepared, out=None) -> np.ndarray:
        """the same from the compact host format: int32 limbs in, int32 limbs out (half the PCIe bytes)"""
        a = np.ascontiguousarray(addr_limbs, dtype=np.int32).reshape(-1)
        if out is None:
            out = np.zeros((n, self.params.word_size(), self.params.glwe_len()), dtype=np.int32)
        P32 = C.POINTER(C.c_int32)
        _check(lib().fheram_ram_read_batch_host_i32(self.h, a.ctypes.data_as(P32), n, keys.h,
                                                    out.reshape(-1).ctypes.data_as(P32)))
        return out

    def read_batch_host_p17(self, packed: np.ndarray, n: int, keys: EvaluationKeysPrepared, out=None) -> np.ndarray:
        """addresses in the packed host format (api.pack17), int32 limbs out"""
        a = np.ascontiguousarray(packed, dtype=np.uint32).reshape(-1)
        if out is None:
            out = np.zeros((n, self.params.word_size(), self.params.glwe_len()), dtype=np.int32)
        _check(lib().fheram_ram_read_batch_host_p17(self.h, a.ctypes.data_as(C.POINTER(C.c_uint32)), n, keys.h,
                                                    out.reshape(-1).ctypes.data_as(C.POINTER(C.c_int32))))
        return out

    def read_batch_host_seeded(self, bodies_p17: np.ndarray, seeds, n: int, keys: EvaluationKeysPrepared,
                               out=None) -> np.ndarray:
        """n seeded addresses: their bodies packed by `pack17` and one seed each; int32 limbs out"""
        a = np.ascontiguousarray(bodies_p17, dtype=np.uint32).reshape(-1)
        if a.size != n * self.params.n_ggsw() * self.params.ggsw_len() // 2 * 17 // 32:
            raise FheRamError(-1, "bodies_p17 does not hold n packed addresses")
        if out is None:
            out = np.zeros((n, self.params.word_size(), self.params.glwe_len()), dtype=np.int32)
        _check(lib().fheram_ram_read_batch_host_seeded(self.h, a.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                       _ps(_seeds(seeds), n), n, keys.h,
                                                       out.reshape(-1).ctypes.data_as(C.POINTER(C.c_int32))))
        return out

    def read_batch_device(self, addresses: Address, keys: EvaluationKeysPrepared) -> int:
        """Device-resident batched read; returns the device pointer of the int32 result arena."""
        d = C.c_void_p()
        _check(lib().fheram_ram_read_batch_device(self.h, addresses.device(), keys.h, C.byref(d)))
        return int(d.value)

    # ---- plaintext addresses (include/fheram.h): the address is disclosed to the server, the words stay encrypted ----
    @staticmethod
    def _addrs(addrs) -> np.ndarray:
        a = np.asarray(addrs, dtype=np.int64).reshape(-1)
        if a.size and (a.min() < 0 or a.max() >= 1 << 32):
            raise FheRamError(-1, "addresses must be in [0, 2^32)")
        return np.ascontiguousarray(a, dtype=np.uint32)

    def read_plain(self, addrs, keys: EvaluationKeysPrepared, out=None) -> np.ndarray:
        """[n][word_size] GLWE: TRACE(data[s][h] X^-j) for each address a = h N + j.  A shard without a communicator
        fills the entries of the addresses it holds and leaves the rest of `out` (zeros when not passed) as it is."""
        a = self._addrs(addrs)
        out = self._out(a.size) if out is None else out
        assert out.dtype == np.int64 and out.flags.c_contiguous and out.size == a.size * self.params.word_size() * \
            self.params.glwe_len()
        _check(lib().fheram_ram_read_plain(self.h, a.ctypes.data_as(C.POINTER(C.c_uint32)), int(a.size), keys.h,
                                           _p(out.reshape(-1))))
        return out

    def read_plain_device(self, addrs, keys: EvaluationKeysPrepared) -> int:
        """read_plain into the RAM's device arena ([n][word_size] GLWE, int32 limbs); returns its device pointer"""
        a = self._addrs(addrs)
        d = C.c_void_p()
        _check(lib().fheram_ram_read_plain_device(self.h, a.ctypes.data_as(C.POINTER(C.c_uint32)), int(a.size),
                                                  keys.h, C.byref(d)))
        return int(d.value)

    def write_plain(self, addr: int, w, keys: EvaluationKeysPrepared) -> None:
        """data[s][h] = normalize(data[s][h] - TRACE(data[s][h] X^-j) X^j + w[s] X^j) for a = h N + j; w = word_size
        GLWE as `write` takes it (sharded RAM with a communicator: rank 0's, the other ranks may pass None)"""
        if not 0 <= int(addr) < 1 << 32:
            raise FheRamError(-1, "addresses must be in [0, 2^32)")
        if w is None:
            _check(lib().fheram_ram_write_plain(self.h, int(addr), None, keys.h))
            return
        w = np.ascontiguousarray(w, dtype=np.int64).reshape(-1)
        if w.size != self.params.word_size() * self.params.glwe_len():
            raise FheRamError(-1, "w must hold word_size GLWE")
        _check(lib().fheram_ram_write_plain(self.h, int(addr), _p(w), keys.h))

    def close(self):
        if self.h is not None:
            lib().fheram_ram_destroy(self.h)
            self.h = None


# ---- examples/fhe-ram.rs helpers ------------------------------------------------------
def cast_u8_to_signed(value: int, bit_length: int) -> int:      # examples/fhe-ram.rs:25-32
    assert 1 <= bit_length <= 8, "bit_length must be between 1 and 8"
    shift = 8 - bit_length
    v = (value << shift) & 0xFF
    v = v - 256 if v >= 128 else v
    return v >> shift


def encrypt_glwe(params: Parameters, value: int, sk: GLWESecret, source_xa=None, source_xe=None) -> np.ndarray:
    """examples/fhe-ram.rs:179-210 (fresh Source([1;32]) per call, :199-200)."""
    out = np.zeros(params.glwe_len(), dtype=np.int64)
    xa = source_xa or Source(1)
    xe = source_xe or Source(1)
    _check(lib().fheram_encrypt_word(C.byref(params.c), int(value), _p(sk.data), xa.h, xe.h, _p(out)))
    return out


def decrypt_glwe(params: Parameters, ct: np.ndarray, want: int, sk: GLWESecret):
    """examples/fhe-ram.rs:212-237: (decrypted_value, noise)."""
    v = C.c_int64()
    noise = C.c_double()
    ct = np.ascontiguousarray(ct, dtype=np.int64)
    _check(lib().fheram_decrypt_word(C.byref(params.c), _p(ct), _p(sk.data), int(want), C.byref(v), C.byref(noise)))
    return int(v.value), float(noise.value)


def _sk_limbs(sk) -> np.ndarray:
    return np.ascontiguousarray(sk.data if isinstance(sk, GLWESecret) else sk, dtype=np.int64)


def _dec_out(params: Parameters, values, err):
    shape = (params.max_addr(), params.word_size())
    values = np.zeros(shape, dtype=np.int16) if values is None else values
    err = np.zeros(shape, dtype=np.int64) if err is None else err
    assert values.dtype == np.int16 and values.shape == shape and values.flags.c_contiguous
    assert err.dtype == np.int64 and err.shape == shape and err.flags.c_contiguous
    return values, err


def decrypt_ram(params: Parameters, cts: np.ndarray, sk):
    """Every byte of a RAM in `Ram.encrypt_sk` / `Ram.store` layout, decrypted on the CPU (all host threads):
    (values, err), both [max_addr][word_size].  value = the byte as cast_u8_to_signed(b, min(8, k_pt)) reads it;
    err = the exact phase error at precision k_ct (log2|err| - k_ct is decrypt_glwe's noise)."""
    cts = np.ascontiguousarray(cts, dtype=np.int64).reshape(-1)
    if cts.size != params.word_size() * params.n_glwe() * params.glwe_len():
        raise FheRamError(-1, "cts is not a whole RAM ([word_size][n_glwe] GLWE)")
    values, err = _dec_out(params, None, None)
    _check(lib().fheram_decrypt_ram(C.byref(params.c), _p(cts), _p(_sk_limbs(sk)),
                                    values.ctypes.data_as(C.POINTER(C.c_int16)), _p(err)))
    return values, err


def decrypt_words_device(params: Parameters, d_ptr: int, n: int, sk):
    """Coefficient 0 of n device-resident GLWE(k_ct) (int32 [n][limb][col][N], e.g. `Ram.read_batch_device`'s arena
    with n = reads x word_size), decrypted on the device: (values int16 [n], err int64 [n])."""
    values = np.zeros(n, dtype=np.int16)
    err = np.zeros(n, dtype=np.int64)
    _check(lib().fheram_decrypt_words_device(params.module(), C.c_void_p(int(d_ptr)), int(n), _p(_sk_limbs(sk)),
                                             values.ctypes.data_as(C.POINTER(C.c_int16)), _p(err)))
    return values, err


# ---- op-level entry points (kernel parity tests, BASELINE.json config 2) ----------------
def external_product_batch(params, glwe_in, ggsw):
    glwe_in = np.ascontiguousarray(glwe_in, dtype=np.int64)
    n = glwe_in.size // params.glwe_len()
    out = np.zeros_like(glwe_in)
    _check(lib().fheram_external_product_batch(params.module(), _p(glwe_in.reshape(-1)), n,
                                               _p(np.ascontiguousarray(ggsw, dtype=np.int64)), _p(out.reshape(-1))))
    return out


def coordinate_product(params, glwe_in, ggsws, n_ggsw):
    glwe_in = np.ascontiguousarray(glwe_in, dtype=np.int64)
    n = glwe_in.size // params.glwe_len()
    out = np.zeros_like(glwe_in)
    _check(lib().fheram_coordinate_product(params.module(), _p(glwe_in.reshape(-1)), n,
                                           _p(np.ascontiguousarray(ggsws, dtype=np.int64)), n_ggsw, _p(out.reshape(-1))))
    return out


def glwe_trace(params, keys, glwe_in, start=0, end=None):
    glwe_in = np.ascontiguousarray(glwe_in, dtype=np.int64)
    n = glwe_in.size // params.glwe_len()
    out = np.zeros_like(glwe_in)
    end = params.log_n() if end is None else end
    _check(lib().fheram_glwe_trace(params.module(), keys.h, _p(glwe_in.reshape(-1)), n, start, end, _p(out.reshape(-1))))
    return out


def glwe_pack(params, keys, glwe_in):
    glwe_in = np.ascontiguousarray(glwe_in, dtype=np.int64)
    n = glwe_in.size // params.glwe_len()
    out = np.zeros(params.glwe_len(), dtype=np.int64)
    _check(lib().fheram_glwe_pack(params.module(), keys.h, _p(glwe_in.reshape(-1)), n, _p(out)))
    return out


def glwe_automorphism(params, keys, gal_idx, mode, glwe_in):
    glwe_in = np.ascontiguousarray(glwe_in, dtype=np.int64)
    n = glwe_in.size // params.glwe_len()
    out = np.zeros_like(glwe_in)
    _check(lib().fheram_glwe_automorphism(params.module(), keys.h, gal_idx, mode, 0 if mode == 0 else 1,
                                          _p(glwe_in.reshape(-1)), n, _p(out.reshape(-1))))
    return out


def ggsw_invert(params, keys, ggsw):
    ggsw = np.ascontiguousarray(ggsw, dtype=np.int64)
    n = ggsw.size // params.ggsw_len()
    out = np.zeros_like(ggsw)
    _check(lib().fheram_ggsw_invert(params.module(), keys.h, _p(ggsw.reshape(-1)), n, _p(out.reshape(-1))))
    return out
