"""fhe_ram_b200 -- B200-native (sm_100a) FHE-RAM read / read_prepare_write / write.

The package holds only what the hot path needs: csrc/ (CUDA kernels + the C ABI declared in
include/fheram.h), cpp/ (the compiled-language mirror of the reference's Rust API) and api.py
(ctypes binding used by tests and bench).  See DESIGN.md and INTEGRATION.md.
"""
from .api import (  # noqa: F401
    Address, EvaluationKeys, EvaluationKeysPrepared, FheRamError, GLWESecret, Parameters, Ram,
    Source, cast_u8_to_signed, decrypt_glwe, decrypt_ram, decrypt_words_device, encrypt_glwe, gen_keys,
)
