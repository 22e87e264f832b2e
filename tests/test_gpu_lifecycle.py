"""-m gpu: every device allocation of the library has an owner.  fheram_debug_device_bytes() counts the bytes the
library holds; after creation calls that fail and after a whole lifecycle of handles it is back where it started.
The failures are range errors the library reports for a limb outside +-2^30: nothing goes wrong on the device."""
import contextlib
import ctypes as C
import gc

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ERR_RANGE = -6


def _device_bytes() -> int:
    from fhe_ram_b200 import api
    return int(api.lib().fheram_debug_device_bytes())


@contextlib.contextmanager
def _device_bytes_unchanged():
    # handles of other tests that the garbage collector frees in the middle would move the count
    gc.collect()
    gc.disable()
    try:
        before = _device_bytes()
        yield
        assert _device_bytes() == before
    finally:
        gc.enable()


@pytest.fixture(scope="module")
def params(built):
    import fhe_ram_b200 as fr
    p = fr.Parameters.new(max_addr=1 << 13, word_size=2, k_pt=8)
    p.module()
    yield p
    p.close()


def _fails_without_leaking(attempt, times=20):
    attempt()  # the first call grows the context's staging buffers, which the context keeps
    with _device_bytes_unchanged():
        for _ in range(times):
            attempt()


def test_keys_prepare_range_error_frees_everything(params):
    from fhe_ram_b200 import api
    p = params
    atk = np.zeros(p.n_trace_keys() * p.atk_len(), dtype=np.int64)
    atk[1234] = 1 << 40
    tsk = np.zeros(p.evk_inv_len(), dtype=np.int64)
    inv = np.zeros(p.evk_inv_len(), dtype=np.int64)

    def attempt():
        h = C.c_void_p()
        rc = api.lib().fheram_keys_prepare(p.module(), api._p(atk), api._p(tsk), api._p(inv), C.byref(h))
        assert rc == ERR_RANGE and not h.value

    _fails_without_leaking(attempt)


def test_address_load_batch_range_error_frees_everything(params):
    from fhe_ram_b200 import api
    p, n = params, 8
    limbs = np.zeros(n * p.n_ggsw() * p.ggsw_len(), dtype=np.int64)
    limbs[-5] = 1 << 40

    def attempt():
        h = C.c_void_p()
        rc = api.lib().fheram_address_load_batch(p.module(), api._p(limbs), n, C.byref(h))
        assert rc == ERR_RANGE and not h.value

    _fails_without_leaking(attempt)


def test_address_load_seeded_range_error_frees_everything(params):
    from fhe_ram_b200 import api
    p, n = params, 8
    bodies = np.zeros(n * p.n_ggsw() * p.ggsw_len() // 2, dtype=np.int64)
    bodies[7] = -(1 << 40)
    seeds = np.zeros(n, dtype=api.SEED_DTYPE)

    def attempt():
        h = C.c_void_p()
        rc = api.lib().fheram_address_load_seeded(p.module(), api._p(bodies), api._ps(seeds, n), n, C.byref(h))
        assert rc == ERR_RANGE and not h.value

    _fails_without_leaking(attempt)


def test_full_lifecycle_returns_every_byte(built):
    """context with phase counters on, keys, addresses, RAM, a host-pipeline batch, rpw + write and a device decrypt
    at 2^18 x 4 B, then every handle destroyed"""
    import fhe_ram_b200 as fr
    from fhe_ram_b200 import api
    p = fr.Parameters.new(max_addr=1 << 18, word_size=4, k_pt=8)
    sk, evk = fr.gen_keys(p)
    data = fr.Source(5).fill_bytes(p.max_addr() * p.word_size())
    xa, xe = fr.Source(11), fr.Source(12)
    idxs = [3, 200_001]
    limbs = np.concatenate([fr.Address.alloc(p).encrypt_sk(p, i, sk, xa, xe).data for i in idxs])
    w = np.stack([fr.encrypt_glwe(p, v, sk) for v in (1, 2, 3, 4)])
    with _device_bytes_unchanged():
        before = _device_bytes()
        api._check(api.lib().fheram_debug_phase_cycles(p.module(), 1, (C.c_longlong * 8)()))
        keys = fr.EvaluationKeysPrepared.alloc(p).prepare(evk)
        ram = fr.Ram.new(p)
        ram.encrypt_sk(data, sk, xa, xe)
        got = ram.read_batch_host_i32(limbs, len(idxs), keys)
        addr = fr.Address.from_limbs(p, limbs[:limbs.size // 2])
        ram.read_prepare_write(addr, keys)
        ram.write(w, addr, keys)
        values, _ = ram.decrypt_sk(sk)
        assert _device_bytes() > before
        ram.close()
        addr.close()
        keys.close()
        p.close()
    # the calls did their work: the batch read the two entries, the write landed at entry 3
    for j, i in enumerate(idxs):
        for b in range(p.word_size()):
            want = fr.cast_u8_to_signed(int(data[i * p.word_size() + b]), p.k_glwe_pt())
            assert fr.decrypt_glwe(p, got[j, b].astype(np.int64), want, sk)[0] == want
    assert list(values[3]) == [1, 2, 3, 4]
