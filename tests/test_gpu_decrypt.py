"""Decryption on the device (DESIGN.md 3.7): fheram_ram_decrypt_sk returns, bit for bit, what the CPU client side
(fheram_decrypt_ram, checked against an exact restatement in test_decrypt_client.py) returns on fheram_ram_store's
output, before and after writes, on sharded RAMs too; fheram_decrypt_words_device decodes read results as
fheram_decrypt_word does."""
import numpy as np
import pytest

SETS = [(1 << 13, 2, 8), (1 << 12, 1, 3), (5000, 3, 9), (1 << 18, 4, 9)]


def _plaintext(fr, params, data):
    w = min(8, params.k_glwe_pt())
    table = np.array([fr.cast_u8_to_signed(b, w) for b in range(256)], dtype=np.int16)
    return table[np.asarray(data, dtype=np.uint8).reshape(params.max_addr(), params.word_size())]


def _setup(max_addr, word_size, k_pt):
    import fhe_ram_b200 as fr
    params = fr.Parameters.new(max_addr=max_addr, word_size=word_size, k_pt=k_pt)
    sk = fr.GLWESecret.fill_ternary_prob(params, 0.5, fr.Source(7))
    data = fr.Source(5).fill_bytes(max_addr * word_size)
    return fr, params, sk, data


@pytest.mark.gpu
@pytest.mark.parametrize("max_addr,word_size,k_pt", SETS)
def test_fresh_ram_decrypts_as_the_client_side(built, max_addr, word_size, k_pt):
    fr, params, sk, data = _setup(max_addr, word_size, k_pt)
    ram = fr.Ram.new(params)
    ram.encrypt_sk_gpu(data, sk, fr.Source(21), fr.Source(22))
    values, err = ram.decrypt_sk(sk)
    want_v, want_e = fr.decrypt_ram(params, ram.store(), sk)
    assert np.array_equal(values, want_v)
    assert np.array_equal(err, want_e)
    assert np.array_equal(values, _plaintext(fr, params, data))
    ram.close()


def _word(fr, params, value, sk):
    return fr.encrypt_glwe(params, int(value), sk)


@pytest.mark.gpu
def test_decrypted_ram_follows_writes(built):
    fr, params, sk, data = _setup(1 << 13, 2, 8)
    ws = params.word_size()
    keys = fr.EvaluationKeysPrepared.encrypt_sk_gpu(params, sk, fr.Source(3), fr.Source(4))
    ram = fr.Ram.new(params)
    ram.encrypt_sk_gpu(data, sk, fr.Source(21), fr.Source(22))
    model = data.copy()
    xa, xe = fr.Source(31), fr.Source(32)
    for idx, word in [(5, (1, 2)), (4095, (200, 17)), (4096, (128, 255)), (5, (99, 0)), (8191, (7, 77))]:
        addr = fr.Address.alloc(params).encrypt_sk(params, idx, sk, xa, xe)
        ram.read_prepare_write(addr, keys)
        ram.write(np.stack([_word(fr, params, v, sk) for v in word]), addr, keys)
        model[idx * ws:(idx + 1) * ws] = word
        addr.close()
    values, err = ram.decrypt_sk(sk)
    assert np.array_equal(values, _plaintext(fr, params, model))
    want_v, want_e = fr.decrypt_ram(params, ram.store(), sk)
    assert np.array_equal(values, want_v) and np.array_equal(err, want_e)
    ram.close(); keys.close()


@pytest.mark.gpu
def test_errors_and_recovery(built):
    fr, params, sk, data = _setup(1 << 13, 2, 8)
    keys = fr.EvaluationKeysPrepared.encrypt_sk_gpu(params, sk, fr.Source(3), fr.Source(4))
    never = fr.Ram.new(params)
    with pytest.raises(fr.FheRamError) as e:
        never.decrypt_sk(sk)
    assert e.value.code == -4
    never.close()
    ram = fr.Ram.new(params)
    ram.encrypt_sk_gpu(data, sk, fr.Source(21), fr.Source(22))
    bad = sk.data.copy()
    bad[3] = -2
    with pytest.raises(fr.FheRamError) as e:
        ram.decrypt_sk(bad)
    assert e.value.code == -1
    idx = 777
    addr = fr.Address.alloc(params).encrypt_sk(params, idx, sk, fr.Source(31), fr.Source(32))
    ram.read_prepare_write(addr, keys)
    with pytest.raises(fr.FheRamError) as e:
        ram.decrypt_sk(sk)
    assert e.value.code == -2
    ram.write(np.stack([_word(fr, params, v, sk) for v in (42, 211)]), addr, keys)
    got = ram.read(addr, keys)
    for i, v in enumerate((42, 211)):
        w = fr.cast_u8_to_signed(v, 8)
        assert fr.decrypt_glwe(params, got[i], w, sk)[0] == w
    model = data.copy()
    model[2 * idx:2 * idx + 2] = (42, 211)
    values, _ = ram.decrypt_sk(sk)
    assert np.array_equal(values, _plaintext(fr, params, model))
    ram.close(); addr.close(); keys.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_shards", [2, 4])
def test_sharded_ram_fills_its_own_entries(built, n_shards):
    fr, params, sk, data = _setup(3 * 4096 + 100, 2, 8)  # four polynomials, the last one partly used
    n, ws = params.n(), params.word_size()
    full = fr.Ram.new(params)
    full.encrypt_sk_gpu(data, sk, fr.Source(21), fr.Source(22))
    want_v, want_e = full.decrypt_sk(sk)
    full.close()
    h_of = np.arange(params.max_addr()) // n
    union_v = np.full_like(want_v, -32768)
    union_e = np.full_like(want_e, -(1 << 62))
    for shard in range(n_shards):
        r = fr.Ram(params, shard, n_shards)
        r.encrypt_sk_gpu(data, sk, fr.Source(21), fr.Source(22))
        v = np.full_like(want_v, -32768)
        e = np.full_like(want_e, -(1 << 62))
        r.decrypt_sk(sk, v, e)
        mine = h_of % n_shards == shard
        assert np.array_equal(v[mine], want_v[mine]) and np.array_equal(e[mine], want_e[mine])
        assert (v[~mine] == -32768).all() and (e[~mine] == -(1 << 62)).all()
        union_v[mine], union_e[mine] = v[mine], e[mine]
        r.close()
    assert np.array_equal(union_v, want_v) and np.array_equal(union_e, want_e)
    assert np.array_equal(union_v, _plaintext(fr, params, data))


@pytest.mark.gpu
def test_decrypt_words_device_on_a_read_batch(built):
    import ctypes as C
    from fhe_ram_b200 import api
    fr, params, sk, data = _setup(1 << 13, 2, 8)
    ws = params.word_size()
    keys = fr.EvaluationKeysPrepared.encrypt_sk_gpu(params, sk, fr.Source(3), fr.Source(4))
    ram = fr.Ram.new(params)
    ram.encrypt_sk_gpu(data, sk, fr.Source(21), fr.Source(22))
    idxs = (np.arange(64) * 127 + 3) % params.max_addr()
    addrs = fr.Address.encrypt_sk_gpu(params, idxs, sk, fr.Source(41), fr.Source(42))
    d = ram.read_batch_device(addrs, keys)
    n = len(idxs) * ws
    values, err = fr.decrypt_words_device(params, d, n, sk)
    want = _plaintext(fr, params, data)[idxs].reshape(-1)
    assert np.array_equal(values, want)
    limbs = np.zeros(n * params.glwe_len(), dtype=np.int64)
    api._check(api.lib().fheram_download_glwe(params.module(), C.c_void_p(d), n, api._p(limbs)))
    limbs = limbs.reshape(n, -1)
    k_pt, k_ct = params.k_glwe_pt(), params.k_glwe_ct()
    for j in range(n):
        raw, _ = fr.decrypt_glwe(params, limbs[j], 0, sk)
        _, noise = fr.decrypt_glwe(params, limbs[j], raw, sk)
        assert values[j] == ((raw + (1 << (k_pt - 1))) & ((1 << k_pt) - 1)) - (1 << (k_pt - 1))
        e = int(err[j])
        assert noise == (np.log2(float(abs(e))) - k_ct if e else -np.inf)
    ram.close(); addrs.close(); keys.close()
