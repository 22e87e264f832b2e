"""CPU: fheram_decrypt_ram (client.cpp) returns every byte of a RAM from fheram_encrypt_ram's output, its errors equal an
exact integer restatement of the decryption (mask * s by signed shifts over the secret's nonzero coefficients), and
coefficient 0 of every GLWE agrees with fheram_decrypt_word.  No GPU is needed."""
import ctypes as C

import numpy as np
import pytest

SETS = [(1 << 13, 2, 8), (1 << 12, 1, 3), (5000, 3, 9)]  # the last: max_addr not a multiple of N


def _encrypted(max_addr, word_size, k_pt, seed=5):
    import fhe_ram_b200 as fr
    from fhe_ram_b200 import api
    params = fr.Parameters.new(max_addr=max_addr, word_size=word_size, k_pt=k_pt)
    sk = fr.GLWESecret.fill_ternary_prob(params, 0.5, fr.Source(seed))
    data = fr.Source(seed + 1).fill_bytes(max_addr * word_size)
    cts = np.zeros(word_size * params.n_glwe() * params.glwe_len(), dtype=np.int64)
    api._check(api.lib().fheram_encrypt_ram(C.byref(params.c), data.ctypes.data_as(api._PU8), api._p(sk.data),
                                            fr.Source(seed + 2).h, fr.Source(seed + 3).h, api._p(cts)))
    return fr, params, sk, data, cts


def _plaintext(fr, params, data):
    w = min(8, params.k_glwe_pt())
    table = np.array([fr.cast_u8_to_signed(b, w) for b in range(256)], dtype=np.int16)
    return table[data.reshape(params.max_addr(), params.word_size())]


def _reference(params, cts, sk):
    """items 1-5 of the decryption in exact integers: (values, err) [max_addr][word_size]"""
    n, K, k_ct, k_pt, ws, G = params.n(), params.basek(), params.k_glwe_ct(), params.k_glwe_pt(), \
        params.word_size(), params.n_glwe()
    S = -(-k_ct // K)
    c = cts.reshape(ws * G, S, 2, n)
    a = c[:, :, 1, :].reshape(-1, n)
    prod = np.zeros_like(a)
    for k in np.flatnonzero(sk):  # a * X^k, negacyclic: the k entries that wrap change sign
        r = np.roll(a, k, axis=1)
        r[:, :k] *= -1
        prod += int(sk[k]) * r
    big = c[:, :, 0, :] + prod.reshape(ws * G, S, n)
    pt = np.zeros_like(big)
    carry = np.zeros((ws * G, n), dtype=np.int64)
    for l in range(S - 1, -1, -1):  # client.cpp normalize: balanced digits, top carry dropped
        t = big[:, l, :] + carry
        d = ((t + (1 << (K - 1))) & ((1 << K) - 1)) - (1 << (K - 1))
        carry = (t - d) >> K
        pt[:, l, :] = d
    v = sum(pt[:, l, :] << (K * (S - 1 - l)) for l in range(S)) >> (S * K - k_ct)
    ls = k_ct - k_pt
    half = 1 << (ls - 1)
    raw = np.where(v >= 0, (v + half) >> ls, -((half - v) >> ls))
    err = v - raw * (1 << ls)
    value = ((raw + (1 << (k_pt - 1))) & ((1 << k_pt) - 1)) - (1 << (k_pt - 1))
    # GLWE (i, h) coefficient j -> entry [h N + j][i]
    value = value.reshape(ws, G * n).T[:params.max_addr()]
    err = err.reshape(ws, G * n).T[:params.max_addr()]
    return value.astype(np.int16), np.ascontiguousarray(err)


@pytest.mark.parametrize("max_addr,word_size,k_pt", SETS)
def test_decrypt_ram_returns_the_plaintext_and_exact_errors(built, max_addr, word_size, k_pt):
    fr, params, sk, data, cts = _encrypted(max_addr, word_size, k_pt)
    values, err = fr.decrypt_ram(params, cts, sk)
    assert values.shape == (max_addr, word_size) and values.dtype == np.int16
    assert np.array_equal(values, _plaintext(fr, params, data))
    want_v, want_e = _reference(params, cts, sk.data)
    assert np.array_equal(values, want_v)
    assert np.array_equal(err, want_e)
    # fresh encryption noise: sigma 3.2 at 2^-k_ct, far below the 2^(k_ct - k_pt - 1) decision bound
    assert np.abs(err).max() < 1 << 8


@pytest.mark.parametrize("max_addr,word_size,k_pt", SETS)
def test_coefficient_zero_agrees_with_decrypt_word(built, max_addr, word_size, k_pt):
    fr, params, sk, data, cts = _encrypted(max_addr, word_size, k_pt)
    values, err = fr.decrypt_ram(params, cts, sk)
    n, G = params.n(), params.n_glwe()
    c = cts.reshape(word_size, G, -1)
    for i in range(word_size):
        for h in range(G):
            raw, _ = fr.decrypt_glwe(params, c[i, h], 0, sk)
            got, noise = fr.decrypt_glwe(params, c[i, h], raw, sk)
            assert got == raw
            red = ((raw + (1 << (k_pt - 1))) & ((1 << k_pt) - 1)) - (1 << (k_pt - 1))
            assert values[h * n, i] == red
            e = int(err[h * n, i])
            assert noise == (np.log2(float(abs(e))) - params.k_glwe_ct() if e else -np.inf)


def test_errors_are_optional(built):
    from fhe_ram_b200 import api
    fr, params, sk, data, cts = _encrypted(1 << 12, 1, 3)
    values = np.zeros((params.max_addr(), 1), dtype=np.int16)
    api._check(api.lib().fheram_decrypt_ram(C.byref(params.c), api._p(cts), api._p(sk.data),
                                            values.ctypes.data_as(C.POINTER(C.c_int16)), None))
    assert np.array_equal(values, _plaintext(fr, params, data))


def test_non_ternary_secret_is_rejected(built):
    fr, params, sk, data, cts = _encrypted(1 << 12, 1, 3)
    bad = sk.data.copy()
    bad[17] = 2
    with pytest.raises(fr.FheRamError) as e:
        fr.decrypt_ram(params, cts, bad)
    assert e.value.code == -1 and "ternary" in str(e.value)
