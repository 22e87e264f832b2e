"""CPU: the seeded client side (client.cpp).  A seeded RAM is the body columns of fheram_encrypt_ram plus one seed, and
expands to exactly its limbs.  A seeded address keeps the rows with ci = 0 of fheram_encrypt_address; the rows with
ci = 1 carry their plaintext X^pos * s in the body instead of X^pos in the mask, with the same phase.  The oracle reads
with the expanded address and the result decrypts.  No GPU is needed."""
import ctypes as C

import numpy as np
import pytest

SETS = [(1 << 13, 2, 8), (1 << 18, 4, 9), (3 * 4096, 2, 8)]


def _setup(max_addr, word_size, k_pt):
    import fhe_ram_b200 as fr
    params = fr.Parameters.new(max_addr=max_addr, word_size=word_size, k_pt=k_pt)
    sk = fr.GLWESecret.fill_ternary_prob(params, 0.5, fr.Source(7))
    return fr, params, sk


def _full_ram(fr, params, data, sk, xa, xe):
    from fhe_ram_b200 import api
    cts = np.zeros(params.word_size() * params.n_glwe() * params.glwe_len(), dtype=np.int64)
    api._check(api.lib().fheram_encrypt_ram(C.byref(params.c), data.ctypes.data_as(api._PU8), api._p(sk.data),
                                            xa.h, xe.h, api._p(cts)))
    return cts


def _monomials(params, value):
    """client.cpp fheram_address_monomials restated: (pos, sign) of every GGSW"""
    n, out, remain2d = params.n(), [], value
    for digits in params.base2d():
        mx = 1 << sum(digits)
        v = -(remain2d & (mx - 1))
        sign = 1 if v > 0 else (-1 if v < 0 else 0)
        remain, tot = abs(v), 0
        for base in digits:
            chunk = (remain & ((1 << base) - 1)) << tot
            out.append((n - chunk, -1) if sign < 0 and chunk != 0 else (chunk, 1))
            remain >>= base
            tot += base
        remain2d //= mx
    return out


def _normalize(big, K):
    """client.cpp normalize over axis -2 (limbs, most significant first): balanced digits, top carry dropped"""
    out = np.zeros_like(big)
    carry = np.zeros(big.shape[:-2] + big.shape[-1:], dtype=np.int64)
    for l in range(big.shape[-2] - 1, -1, -1):
        t = big[..., l, :] + carry
        d = ((t + (1 << (K - 1))) & ((1 << K) - 1)) - (1 << (K - 1))
        carry = (t - d) >> K
        out[..., l, :] = d
    return out


def _monomial_times(sk, pos, sign):
    """sign * X^pos * s, negacyclic, exact"""
    r = np.roll(sk, pos)
    r[:pos] *= -1
    return sign * r


def _mul_s(a, sk):
    """a * s negacyclic over the last axis; exact: |a| <= 2^17, s ternary, |result| < 2^30 << 2^52"""
    n = a.shape[-1]
    c = np.fft.irfft(np.fft.rfft(a.astype(np.float64), 2 * n) * np.fft.rfft(sk.astype(np.float64), 2 * n), 2 * n)
    c = np.rint(c).astype(np.int64)
    return c[..., :n] - c[..., n:]


def _phase(rows, sk, K):
    """normalize(body + mask * s) of GLWE rows [..., S, 2, N]"""
    return _normalize(rows[..., 0, :] + _mul_s(rows[..., 1, :], sk), K)


@pytest.mark.parametrize("max_addr,word_size,k_pt", SETS)
def test_seeded_ram_is_the_full_encryption(built, max_addr, word_size, k_pt):
    fr, params, sk = _setup(max_addr, word_size, k_pt)
    data = fr.Source(5).fill_bytes(max_addr * word_size)
    xa0, xe0, xa1, xe1 = fr.Source(21), fr.Source(22), fr.Source(21), fr.Source(22)
    xa0.next_u32(); xa1.next_u32()  # a seed that is not at a block or draw boundary
    full = _full_ram(fr, params, data, sk, xa0, xe0)
    seed_before = xa1.seed()
    bodies = np.zeros(full.size // 2, dtype=np.int64)
    seed = np.zeros(1, dtype=fr.api.SEED_DTYPE)
    fr.api._check(fr.api.lib().fheram_encrypt_ram_seeded(C.byref(params.c), data.ctypes.data_as(fr.api._PU8),
                                                         fr.api._p(sk.data), xa1.h, xe1.h, fr.api._p(bodies),
                                                         fr.api._ps(seed, 1)))
    assert seed.tobytes() == seed_before.tobytes()
    S, n = -(-params.k_glwe_ct() // params.basek()), params.n()
    assert np.array_equal(bodies.reshape(-1, S, n), full.reshape(-1, S, 2, n)[:, :, 0, :])
    assert np.array_equal(fr.Ram.expand(params, bodies, seed), full)
    assert xa0.position() == xa1.position() and xe0.position() == xe1.position()
    assert xa0.next_u32() == xa1.next_u32() and xe0.next_u32() == xe1.next_u32()


@pytest.mark.parametrize("max_addr,word_size,k_pt", SETS)
def test_seeded_address_rows(built, max_addr, word_size, k_pt):
    fr, params, sk = _setup(max_addr, word_size, k_pt)
    K, n = params.basek(), params.n()
    S = -(-params.k_ggsw_addr() // K)
    dnum = params.dnum_ct()
    for value in (0, 1, max_addr - 1, (max_addr * 5) // 7):
        xa0, xe0, xa1, xe1 = fr.Source(31), fr.Source(32), fr.Source(31), fr.Source(32)
        full = fr.Address.alloc(params).encrypt_sk(params, value, sk, xa0, xe0).data
        bodies, seed = fr.Address.encrypt_sk_seeded(params, value, sk, xa1, xe1)
        assert xa0.position() == xa1.position() and xe0.position() == xe1.position()
        seeded = fr.Address.expand(params, bodies, seed).data
        full = full.reshape(-1, dnum, 2, S, 2, n)           # [g][row][ci][limb][col][N]
        seeded = seeded.reshape(full.shape)
        assert np.array_equal(bodies.reshape(-1, dnum, 2, S, n), seeded[..., 0, :])
        assert np.array_equal(seeded[:, :, 0], full[:, :, 0])  # ci = 0: fheram_encrypt_address's rows
        mono = _monomials(params, value)
        assert len(mono) == full.shape[0]
        for g, (pos, sign) in enumerate(mono):
            for r in range(dnum):
                want_mask = full[g, r, 1, :, 1, :].copy()
                want_mask[r, pos] -= sign                      # the plaintext leaves the mask ...
                assert np.array_equal(seeded[g, r, 1, :, 1, :], want_mask)
                big = full[g, r, 1, :, 0, :].copy()
                big[r] += _monomial_times(sk.data, pos, sign)  # ... and enters the body as X^pos * s
                assert np.array_equal(seeded[g, r, 1, :, 0, :], _normalize(big, K))
        # every row: the phase of the full encryption, bit for bit
        assert np.array_equal(_phase(seeded, sk.data, K), _phase(full, sk.data, K))


@pytest.mark.parametrize("max_addr,word_size,k_pt", [(1 << 13, 2, 8), (3 * 4096, 2, 8)])
def test_oracle_reads_with_an_expanded_seeded_address(built, max_addr, word_size, k_pt):
    from oracle.oracle import Oracle
    fr, params, sk = _setup(max_addr, word_size, k_pt)
    evk = fr.EvaluationKeys.encrypt_sk(params, sk, fr.Source(8), fr.Source(9))
    data = fr.Source(5).fill_bytes(max_addr * word_size)
    cts = _full_ram(fr, params, data, sk, fr.Source(11), fr.Source(12))
    orc = Oracle(backend="fft64", max_addr=max_addr, word_size=word_size, k_pt=k_pt)
    okeys = orc.keys_prepare(evk.atk_glwe, evk.gglwe_to_ggsw_key, evk.atk_ggsw_inv)
    oram = orc.ram_new(cts.copy())
    xa, xe = fr.Source(21), fr.Source(22)
    for idx in (0, max_addr - 1, 4097 % max_addr):
        bodies, seed = fr.Address.encrypt_sk_seeded(params, idx, sk, xa, xe)
        rc, got = orc.ram_read(oram, fr.Address.expand(params, bodies, seed).data, okeys)
        assert rc == 0
        for i in range(word_size):
            w = fr.cast_u8_to_signed(int(data[i + word_size * idx]), min(8, k_pt))
            v, noise = fr.decrypt_glwe(params, got[i], w, sk)
            assert v == w and noise < -(k_pt + 1), (idx, i, v, w, noise)


def test_bad_arguments_are_refused(built):
    import fhe_ram_b200 as fr
    from fhe_ram_b200 import api
    _, params, sk = _setup(1 << 13, 2, 8)
    L = api.lib()
    xa, xe = fr.Source(1), fr.Source(2)
    bodies = np.zeros(params.n_ggsw() * params.ggsw_len() // 2, dtype=np.int64)
    seed = np.zeros(1, dtype=api.SEED_DTYPE)
    ps = api._ps(seed, 1)
    pc = C.byref(params.c)
    pos = (xa.position(), xe.position())
    assert L.fheram_encrypt_address_seeded(pc, 3, api._p(sk.data), xa.h, xa.h, api._p(bodies), ps) == -1  # xa == xe
    assert L.fheram_encrypt_address_seeded(pc, params.max_addr(), api._p(sk.data), xa.h, xe.h, api._p(bodies),
                                           ps) == -1  # address out of range
    assert "out of range" in L.fheram_last_error().decode()
    assert L.fheram_encrypt_address_seeded(pc, 3, api._p(sk.data), xa.h, xe.h, None, ps) == -1
    assert L.fheram_encrypt_address_seeded(pc, 3, api._p(sk.data), xa.h, xe.h, api._p(bodies), None) == -1
    assert L.fheram_encrypt_address_seeded(pc, 3, None, xa.h, xe.h, api._p(bodies), ps) == -1
    assert (xa.position(), xe.position()) == pos  # nothing was drawn
    data = np.zeros(params.max_addr() * params.word_size(), dtype=np.uint8)
    rb = np.zeros(params.word_size() * params.n_glwe() * params.glwe_len() // 2, dtype=np.int64)
    pd = data.ctypes.data_as(api._PU8)
    assert L.fheram_encrypt_ram_seeded(pc, pd, api._p(sk.data), xe.h, xe.h, api._p(rb), ps) == -1
    assert L.fheram_encrypt_ram_seeded(pc, None, api._p(sk.data), xa.h, xe.h, api._p(rb), ps) == -1
    assert L.fheram_encrypt_ram_seeded(pc, pd, api._p(sk.data), xa.h, xe.h, api._p(rb), None) == -1
    assert (xa.position(), xe.position()) == pos
    out = np.zeros(2 * rb.size, dtype=np.int64)
    assert L.fheram_ram_expand(pc, None, ps, api._p(out)) == -1
    assert L.fheram_ram_expand(pc, api._p(rb), None, api._p(out)) == -1
    assert L.fheram_address_expand(pc, api._p(bodies), ps, None) == -1
    assert L.fheram_source_seed(None, ps) == -1 and L.fheram_source_seed(xa.h, None) == -1
    bad = fr.Parameters.new(max_addr=1 << 13, word_size=2, k_pt=8, n_decomp=0)
    assert L.fheram_address_expand(C.byref(bad.c), api._p(bodies), ps, api._p(out)) == -1
