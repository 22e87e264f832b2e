"""CPU: the definitions of read_plain and write_plain (include/fheram.h, DESIGN.md 3.8), restated with the oracle's
glwe_rotate, trace and glwe_normalize plus numpy integer arithmetic, on an oracle-encrypted RAM.

  read_plain:  out[s] = TRACE(rot(2N - j, data[s][h]))                            for a = h N + j
  write_plain: data[s][h] <- normalize(data[s][h] - rot(j, T_s) + rot(j, w_s)),   T_s = TRACE(rot(2N - j, data[s][h]))

The read decrypts to the byte at a; after the write, the RAM decrypts to the old bytes everywhere except the word_size
bytes of a, with every error far inside the rounding margin."""
import numpy as np
import pytest

MAX_ADDR, WS, K_PT = 1 << 13, 2, 8


def plain_read(orc, okeys, cts, a):
    """[word_size] GLWE: the restated read_plain of address a"""
    N = orc.n
    h, j = a // N, a % N
    polys = cts.reshape(WS, orc.n_glwe, orc.glwe_len)
    return np.stack([orc.trace(okeys, orc.glwe_rotate(2 * N - j, polys[s, h])) for s in range(WS)])


def plain_write(orc, okeys, cts, a, w):
    """the RAM after the restated write_plain of the words w ([word_size] GLWE) at address a"""
    N = orc.n
    h, j = a // N, a % N
    out = cts.copy().reshape(WS, orc.n_glwe, orc.glwe_len)
    T = plain_read(orc, okeys, cts, a)
    for s in range(WS):
        out[s, h] = orc.glwe_normalize(out[s, h] - orc.glwe_rotate(j, T[s]) + orc.glwe_rotate(j, w[s]))
    return out.reshape(-1)


@pytest.fixture(scope="module")
def setup(built):
    import fhe_ram_b200 as fr
    from oracle.oracle import Oracle
    orc = Oracle(backend="fft64", max_addr=MAX_ADDR, word_size=WS, k_pt=K_PT)
    sk = orc.secret_gen(orc.source(0))
    atk, tsk, inv = orc.keygen(sk, orc.source(1), orc.source(2))
    okeys = orc.keys_prepare(atk, tsk, inv)
    data = orc.source_bytes(orc.source(5), MAX_ADDR * WS)
    cts = orc.ram_encrypt(data, sk, orc.source(11), orc.source(12))
    params = fr.Parameters.new(max_addr=MAX_ADDR, word_size=WS, k_pt=K_PT)
    return fr, orc, okeys, sk, data, cts, params


def _byte(orc, b):
    return orc.cast_u8_to_signed(int(b), min(8, K_PT))


@pytest.mark.parametrize("a", [0, 1, 4095, 4096, MAX_ADDR - 1])
def test_restated_read_plain_decrypts_to_the_data(setup, a):
    fr, orc, okeys, sk, data, cts, params = setup
    got = plain_read(orc, okeys, cts, a)
    for s in range(WS):
        want = _byte(orc, data[a * WS + s])
        v, noise = orc.decrypt_glwe(got[s], sk, want)
        assert v == want and noise < -(K_PT + 1), (a, s, v, want, noise)


@pytest.mark.parametrize("a", [1, 4095, 4096 + 77])
def test_restated_write_plain_changes_exactly_one_word(setup, a):
    fr, orc, okeys, sk, data, cts, params = setup
    new = np.array([200, 7], dtype=np.uint8)
    w = np.stack([orc.encrypt_byte(int(new[s]), sk, orc.source(30 + s), orc.source(40 + s)) for s in range(WS)])
    after = plain_write(orc, okeys, cts, a, w)
    values, err = fr.decrypt_ram(params, after, sk)
    want = np.array([_byte(orc, b) for b in data], dtype=np.int16).reshape(MAX_ADDR, WS)
    want[a] = [_byte(orc, b) for b in new]
    assert np.array_equal(values, want), np.argwhere(values != want)[:8]
    # one trace's noise on the N cells of polynomial h; the rounding margin is 2^(k_ct - k_pt - 1)
    ls = params.k_glwe_ct() - K_PT
    worst = int(np.abs(err).max())
    assert worst < 1 << (ls - 10), (worst.bit_length(), ls)
    # the other polynomials keep their limbs
    h = a // orc.n
    before = cts.reshape(WS, orc.n_glwe, -1)
    moved = after.reshape(WS, orc.n_glwe, -1)
    for hh in range(orc.n_glwe):
        assert np.array_equal(before[:, hh], moved[:, hh]) == (hh != h)
