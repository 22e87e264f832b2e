"""CPU: the address decomposition `decomp_n` (Parameters.new(decomp_n=...), Ram::new_from_ram_params) at every shape
the library must handle, not only the default [3, 3, 3, 3].  The digit table sets the Base2D coordinates (src/base.rs:
84-108), hence the number of GGSWs of an address and the monomial each GGSW encrypts (src/address.rs:102-108,
src/coordinate.rs:148-179).  For each table below the host side must agree with a plain restatement of those rules and
with the oracle limb for limb, in the full and in the seeded form.  No GPU is needed."""
import ctypes as C

import numpy as np
import pytest

# (decomp_n, max_addr, word_size, Base2D coordinates); tests/test_gpu_decompositions.py runs the same sets on the device
SETS = [
    ([12], 1 << 13, 2, [[12], [1]]),
    ([5, 7], 1 << 12, 1, [[5, 7]]),
    ([4, 4, 4], 5 * 4096 + 17, 1, [[4, 4, 4], [3]]),
    ([2] * 6, 1 << 14, 2, [[2] * 6, [2]]),
    ([1, 11], 1 << 15, 1, [[1, 11], [1, 2]]),
    ([1] * 7 + [5], 1 << 20, 1, [[1] * 7 + [5], [1] * 8]),
    ([3, 3, 3, 3], 1 << 21, 1, [[3, 3, 3, 3], [3, 3, 3]]),
]
IDS = ["-".join(map(str, d)) for d, *_ in SETS]


def _params(decomp, max_addr, word_size):
    import fhe_ram_b200 as fr
    return fr.Parameters.new(max_addr=max_addr, word_size=word_size, k_pt=8, decomp_n=decomp)


def _base2d(max_addr, decomp):
    """get_base_2d (src/base.rs:84-108): the bits of max_addr - 1 cut into coordinates, each taking the digits of
    decomp_n in turn, the last digit cut short where the bits run out"""
    bits, out = (max_addr - 1).bit_length(), []
    while bits:
        coord = []
        for b in decomp:
            if b > bits:
                if bits:
                    coord.append(bits)
                    bits = 0
                break
            coord.append(b)
            bits -= b
        out.append(coord)
    return out


def _monomials(value, coords, n):
    """(pos, sign) of every GGSW of Address::encrypt_sk(value): coordinate c holds the value's next sum(coords[c])
    bits, and its digit d_j at bit offset o_j is encrypted as X^-(d_j << o_j)"""
    out = []
    for digits in coords:
        x = value & ((1 << sum(digits)) - 1)
        value >>= sum(digits)
        off = 0
        for b in digits:
            e = ((x >> off) & ((1 << b) - 1)) << off
            out.append((n - e, -1) if e else (0, 1))
            off += b
    return out


def _values(max_addr, coords):
    """0, 1, max_addr - 1 and, for every digit, the address with that digit at its maximum and all others zero"""
    vals, off = {0, 1, max_addr - 1}, 0
    for digits in coords:
        for b in digits:
            vals.add(((1 << b) - 1) << off)
            off += b
    return sorted(v for v in vals if v < max_addr)


def test_the_table_restates_base2d():
    for decomp, max_addr, _, coords in SETS:
        assert _base2d(max_addr, decomp) == coords, decomp


@pytest.mark.parametrize("decomp,max_addr,word_size,coords", SETS, ids=IDS)
def test_digit_counts_match_the_oracle(built, decomp, max_addr, word_size, coords):
    from oracle.oracle import Oracle
    p = _params(decomp, max_addr, word_size)
    o = Oracle(backend="fft64", max_addr=max_addr, word_size=word_size, k_pt=8, decomp_n=decomp)
    assert p.decomp_n() == decomp
    assert p.base2d() == o.base2d() == coords
    assert p.n_ggsw() == o.n_ggsw == sum(map(len, coords))
    assert p.n_glwe() == o.n_glwe == -(-max_addr // p.n())


@pytest.mark.parametrize("decomp,max_addr,word_size,coords", SETS, ids=IDS)
def test_address_encodes_the_restated_monomials(built, decomp, max_addr, word_size, coords):
    """every GGSW of Address::encrypt_sk(v) decrypts (row 0, first limb) to the monomial of the restatement"""
    import fhe_ram_b200 as fr
    from oracle.oracle import Oracle
    p = _params(decomp, max_addr, word_size)
    o = Oracle(backend="fft64", max_addr=max_addr, word_size=word_size, k_pt=8, decomp_n=decomp)
    sk = fr.GLWESecret.fill_ternary_prob(p, 0.5, fr.Source(0))
    vals = _values(max_addr, coords)
    assert len(vals) >= sum(map(len, coords))
    L, n = p.ggsw_len(), p.n()
    for v in vals:
        a = fr.Address.alloc(p).encrypt_sk(p, v, sk, fr.Source(9), fr.Source(10))
        for g, (pos, sign) in enumerate(_monomials(v, coords, n)):
            pt = o.ggsw_decrypt_row(a.data[g * L:(g + 1) * L], 0, 0, sk.data)[0]
            want = np.zeros(n, dtype=np.int64)
            want[pos] = sign
            assert np.array_equal(pt, want), (v, g, pos, sign, np.nonzero(pt)[0][:4])
    with pytest.raises(fr.FheRamError):  # address out of range
        fr.Address.alloc(p).encrypt_sk(p, max_addr, sk, fr.Source(9), fr.Source(10))


def _normalize(big, K):
    """balanced base-2^K digits over axis -2 (limbs, most significant first), top carry dropped"""
    out = np.zeros_like(big)
    carry = np.zeros(big.shape[:-2] + big.shape[-1:], dtype=np.int64)
    for l in range(big.shape[-2] - 1, -1, -1):
        t = big[..., l, :] + carry
        d = ((t + (1 << (K - 1))) & ((1 << K) - 1)) - (1 << (K - 1))
        carry = (t - d) >> K
        out[..., l, :] = d
    return out


def _phase(rows, sk, K):
    """normalize(body + mask * s) of GLWE rows [..., limbs, 2, N]; the product is exact in float64
    (|mask| <= 2^16, s ternary, N = 4096: |result| < 2^29)"""
    n = rows.shape[-1]
    a = rows[..., 1, :].astype(np.float64)
    c = np.fft.irfft(np.fft.rfft(a, 2 * n) * np.fft.rfft(sk.astype(np.float64), 2 * n), 2 * n)
    c = np.rint(c).astype(np.int64)
    return _normalize(rows[..., 0, :] + c[..., :n] - c[..., n:], K)


@pytest.mark.parametrize("decomp,max_addr,word_size,coords", SETS, ids=IDS)
def test_address_limbs_match_the_oracle(built, decomp, max_addr, word_size, coords):
    """Address::encrypt_sk against the oracle's restatement, and the seeded form expanded on the CPU against it (same
    mask rows for ci = 0, same phase for every row)"""
    import fhe_ram_b200 as fr
    from oracle.oracle import Oracle
    p = _params(decomp, max_addr, word_size)
    o = Oracle(backend="fft64", max_addr=max_addr, word_size=word_size, k_pt=8, decomp_n=decomp)
    sk = fr.GLWESecret.fill_ternary_prob(p, 0.5, fr.Source(0))
    assert np.array_equal(sk.data, o.secret_gen(o.source(0)))
    K, n, dnum = p.basek(), p.n(), p.dnum_ct()
    S = -(-p.k_ggsw_addr() // K)
    for v in (max_addr - 1, _values(max_addr, coords)[-2]):
        full = fr.Address.alloc(p).encrypt_sk(p, v, sk, fr.Source(9), fr.Source(10)).data
        assert full.size == p.n_ggsw() * p.ggsw_len()
        assert np.array_equal(full, o.address_encrypt(v, sk.data, o.source(9), o.source(10))), v
        bodies, seed = fr.Address.encrypt_sk_seeded(p, v, sk, fr.Source(9), fr.Source(10))
        seeded = fr.Address.expand(p, bodies, seed).data.reshape(-1, dnum, 2, S, 2, n)  # [g][row][ci][limb][col][N]
        full = full.reshape(seeded.shape)
        assert np.array_equal(seeded[..., 0, :], bodies.reshape(-1, dnum, 2, S, n))
        assert np.array_equal(seeded[:, :, 0], full[:, :, 0]), v
        assert np.array_equal(_phase(seeded, sk.data, K), _phase(full, sk.data, K)), v


@pytest.mark.parametrize("decomp,n_decomp", [([3, 3, 3], 3), ([4, 4, 5], 3), ([6, 7], 2), ([0, 6, 6], 3),
                                             ([3, 0, 3, 3, 3], 5), ([1] * 8, 9), ([3, 3, 3, 3], 0)])
def test_invalid_tables_are_refused(built, decomp, n_decomp):
    """sum(decomp_n) != log_n, a zero digit, more than eight entries or none: FHERAM_ERR_INVALID from every entry point
    that takes parameters, before any device is touched"""
    import fhe_ram_b200 as fr
    from fhe_ram_b200 import api
    p = _params(decomp, 1 << 13, 1)
    p.c.n_decomp = n_decomp
    L = api.lib()
    lens, digits = (C.c_int32 * 8)(), (C.c_int32 * 64)()
    assert L.fheram_base2d(C.byref(p.c), lens, digits) == -1
    assert L.fheram_n_ggsw(C.byref(p.c)) == 0 and L.fheram_ggsw_len(C.byref(p.c)) == 0
    sk = np.zeros(4096, dtype=np.int64)
    out = np.zeros(16 * 196608, dtype=np.int64)
    xa, xe = fr.Source(1), fr.Source(2)
    assert L.fheram_encrypt_address(C.byref(p.c), 0, api._p(sk), xa.h, xe.h, api._p(out)) == -1
    assert xa.position() == 0 and xe.position() == 0
    with pytest.raises(fr.FheRamError) as e:
        p.module()
    assert e.value.code == -1, str(e.value)
    if n_decomp <= 8:
        with pytest.raises(fr.FheRamError) as e:
            fr.Ram.new_from_ram_params(1, decomp[:n_decomp], 1 << 13)
        assert e.value.code == -1, str(e.value)
