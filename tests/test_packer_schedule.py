"""CPU: the level schedule the GPU runs for a packer tree whose width m is not a power of two (fheram_cuda.cu:
packer_order, run_pack_tree, run_combine_mixed), restated with the oracle's arithmetic, equals GLWEPacker fed as
src/ram.rs:424-449 feeds it (bit-reversed order, None for the inputs h >= m).

With L = ceil(log2 m) and H = 2^(L-1): the inputs are kept in compact order (for each pair i < H, a_i = input
bitrev_{L-1}(i), then b_i = a_i + H when that is < m); levels 0 .. 11-L are one-sided for every input (one trace chain);
level 12-L combines a_i with b_i where b_i exists and takes the one-sided combine otherwise (the mixed level); the
levels above it are two-sided over width H."""
import numpy as np
import pytest

from oracle.oracle import Oracle


def rev(x, n):
    r = 0
    for i in range(n):
        r |= ((x >> i) & 1) << (n - 1 - i)
    return r


def packer_order(m):
    """(order, ops) as fheram_cuda.cu's packer_order builds them"""
    L = (m - 1).bit_length()
    if m & (m - 1) == 0:
        return [rev(p, L) for p in range(m)], []
    H = 1 << (L - 1)
    order, ops = [], []
    for i in range(H):
        h = rev(i, L - 1)
        two = h + H < m
        ops.append(len(order) << 1 | int(two))
        order.append(h)
        if two:
            order.append(h + H)
    return order, ops


@pytest.fixture(scope="module")
def orc():
    o = Oracle(backend="fft64", max_addr=1 << 13, word_size=1, k_pt=8)
    sk = o.secret_gen(o.source(0))
    keys = o.keys_prepare(*o.keygen(sk, o.source(1), o.source(2)))
    return o, keys


@pytest.mark.parametrize("m", [3, 5, 6, 7, 12, 48, 100, 4095])
def test_packer_order_covers_every_input_once(m):
    order, ops = packer_order(m)
    assert sorted(order) == list(range(m))
    L = (m - 1).bit_length()
    H = 1 << (L - 1)
    assert len(ops) == H and sum(op & 1 for op in ops) == m - H
    for i, op in enumerate(ops):
        assert order[op >> 1] == rev(i, L - 1)
        if op & 1:
            assert order[(op >> 1) + 1] == order[op >> 1] + H


@pytest.mark.parametrize("m", [3, 5, 6, 7, 12, 48, 100])
def test_mixed_schedule_equals_the_packer(orc, m):
    o, k = orc
    N, log_n = o.n, int(o.params.log_n)
    rng = np.random.default_rng(1000 + m)
    cts = rng.integers(-(1 << 16), 1 << 16, size=(m, o.glwe_len), dtype=np.int64)

    order, ops = packer_order(m)
    L = (m - 1).bit_length()
    H, one_sided = 1 << (L - 1), log_n - L
    # one trace chain over the m present inputs: levels 0 .. one_sided - 1 (run_trace_chain)
    buf = [o.trace(k, cts[h], 0, one_sided) for h in order]
    # the mixed level (run_combine_mixed): pair i reads a at ops[i] >> 1, b after it when ops[i] & 1
    level = one_sided
    buf = [o.packer_combine(k, level, buf[op >> 1], buf[(op >> 1) + 1] if op & 1 else None) for op in ops]
    assert len(buf) == H
    # the two-sided levels above it (run_pack_levels over width H)
    while len(buf) > 1:
        level += 1
        buf = [o.packer_combine(k, level, buf[2 * i], buf[2 * i + 1]) for i in range(len(buf) // 2)]
    assert level == log_n - 1

    feed = []
    for j in range(N):
        h = rev(j, log_n)
        feed.append(cts[h] if h < m else None)
    want = o.pack(k, feed)
    assert np.array_equal(buf[0], want), np.count_nonzero(buf[0] != want)


def test_one_sided_combine_is_a_trace_step(orc):
    """the one-sided path of the mixed kernels is their TRACE step with the level's key and no rotation"""
    o, k = orc
    rng = np.random.default_rng(7)
    a = rng.integers(-(1 << 16), 1 << 16, size=o.glwe_len, dtype=np.int64)
    for level in (0, 5, 11):
        assert np.array_equal(o.packer_combine(k, level, a, None), o.trace(k, a, level, level + 1))
