"""-m gpu: the whole read / read_prepare_write / write path at address decompositions other than the default, limb for
limb against the CPU oracle at the same decomposition.

decomp_n (Parameters.new(decomp_n=...), Ram::new_from_ram_params) sets the Base2D coordinates, hence the length of
every external-product chain (the first-coordinate chain of a read, the second-coordinate chain, both inverse chains
of a write), the monomials of the device address encryption and of the seeded address layout, and the split of the
host pipeline's prepared GGSWs between the two coordinates.  The sets below reach one-step chains, a single uneven
coordinate, a mixed packer level, chains of 6 and 8 steps, a two-step second coordinate and the default table at 2^21;
tests/test_decomposition_client.py checks the same sets on the client side."""
import ctypes as C
import os
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent

# (decomp_n, max_addr, word_size, Base2D coordinates)
SETS = [
    ([12], 1 << 13, 2, [[12], [1]]),                             # one-step chains, 12-bit monomials
    ([5, 7], 1 << 12, 1, [[5, 7]]),                              # one coordinate, uneven digits
    ([4, 4, 4], 5 * 4096 + 17, 1, [[4, 4, 4], [3]]),             # 3-step chain, mixed packer level (G = 6)
    ([2] * 6, 1 << 14, 2, [[2] * 6, [2]]),                       # 6-step chain
    ([1, 11], 1 << 15, 1, [[1, 11], [1, 2]]),                    # 2-step second coordinate
    ([1] * 7 + [5], 1 << 20, 1, [[1] * 7 + [5], [1] * 8]),       # 8-step chains, 16 GGSWs
    ([3, 3, 3, 3], 1 << 21, 1, [[3, 3, 3, 3], [3, 3, 3]]),       # the default table, odd 3-step second coordinate
]


def _id(decomp, max_addr):
    return ("small_" if max_addr <= 1 << 15 else "large_") + "-".join(map(str, decomp))


CASES = [pytest.param(*s, id=_id(s[0], s[1])) for s in SETS]


class Setup:
    """keys, RAM and oracle of one decomposition, client side as conftest.Scenario builds them"""

    def __init__(self, decomp, max_addr, word_size):
        import fhe_ram_b200 as fr
        from fhe_ram_b200 import api
        from oracle.oracle import Oracle, host_threads
        self.fr = fr
        self.params = p = fr.Parameters.new(max_addr=max_addr, word_size=word_size, k_pt=8, decomp_n=decomp)
        self.sk, self.evk = fr.gen_keys(p)
        self.keys = fr.EvaluationKeysPrepared.alloc(p).prepare(self.evk)
        self.src = fr.Source(5)
        self.data = self.src.fill_bytes(max_addr * word_size)
        self.cts = np.zeros(word_size * p.n_glwe() * p.glwe_len(), dtype=np.int64)
        api._check(api.lib().fheram_encrypt_ram(C.byref(p.c), self.data.ctypes.data_as(api._PU8), api._p(self.sk.data),
                                                fr.Source(11).h, fr.Source(12).h, api._p(self.cts)))
        self.orc = Oracle(backend="fft64", max_addr=max_addr, word_size=word_size, k_pt=8, decomp_n=decomp)
        self.threads = min(8, host_threads())
        self.orc.set_ram_threads(self.threads)  # sub-RAMs on several threads: same limbs, shorter test
        self.okeys = self.orc.keys_prepare(self.evk.atk_glwe, self.evk.gglwe_to_ggsw_key, self.evk.atk_ggsw_inv)
        self.xa, self.xe = fr.Source(21), fr.Source(22)

    def address(self, idx):
        return self.fr.Address.alloc(self.params).encrypt_sk(self.params, idx, self.sk, self.xa, self.xe)

    def check_decrypt(self, cts, idx, data=None):
        data = self.data if data is None else data
        p = self.params
        for i in range(p.word_size()):
            w = self.fr.cast_u8_to_signed(int(data[i + p.word_size() * idx]), min(8, p.k_glwe_pt()))
            v, noise = self.fr.decrypt_glwe(p, cts[i], w, self.sk)
            assert v == w and noise < -(p.k_glwe_pt() + 1), (idx, i, v, w, noise)


_setups = {}


@pytest.fixture(scope="module")
def setup(built):
    def get(decomp, max_addr, word_size, coords):
        key = (tuple(decomp), max_addr, word_size)
        if key not in _setups:
            _setups[key] = Setup(decomp, max_addr, word_size)
        s = _setups[key]
        assert s.params.base2d() == coords
        return s
    return get


def _batch_idxs(max_addr):
    return sorted({0, max_addr - 1, (max_addr * 3) // 5, (max_addr * 5) // 7 + 1, 4097 % max_addr})


@pytest.mark.parametrize("decomp,max_addr,word_size,coords", CASES)
def test_read_rpw_write_match_the_oracle(setup, decomp, max_addr, word_size, coords):
    s = setup(decomp, max_addr, word_size, coords)
    fr, p, keys = s.fr, s.params, s.keys
    ram = fr.Ram.new(p)
    ram.load(s.cts)
    oram = s.orc.ram_new(s.cts.copy())
    idx = (max_addr * 5) // 7
    addr = s.address(idx)
    two = len(coords) > 1

    got = ram.read(addr, keys)
    rc, want = s.orc.ram_read(oram, addr.data, s.okeys)
    assert rc == 0 and np.array_equal(got, want), ("read", np.count_nonzero(got != want))
    s.check_decrypt(got, idx)

    got = ram.read_prepare_write(addr, keys)
    rc, want = s.orc.ram_read_prepare_write(oram, addr.data, s.okeys)
    assert rc == 0 and np.array_equal(got, want), ("read_prepare_write", np.count_nonzero(got != want))
    s.check_decrypt(got, idx)
    assert np.array_equal(ram.store(), s.orc.ram_store(oram)), "read_prepare_write: RAM limbs"
    if two:
        assert np.array_equal(ram.tree_store(), s.orc.ram_tree_store(oram)), "read_prepare_write: tree limbs"

    value = fr.Source(40).fill_bytes(word_size)
    w = np.stack([fr.encrypt_glwe(p, int(v), s.sk) for v in value])
    ram.write(w, addr, keys)
    assert s.orc.ram_write(oram, w.reshape(-1), addr.data, s.okeys) == 0
    store = ram.store()
    assert np.array_equal(store, s.orc.ram_store(oram)), ("write: RAM limbs", np.count_nonzero(store != s.orc.ram_store(oram)))
    if two:
        assert np.array_equal(ram.tree_store(), s.orc.ram_tree_store(oram)), "write: tree limbs"

    data2 = s.data.copy()
    data2[idx * word_size:(idx + 1) * word_size] = value
    got = ram.read(addr, keys)
    rc, want = s.orc.ram_read(oram, addr.data, s.okeys)
    assert rc == 0 and np.array_equal(got, want), "read after write"
    s.check_decrypt(got, idx, data2)
    for other in ((idx + 1) % max_addr, (idx + p.n() + 3) % max_addr):  # a neighbour and another polynomial
        a = s.address(other)
        got = ram.read(a, keys)
        rc, want = s.orc.ram_read(oram, a.data, s.okeys)
        assert rc == 0 and np.array_equal(got, want), ("read of an untouched word", other)
        s.check_decrypt(got, other, data2)
    ram.close()


@pytest.mark.parametrize("decomp,max_addr,word_size,coords", CASES)
def test_batched_reads_match_the_oracle(setup, monkeypatch, decomp, max_addr, word_size, coords):
    """read_batch, the host pipeline in its three input formats (several chunks, the last one short), and addresses
    encrypted on the device"""
    monkeypatch.setenv("FHERAM_CHUNK", "3")
    s = setup(decomp, max_addr, word_size, coords)
    fr, p, keys = s.fr, s.params, s.keys
    from fhe_ram_b200 import api
    ram = fr.Ram.new(p)
    ram.load(s.cts)
    oram = s.orc.ram_new(s.cts.copy())
    idxs = _batch_idxs(max_addr)
    xa, xe = fr.Source(31), fr.Source(32)
    addrs = [fr.Address.alloc(p).encrypt_sk(p, i, s.sk, xa, xe) for i in idxs]
    limbs = np.stack([a.data for a in addrs])
    rc, want = s.orc.ram_read_many(oram, limbs.reshape(-1), len(idxs), s.okeys, s.threads)
    assert rc == 0
    got = ram.read_batch(fr.Address.batch(p, addrs), keys)
    for b, i in enumerate(idxs):
        assert np.array_equal(got[b], want[b]), ("read_batch", i, np.count_nonzero(got[b] != want[b]))
        s.check_decrypt(got[b], i)
    assert np.array_equal(ram.read_batch_host(limbs, len(idxs), keys), want), "read_batch_host"
    got17 = ram.read_batch_host_p17(api.pack17(limbs), len(idxs), keys)
    assert np.array_equal(got17.astype(np.int64), want), "read_batch_host_p17"

    # the same addresses encrypted on the device from the same Sources: the same limbs
    dev = fr.Address.encrypt_sk_gpu(p, idxs, s.sk, fr.Source(31), fr.Source(32))
    assert np.array_equal(dev.download_raw(), limbs.reshape(-1)), "device address encryption"
    assert np.array_equal(ram.read_batch(dev, keys), want)
    dev.close()

    # seeded addresses through the host pipeline, against the oracle on their CPU expansion
    sx, se = fr.Source(33), fr.Source(34)
    seeded = [fr.Address.encrypt_sk_seeded(p, i, s.sk, sx, se) for i in idxs]
    bodies = np.stack([b for b, _ in seeded])
    seeds = np.concatenate([x for _, x in seeded])
    full = fr.Address.expand(p, bodies, seeds, len(idxs)).data
    rc, want_s = s.orc.ram_read_many(oram, full, len(idxs), s.okeys, s.threads)
    assert rc == 0
    got_s = ram.read_batch_host_seeded(api.pack17(bodies), seeds, len(idxs), keys)
    for b, i in enumerate(idxs):
        assert np.array_equal(got_s[b].astype(np.int64), want_s[b]), ("read_batch_host_seeded", i)
        s.check_decrypt(want_s[b], i)
    ram.close()


@pytest.mark.parametrize("n_shards", [2, 4])
def test_sharded_stages_on_one_gpu(setup, n_shards):
    """decomp_n [2]*6 at 2^14 x 2 through the sharded stages with every shard on one GPU (as
    test_gpu_parity.py::test_sharded_stages_on_one_gpu): must equal the unsharded read / read_prepare_write / write"""
    import torch
    from fhe_ram_b200 import api
    s = setup([2] * 6, 1 << 14, 2, [[2] * 6, [2]])
    fr, p, keys = s.fr, s.params, s.keys
    L = p.word_size() * p.glwe_len()
    idxs = [5, 4096 + 9, 3 * 4096 + 2741, (1 << 14) - 1]
    addrs = [s.address(i) for i in idxs]
    batch = fr.Address.batch(p, addrs)
    ref = fr.Ram.new(p)
    ref.load(s.cts)
    want = ref.read_batch(batch, keys)
    shards = [fr.Ram(p, shard=g, n_shards=n_shards) for g in range(n_shards)]
    for r in shards:
        r.load(s.cts)

    def gather(fn, n):
        parts = []
        for r in shards:
            d = C.c_void_p()
            api._check(fn(r, C.byref(d)))
            host = np.zeros(n * p.word_size() * p.glwe_len(), dtype=np.int64)
            api._check(api.lib().fheram_download_glwe(p.module(), d, n * p.word_size(), api._p(host)))
            parts.append(host)
        return torch.from_numpy(np.concatenate(parts).astype(np.int32)).cuda()  # what the exchange produces

    g = gather(lambda r, d: api.lib().fheram_ram_read_local_device(r.h, batch.device(), keys.h, d), batch.count)
    for r in shards:
        d = C.c_void_p()
        api._check(api.lib().fheram_ram_read_finish_device(r.h, C.c_void_p(g.data_ptr()), batch.count, 0,
                                                           batch.count, batch.device(), 0, keys.h, C.byref(d)))
        got = np.zeros(batch.count * L, dtype=np.int64)
        api._check(api.lib().fheram_download_glwe(p.module(), d, batch.count * p.word_size(), api._p(got)))
        assert np.array_equal(got.reshape(want.shape), want)

    a = addrs[2]
    want_rpw = ref.read_prepare_write(a, keys)
    g = gather(lambda r, d: api.lib().fheram_ram_rpw_local_device(r.h, a.device(), keys.h, d), 1)
    for r in shards:
        d = C.c_void_p()
        api._check(api.lib().fheram_ram_rpw_finish_device(r.h, C.c_void_p(g.data_ptr()), a.device(), keys.h, C.byref(d)))
        got = np.zeros(L, dtype=np.int64)
        api._check(api.lib().fheram_download_glwe(p.module(), d, p.word_size(), api._p(got)))
        assert np.array_equal(got.reshape(want_rpw.shape), want_rpw)
    w = np.stack([fr.encrypt_glwe(p, 33 + i, s.sk) for i in range(p.word_size())])
    ref.write(w, a, keys)
    full = ref.store().reshape(p.word_size(), p.n_glwe(), -1)
    for gi, r in enumerate(shards):
        r.write(w, a, keys)
        mine = r.store().reshape(p.word_size(), p.n_glwe(), -1)
        for h in range(gi, p.n_glwe(), n_shards):
            assert np.array_equal(mine[:, h], full[:, h]), (gi, h)
        assert np.array_equal(r.tree_store(), ref.tree_store())
        r.close()
    ref.close()


@pytest.mark.parametrize("name", ["ext8", "ext9", "ext9c4"])
def test_small_sets_under_each_external_product_kernel(built, name):
    """the small sets' reads, writes and batches with each external-product kernel forced by FHERAM_KERNEL (the default
    rule gives these narrow launches to k_ext9<8> only)"""
    env = dict(os.environ)
    env["FHERAM_KERNEL"] = name
    r = subprocess.run([sys.executable, "-m", "pytest", str(Path(__file__)), "-m", "gpu", "-x", "-q", "-k",
                        "(read_rpw_write_match or batched_reads_match) and small"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"FHERAM_KERNEL={name}:\n{r.stdout[-3000:]}\n{r.stderr[-1000:]}"
    assert re.search(r"\b10 passed\b", r.stdout), r.stdout[-500:]
