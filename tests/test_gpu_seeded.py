"""-m gpu: seeded ciphertexts on the device.  k_glwe_expand (behind fheram_address_load_seeded,
fheram_ram_read_batch_host_seeded and fheram_ram_load_seeded) must build, bit for bit, the limbs the CPU expansion
(fheram_address_expand / fheram_ram_expand) builds, and every operation with a seeded address must give the oracle's
limbs on the expanded address and decrypt correctly.  The multi-GPU case needs >= 2 GPUs."""
import ctypes as C
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


class World:
    """keys, RAM contents and the oracle for one parameter set"""

    def __init__(self, max_addr, word_size, k_pt):
        import fhe_ram_b200 as fr
        from oracle.oracle import Oracle
        self.fr = fr
        self.params = p = fr.Parameters.new(max_addr=max_addr, word_size=word_size, k_pt=k_pt)
        self.sk, self.evk = fr.gen_keys(p)
        self.keys = fr.EvaluationKeysPrepared.alloc(p).prepare(self.evk)
        self.data = fr.Source(5).fill_bytes(max_addr * word_size)
        self.bodies, self.seed = self.seeded_ram()
        self.cts = fr.Ram.expand(p, self.bodies, self.seed)
        self.orc = Oracle(backend="fft64", max_addr=max_addr, word_size=word_size, k_pt=k_pt)
        self.okeys = self.orc.keys_prepare(self.evk.atk_glwe, self.evk.gglwe_to_ggsw_key, self.evk.atk_ggsw_inv)

    def seeded_ram(self):
        from fhe_ram_b200 import api
        p = self.params
        bodies = np.zeros(p.word_size() * p.n_glwe() * p.glwe_len() // 2, dtype=np.int64)
        seed = np.zeros(1, dtype=api.SEED_DTYPE)
        xa = self.fr.Source(11)
        xa.next_u32()  # the RAM's mask stream does not start at a block boundary
        api._check(api.lib().fheram_encrypt_ram_seeded(C.byref(p.c), self.data.ctypes.data_as(api._PU8),
                                                       api._p(self.sk.data), xa.h, self.fr.Source(12).h,
                                                       api._p(bodies), api._ps(seed, 1)))
        return bodies, seed

    def addresses(self, idxs, skew=0):
        """seeded addresses from one Source pair in turn: (bodies [n][...], seeds [n])"""
        xa, xe = self.fr.Source(21), self.fr.Source(22)
        for _ in range(skew):
            xa.next_u32()
        out = [self.fr.Address.encrypt_sk_seeded(self.params, int(i), self.sk, xa, xe) for i in idxs]
        return np.stack([b for b, _ in out]), np.concatenate([s for _, s in out])

    def check_decrypt(self, got, idx, data=None):
        data = self.data if data is None else data
        p = self.params
        for i in range(p.word_size()):
            w = self.fr.cast_u8_to_signed(int(data[i + p.word_size() * idx]), min(8, p.k_glwe_pt()))
            v, noise = self.fr.decrypt_glwe(p, got[i], w, self.sk)
            assert v == w and noise < -(p.k_glwe_pt() + 1), (idx, i, v, w, noise)


_worlds = {}


@pytest.fixture(scope="module")
def world(built):
    def get(max_addr, word_size, k_pt=8):
        key = (max_addr, word_size, k_pt)
        if key not in _worlds:
            _worlds[key] = World(*key)
        return _worlds[key]
    return get


@pytest.mark.parametrize("max_addr,word_size,k_pt", [(1 << 13, 2, 8), (1 << 18, 4, 9)])
@pytest.mark.parametrize("n,skew", [(1, 0), (5, 3)])
def test_device_address_expansion_equals_cpu(world, max_addr, word_size, k_pt, n, skew):
    w = world(max_addr, word_size, k_pt)
    fr, p = w.fr, w.params
    bodies, seeds = w.addresses([(7919 * i + 3) % max_addr for i in range(n)], skew)
    got = fr.Address.load_seeded(p, bodies, seeds, n)
    want = fr.Address.expand(p, bodies, seeds, n)
    assert np.array_equal(got.download_raw(), want.data)
    got.close()


@pytest.mark.parametrize("max_addr,word_size,k_pt", [(1 << 13, 2, 8), (1 << 18, 4, 9)])
def test_device_ram_expansion_equals_cpu(world, max_addr, word_size, k_pt):
    w = world(max_addr, word_size, k_pt)
    ram = w.fr.Ram.new(w.params)
    ram.load_seeded(w.bodies, w.seed)
    assert np.array_equal(ram.store(), w.cts)
    ram.close()


@pytest.mark.parametrize("max_addr,word_size", [(1 << 13, 2), (3 * 4096, 2)])
def test_read_rpw_write_with_seeded_addresses_match_the_oracle(world, max_addr, word_size):
    w = world(max_addr, word_size)
    fr, p, keys = w.fr, w.params, w.keys
    ram = fr.Ram.new(p)
    ram.load_seeded(w.bodies, w.seed)
    oram = w.orc.ram_new(w.cts.copy())
    idxs = [0, max_addr - 1, 4097 % max_addr]
    bodies, seeds = w.addresses(idxs)
    data = w.data.copy()
    for j, idx in enumerate(idxs):
        dev = fr.Address.load_seeded(p, bodies[j], seeds[j:j + 1])
        full = fr.Address.expand(p, bodies[j], seeds[j:j + 1]).data
        got = ram.read(dev, keys)
        rc, want = w.orc.ram_read(oram, full, w.okeys)
        assert rc == 0 and np.array_equal(got, want), "read"
        w.check_decrypt(got, idx, data)
        got = ram.read_prepare_write(dev, keys)
        rc, want = w.orc.ram_read_prepare_write(oram, full, w.okeys)
        assert rc == 0 and np.array_equal(got, want), "read_prepare_write"
        w.check_decrypt(got, idx, data)
        assert np.array_equal(ram.store(), w.orc.ram_store(oram)), "read_prepare_write: RAM limbs"
        assert np.array_equal(ram.tree_store(), w.orc.ram_tree_store(oram)), "read_prepare_write: tree limbs"
        value = fr.Source(40 + j).fill_bytes(word_size)
        wd = np.stack([fr.encrypt_glwe(p, int(v), w.sk) for v in value])
        ram.write(wd, dev, keys)
        assert w.orc.ram_write(oram, wd.reshape(-1), full, w.okeys) == 0
        assert np.array_equal(ram.store(), w.orc.ram_store(oram)), "write: RAM limbs"
        data[idx * word_size:(idx + 1) * word_size] = value
        got = ram.read(dev, keys)
        rc, want = w.orc.ram_read(oram, full, w.okeys)
        assert rc == 0 and np.array_equal(got, want), "read after write"
        w.check_decrypt(got, idx, data)
        dev.close()
    ram.close()


@pytest.mark.parametrize("max_addr,word_size", [(1 << 13, 2), (3 * 4096, 2)])
def test_read_batch_host_seeded_equals_read_batch(world, monkeypatch, max_addr, word_size):
    monkeypatch.setenv("FHERAM_CHUNK", "3")  # several chunks, the last one short
    w = world(max_addr, word_size)
    fr, p, keys = w.fr, w.params, w.keys
    n = 7
    idxs = [(104729 * i + 11) % max_addr for i in range(n)]
    bodies, seeds = w.addresses(idxs, skew=1)
    ram = fr.Ram.new(p)
    ram.load_seeded(w.bodies, w.seed)
    want = ram.read_batch(fr.Address.expand(p, bodies, seeds, n), keys)
    got = ram.read_batch_host_seeded(fr.api.pack17(bodies), seeds, n, keys)
    assert np.array_equal(got.astype(np.int64), want)
    for q, idx in enumerate(idxs):
        w.check_decrypt(want[q], idx)
    ram.close()


@pytest.mark.parametrize("n_shards", [1, 2, 4])
def test_ram_load_seeded_equals_ram_load(world, n_shards):
    w = world(1 << 15, 2)
    fr, p = w.fr, w.params
    for shard in range(n_shards):
        a, b = fr.Ram(p, shard, n_shards), fr.Ram(p, shard, n_shards)
        a.load_seeded(w.bodies, w.seed)
        b.load(w.cts)
        got, want = a.store(), b.store()
        assert np.array_equal(got, want)
        own = got.reshape(p.word_size(), p.n_glwe(), -1)[:, shard::n_shards]
        assert np.array_equal(own, w.cts.reshape(p.word_size(), p.n_glwe(), -1)[:, shard::n_shards])
        a.close(); b.close()


def test_ram_load_seeded_leaves_a_loaded_ram_ready_to_read(world):
    w = world(1 << 13, 2)
    fr, p, keys = w.fr, w.params, w.keys
    bodies, seeds = w.addresses([5])
    a = fr.Address.load_seeded(p, bodies[0], seeds)
    ram = fr.Ram.new(p)
    with pytest.raises(fr.FheRamError):  # never loaded
        ram.read(a, keys)
    ram.load_seeded(w.bodies, w.seed)
    ram.read_prepare_write(a, keys)
    assert ram.state()
    ram.load_seeded(w.bodies, w.seed)  # clears the prepared-for-write state, as fheram_ram_load does
    assert not ram.state()
    w.check_decrypt(ram.read(a, keys), 5)
    a.close(); ram.close()


def test_bad_arguments_are_refused(world):
    from fhe_ram_b200 import api
    w = world(1 << 13, 2)
    fr, p, keys = w.fr, w.params, w.keys
    L = api.lib()
    bodies, seeds = w.addresses([1, 2])
    b = np.ascontiguousarray(bodies.reshape(-1))
    packed = api.pack17(b)
    ps = api._ps(seeds, 2)
    h = C.c_void_p()
    assert L.fheram_address_load_seeded(p.module(), api._p(b), ps, 0, C.byref(h)) == -1
    assert L.fheram_address_load_seeded(p.module(), None, ps, 2, C.byref(h)) == -1
    assert L.fheram_address_load_seeded(p.module(), api._p(b), None, 2, C.byref(h)) == -1
    assert L.fheram_address_load_seeded(None, api._p(b), ps, 2, C.byref(h)) == -1
    ram = fr.Ram.new(p)
    ram.load_seeded(w.bodies, w.seed)
    out = np.zeros((2, p.word_size(), p.glwe_len()), dtype=np.int32)
    po = out.reshape(-1).ctypes.data_as(C.POINTER(C.c_int32))
    pp = packed.ctypes.data_as(C.POINTER(C.c_uint32))
    assert L.fheram_ram_read_batch_host_seeded(ram.h, pp, ps, 0, keys.h, po) == -1
    assert L.fheram_ram_read_batch_host_seeded(ram.h, pp, None, 2, keys.h, po) == -1
    assert L.fheram_ram_read_batch_host_seeded(ram.h, None, ps, 2, keys.h, po) == -1
    assert L.fheram_ram_read_batch_host_seeded(ram.h, pp, ps, 2, None, po) == -1
    assert L.fheram_ram_load_seeded(ram.h, None, api._ps(w.seed, 1)) == -1
    assert L.fheram_ram_load_seeded(ram.h, api._p(w.bodies), None) == -1
    assert L.fheram_ram_load_seeded(None, api._p(w.bodies), api._ps(w.seed, 1)) == -1
    # keys of another context
    p2 = fr.Parameters.new(max_addr=1 << 13, word_size=2, k_pt=8)
    keys2 = fr.EvaluationKeysPrepared.alloc(p2).prepare(w.evk)
    assert L.fheram_ram_read_batch_host_seeded(ram.h, pp, ps, 2, keys2.h, po) == -1
    assert "different contexts" in L.fheram_last_error().decode()
    # int64 bodies outside the device range
    big = b.copy()
    big[5] = 1 << 40
    assert L.fheram_address_load_seeded(p.module(), api._p(big), ps, 2, C.byref(h)) == -6  # FHERAM_ERR_RANGE
    # the RAM still reads correctly after the refusals
    got = ram.read_batch_host_seeded(packed, seeds, 2, keys)
    want = ram.read_batch(fr.Address.expand(p, bodies, seeds, 2), keys)
    assert np.array_equal(got.astype(np.int64), want)
    keys2.close(); p2.close(); ram.close()


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, str(ROOT))
    import torch
    import torch.distributed as dist
    import fhe_ram_b200 as fr
    from fhe_ram_b200 import api
    from fhe_ram_b200.sharded import ShardedRamLib
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    ws = 2
    p = fr.Parameters.new(device=rank, max_addr=1 << 15, word_size=ws, k_pt=8)
    sk, evk = fr.gen_keys(p)
    keys = fr.EvaluationKeysPrepared.alloc(p).prepare(evk)
    data = fr.Source(5).fill_bytes(p.max_addr() * ws)
    ref = fr.Ram.new(p)                                    # one GPU's RAM
    bodies_ram, seed_ram = ref.encrypt_sk_seeded(data, sk, fr.Source(11), fr.Source(12))
    B = 3 * world                                          # three reads per rank
    idxs = [(9973 * i + 1) % (1 << 15) for i in range(B)]
    xa, xe = fr.Source(21), fr.Source(22)
    enc = [fr.Address.encrypt_sk_seeded(p, i, sk, xa, xe) for i in idxs]
    bodies = np.stack([b for b, _ in enc])
    seeds = np.concatenate([s for _, s in enc])
    want = ref.read_batch(fr.Address.expand(p, bodies, seeds, B), keys)
    lo, hi = rank * (B // world), (rank + 1) * (B // world)
    fails = []
    lib = ShardedRamLib(p, rank, world)
    lib.ram.load_seeded(bodies_ram, seed_ram)              # each rank expands its own polynomials
    mine = lib.store().reshape(ws, p.n_glwe(), -1)
    full = ref.store().reshape(ws, p.n_glwe(), -1)
    if not np.array_equal(mine[:, rank::world], full[:, rank::world]):
        fails.append("ram_load_seeded: own polynomials")
    got = lib.read_batch_host_seeded(api.pack17(bodies[lo:hi]), seeds[lo:hi], hi - lo, keys)
    if not np.array_equal(got.astype(np.int64), want[lo:hi]):
        fails.append("read_batch_host_seeded")
    lib.close()
    Path(f"{out_dir}/r{rank}.txt").write_text("\n".join(fails))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world_size", [2, 4, 8])
def test_seeded_batch_over_nccl_equals_one_gpu(built, tmp_path, world_size):
    import torch
    import torch.multiprocessing as mp
    n = torch.cuda.device_count()
    if n < world_size:
        pytest.skip(f"needs >= {world_size} GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_worker, args=(world_size, port, str(tmp_path)), nprocs=world_size, join=True)
    for r in range(world_size):
        fails = (tmp_path / f"r{r}.txt").read_text()
        assert fails == "", f"rank {r}: {fails}"
