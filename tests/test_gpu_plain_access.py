"""-m gpu: reads and writes at plaintext addresses (include/fheram.h, DESIGN.md 3.8), limb for limb against the
oracle's restatement of the definitions (the restatement itself is checked in test_plain_access_oracle.py):

  read_plain:  out[b][s] = TRACE(rot(2N - j_b, data[s][h_b]))                     for a_b = h_b N + j_b
  write_plain: data[s][h] <- normalize(data[s][h] - rot(j, T_s) + rot(j, w_s)),   T_s = TRACE(rot(2N - j, data[s][h]))

The trace launch runs over n x word_size items, so the widths below reach every trace kernel the launch-width rule
picks (DESIGN.md 3.4); test_kernel_forced_plain repeats them with each key-switch kernel forced."""
import ctypes as C
import os
import re
import socket
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent

# (max_addr, word_size, k_pt): the default, G = 3 polynomials, one coordinate, the README set
SIZES = [(1 << 13, 2, 8), (3 * 4096, 2, 8), (3000, 2, 8), (1 << 18, 4, 9)]
# n * word_size at word_size 2: k_ks8<8>, k_ks8<4>, k_ks6, k_ks5, k_ks7 on a 148-SM B200
WIDTHS = [2, 6, 32, 74, 100, 200]


def _polys(s, cts):
    return cts.reshape(s.params.word_size(), s.params.n_glwe(), s.params.glwe_len())


def plain_read(s, cts, a):
    N = s.params.n()
    h, j = a // N, a % N
    P = _polys(s, cts)
    return np.stack([s.orc.trace(s.okeys, s.orc.glwe_rotate(2 * N - j, P[w, h])) for w in range(s.params.word_size())])


def plain_write(s, cts, a, w):
    N = s.params.n()
    h, j = a // N, a % N
    out = _polys(s, cts).copy()
    T = plain_read(s, cts, a)
    for i in range(s.params.word_size()):
        out[i, h] = s.orc.glwe_normalize(out[i, h] - s.orc.glwe_rotate(j, T[i]) + s.orc.glwe_rotate(j, w[i]))
    return out.reshape(-1)


def _ram(s, cts=None, shard=0, n_shards=1):
    r = s.fr.Ram(s.params, shard, n_shards)
    r.load(s.cts if cts is None else cts)
    return r


def _words(s, values):
    return np.stack([s.fr.encrypt_glwe(s.params, int(v), s.sk) for v in values])


def _download(s, ptr, n_glwe):
    from fhe_ram_b200 import api
    out = np.zeros((n_glwe, s.params.glwe_len()), dtype=np.int64)
    api._check(api.lib().fheram_download_glwe(s.params.module(), C.c_void_p(ptr), n_glwe, api._p(out.reshape(-1))))
    return out


def _addresses(max_addr, n_random, seed):
    N = 4096
    fixed = [a for a in (0, 1, N - 1, N, max_addr - 1) if a < max_addr]
    rng = np.random.default_rng(seed)
    rand = [int(x) for x in rng.integers(0, max_addr, size=n_random)]
    return fixed + rand + [fixed[-1], rand[0] if rand else 0]  # duplicates


@pytest.mark.parametrize("size", SIZES, ids=lambda t: f"{t[0]}x{t[1]}")
def test_read_plain_matches_the_definition(scenario, gpu_keys, size):
    s = scenario(*size)
    keys = gpu_keys(s)
    ram = _ram(s)
    addrs = _addresses(s.params.max_addr(), 3, 7)
    got = ram.read_plain(addrs, keys)
    for b, a in enumerate(addrs):
        assert np.array_equal(got[b], plain_read(s, s.cts, a)), (size, a)
        s.check_decrypt(got[b], a)
    # the device arena holds the same limbs, and decrypts on the device to the data
    ptr = ram.read_plain_device(addrs, keys)
    ws = s.params.word_size()
    assert np.array_equal(_download(s, ptr, len(addrs) * ws), got.reshape(-1, s.params.glwe_len()))
    values, _ = s.fr.decrypt_words_device(s.params, ptr, len(addrs) * ws, s.sk)
    want = [s.want(a, i) for a in addrs for i in range(ws)]
    assert values.tolist() == want
    ram.close()


def _sample(n):
    return sorted({0, n // 2, n - 1})


@pytest.mark.parametrize("width", WIDTHS)
def test_read_plain_at_every_trace_width(scenario, gpu_keys, width):
    s = scenario()
    keys = gpu_keys(s)
    ram = _ram(s)
    ws = s.params.word_size()
    n = width // ws
    addrs = [int(a) for a in np.random.default_rng(width).integers(0, s.params.max_addr(), size=n)]
    got = ram.read_plain(addrs, keys)
    for b in _sample(n):
        assert np.array_equal(got[b], plain_read(s, s.cts, addrs[b])), (width, b)
    ptr = ram.read_plain_device(addrs, keys)
    assert np.array_equal(_download(s, ptr, n * ws), got.reshape(-1, s.params.glwe_len()))
    values, _ = s.fr.decrypt_words_device(s.params, ptr, n * ws, s.sk)
    assert values.tolist() == [s.want(a, i) for a in addrs for i in range(ws)]
    ram.close()


@pytest.mark.parametrize("size", SIZES, ids=lambda t: f"{t[0]}x{t[1]}")
def test_write_plain_matches_the_definition(scenario, gpu_keys, size):
    s = scenario(*size)
    keys = gpu_keys(s)
    ram = _ram(s)
    tree0 = ram.tree_store()
    a = min(4096 + 5, s.params.max_addr() - 1)
    # below 128: encrypt_glwe encodes a byte as unsigned at k_pt = 9, a stored byte reads back signed
    new = [(37 * i + 90) % 128 for i in range(s.params.word_size())]
    w = _words(s, new)
    ram.write_plain(a, w, keys)
    want = plain_write(s, s.cts, a, w)
    assert np.array_equal(ram.store(), want)
    assert np.array_equal(ram.tree_store(), tree0) and not ram.state()
    values, _ = ram.decrypt_sk(s.sk)
    data = s.data.reshape(-1, s.params.word_size()).copy()
    data[a] = new
    k = min(8, s.params.k_glwe_pt())
    table = np.array([s.fr.cast_u8_to_signed(b, k) for b in range(256)], dtype=np.int16)
    assert np.array_equal(values, table[data])
    ram.close()


def test_write_plain_then_oblivious_read(scenario, gpu_keys):
    s = scenario()
    keys = gpu_keys(s)
    ram = _ram(s)
    a = 4096 + 300
    new = [5, 250]
    w = _words(s, new)
    ram.write_plain(a, w, keys)
    want_cts = plain_write(s, s.cts, a, w)
    addr = s.address(a)
    got = ram.read(addr, keys)
    oram = s.orc.ram_new(want_cts.copy())
    rc, want = s.orc.ram_read(oram, addr.data, s.okeys)
    assert rc == 0 and np.array_equal(got, want)
    data = s.data.copy()
    data[a * 2:a * 2 + 2] = new
    s.check_decrypt(got, a, data)
    s.orc.lib.orc_ram_free(oram)
    ram.close()


def test_oblivious_write_then_read_plain(scenario, gpu_keys):
    s = scenario()
    keys = gpu_keys(s)
    ram = _ram(s)
    a = 77
    addr = s.address(a)
    oram = s.orc.ram_new(s.cts.copy())
    ram.read_prepare_write(addr, keys)
    assert s.orc.ram_read_prepare_write(oram, addr.data, s.okeys)[0] == 0
    new = [11, 222]
    w = _words(s, new)
    ram.write(w, addr, keys)
    assert s.orc.ram_write(oram, w.reshape(-1), addr.data, s.okeys) == 0
    after = s.orc.ram_store(oram)
    assert np.array_equal(ram.store(), after)
    got = ram.read_plain([a, a + 1], keys)
    assert np.array_equal(got[0], plain_read(s, after, a)) and np.array_equal(got[1], plain_read(s, after, a + 1))
    data = s.data.copy()
    data[a * 2:a * 2 + 2] = new
    s.check_decrypt(got[0], a, data)
    s.orc.lib.orc_ram_free(oram)
    ram.close()


def test_write_plain_twice_to_one_polynomial(scenario, gpu_keys):
    s = scenario()
    keys = gpu_keys(s)
    ram = _ram(s)
    want = s.cts
    data = s.data.copy()
    for a, new in ((4096 + 9, [1, 2]), (4096 + 4000, [130, 255])):
        w = _words(s, new)
        ram.write_plain(a, w, keys)
        want = plain_write(s, want, a, w)
        data[a * 2:a * 2 + 2] = new
    assert np.array_equal(ram.store(), want)
    for a in (4096 + 9, 4096 + 4000, 4096 + 10):
        s.check_decrypt(ram.read_plain([a], keys)[0], a, data)
    ram.close()


def test_extreme_digits(scenario, gpu_keys):
    """polynomial h = 1 with every limb -2^16: rot(2N - j, .) negates the wrapped limbs to +2^16, outside the balanced
    range, and the kernels must treat them as values"""
    s = scenario()
    keys = gpu_keys(s)
    cts = s.cts.copy()
    P = _polys(s, cts)
    P[:, 1] = -(1 << 16)
    ram = _ram(s, cts)
    a = 4096 + 1234
    got = ram.read_plain([a], keys)
    assert np.array_equal(got[0], plain_read(s, cts, a))
    w = _words(s, [3, 4])
    ram.write_plain(a, w, keys)
    assert np.array_equal(ram.store(), plain_write(s, cts, a, w))
    ram.close()


def test_refusals(scenario, gpu_keys):
    from fhe_ram_b200 import api
    s = scenario()
    fr, p = s.fr, s.params
    keys = gpu_keys(s)
    lib = api.lib()
    ram = _ram(s)
    w = _words(s, [1, 2])
    out = np.zeros((1, p.word_size(), p.glwe_len()), dtype=np.int64)
    d = C.c_void_p()
    a0 = (C.c_uint32 * 1)(0)
    bad = (C.c_uint32 * 2)(0, p.max_addr())
    other = fr.Parameters.new(max_addr=p.max_addr(), word_size=p.word_size(), k_pt=8)
    other_keys = fr.EvaluationKeysPrepared.alloc(other).prepare(s.evk)
    fresh = fr.Ram(p)                                             # never loaded
    stated = _ram(s)
    stated.read_prepare_write(s.address(3), keys)                 # prepared for write
    rotated = _ram(s)
    api._check(lib.fheram_ram_rpw_local_device(rotated.h, s.address(3).device(), keys.h, C.byref(d)))
    calls = [
        (-1, lambda: lib.fheram_ram_read_plain(ram.h, bad, 2, keys.h, api._p(np.zeros(2 * out.size, np.int64)))),
        (-1, lambda: lib.fheram_ram_read_plain_device(ram.h, bad, 2, keys.h, C.byref(d))),
        (-1, lambda: lib.fheram_ram_write_plain(ram.h, p.max_addr(), api._p(w.reshape(-1)), keys.h)),
        (-1, lambda: lib.fheram_ram_read_plain(ram.h, a0, 0, keys.h, api._p(out.reshape(-1)))),
        (-1, lambda: lib.fheram_ram_read_plain_device(ram.h, a0, -1, keys.h, C.byref(d))),
        (-1, lambda: lib.fheram_ram_read_plain(None, a0, 1, keys.h, api._p(out.reshape(-1)))),
        (-1, lambda: lib.fheram_ram_read_plain(ram.h, None, 1, keys.h, api._p(out.reshape(-1)))),
        (-1, lambda: lib.fheram_ram_read_plain(ram.h, a0, 1, None, api._p(out.reshape(-1)))),
        (-1, lambda: lib.fheram_ram_read_plain(ram.h, a0, 1, keys.h, None)),
        (-1, lambda: lib.fheram_ram_read_plain_device(ram.h, a0, 1, keys.h, None)),
        (-1, lambda: lib.fheram_ram_write_plain(ram.h, 0, None, keys.h)),
        (-1, lambda: lib.fheram_ram_write_plain(None, 0, api._p(w.reshape(-1)), keys.h)),
        (-1, lambda: lib.fheram_ram_read_plain(ram.h, a0, 1, other_keys.h, api._p(out.reshape(-1)))),
        (-1, lambda: lib.fheram_ram_write_plain(ram.h, 0, api._p(w.reshape(-1)), other_keys.h)),
        (-4, lambda: lib.fheram_ram_read_plain(fresh.h, a0, 1, keys.h, api._p(out.reshape(-1)))),
        (-4, lambda: lib.fheram_ram_write_plain(fresh.h, 0, api._p(w.reshape(-1)), keys.h)),
        (-2, lambda: lib.fheram_ram_read_plain(stated.h, a0, 1, keys.h, api._p(out.reshape(-1)))),
        (-2, lambda: lib.fheram_ram_write_plain(stated.h, 0, api._p(w.reshape(-1)), keys.h)),
        (-2, lambda: lib.fheram_ram_read_plain_device(rotated.h, a0, 1, keys.h, C.byref(d))),
        (-2, lambda: lib.fheram_ram_write_plain(rotated.h, 0, api._p(w.reshape(-1)), keys.h)),
    ]
    assert len(calls) == 20
    p.synchronize()
    before = lib.fheram_debug_device_bytes()
    for i, (code, call) in enumerate(calls):
        assert call() == code, (i, lib.fheram_last_error().decode())
    assert lib.fheram_debug_device_bytes() == before
    # a refused call leaves the RAM as it was; the prepared RAM still takes its write
    assert stated.state() and not ram.state()
    stated.write(w, s.address(3), keys)
    assert np.array_equal(ram.store(), s.cts)
    with pytest.raises(fr.FheRamError):
        ram.read_plain([p.max_addr()], keys)
    for r in (ram, fresh, stated, rotated):
        r.close()
    other_keys.close()
    other.close()


@pytest.mark.parametrize("n_shards", [2, 4])
def test_emulated_shards(scenario, gpu_keys, n_shards):
    s = scenario(1 << 14, 2)
    keys = gpu_keys(s)
    ws, G, N = s.params.word_size(), s.params.n_glwe(), s.params.n()
    one = _ram(s)
    addrs = _addresses(s.params.max_addr(), 9, 11)
    want = one.read_plain(addrs, keys)
    union = np.zeros_like(want)
    sentinel = -123456789
    w = _words(s, [99, 100])
    a_w = 2 * N + 17
    one.write_plain(a_w, w, keys)
    merged = np.zeros_like(s.cts).reshape(ws, G, -1)
    for shard in range(n_shards):
        r = _ram(s, shard=shard, n_shards=n_shards)
        mine = [b for b, a in enumerate(addrs) if (a // N) % n_shards == shard]
        out = np.full_like(want, sentinel)
        r.read_plain(addrs, keys, out)
        for b in range(len(addrs)):
            if b in mine:
                assert np.array_equal(out[b], want[b]), (shard, b)
                union[b] = out[b]
            else:
                assert (out[b] == sentinel).all(), (shard, b)
        dev = _download(s, r.read_plain_device(addrs, keys), len(addrs) * ws).reshape(want.shape)
        for b in range(len(addrs)):
            assert np.array_equal(dev[b], want[b] if b in mine else np.zeros_like(want[b])), (shard, b)
        r.write_plain(a_w, w, keys)                               # a no-op on the shards without polynomial 2
        merged[:, shard::n_shards] = r.store().reshape(ws, G, -1)[:, shard::n_shards]
        r.close()
    assert np.array_equal(union, want)
    assert np.array_equal(merged.reshape(-1), one.store())
    one.close()


# FHERAM_KERNEL values: every key-switch kernel a trace launch can take
FORCED = ["ks5", "ks6", "ks7", "ks8", "ks8c4"]


@pytest.mark.parametrize("name", FORCED)
def test_kernel_forced_plain(built, name):
    env = dict(os.environ)
    env["FHERAM_KERNEL"] = name
    r = subprocess.run([sys.executable, "-m", "pytest", str(Path(__file__)), "-m", "gpu", "-x", "-q", "-k",
                        "every_trace_width or extreme_digits or twice_to_one"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"FHERAM_KERNEL={name}:\n{r.stdout[-3000:]}\n{r.stderr[-1000:]}"
    assert re.search(r"\b8 passed\b", r.stdout), r.stdout[-500:]


def _nccl_worker(rank, world, port, out_dir):
    sys.path.insert(0, str(ROOT))
    import torch
    import torch.distributed as dist
    import fhe_ram_b200 as fr
    from fhe_ram_b200.sharded import ShardedRamLib
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    ws, N = 2, 4096
    p = fr.Parameters.new(device=rank, max_addr=1 << 15, word_size=ws, k_pt=8)
    sk, evk = fr.gen_keys(p)
    keys = fr.EvaluationKeysPrepared.alloc(p).prepare(evk)
    data = fr.Source(5).fill_bytes(p.max_addr() * ws)
    ref = fr.Ram.new(p)                                    # the unsharded RAM: what one GPU computes
    cts = ref.encrypt_sk(data, sk, fr.Source(11), fr.Source(12))
    addrs = [0, 1, N - 1, N, 3 * N + 5, (1 << 15) - 1, 5 * N + 77, 0]
    fails = []
    lib = ShardedRamLib(p, rank, world, cts)
    if not np.array_equal(lib.read_plain(addrs, keys), ref.read_plain(addrs, keys)):
        fails.append("read_plain")
    w = np.stack([fr.encrypt_glwe(p, 60 + i, sk) for i in range(ws)])
    for a in (N + 3, 2 * N + 9):                           # held by rank 1 and rank 0 of two
        lib.write_plain(a, w if rank == 0 else None, keys)  # rank 0's word is broadcast
        ref.write_plain(a, w, keys)
    mine = lib.store().reshape(ws, p.n_glwe(), -1)
    full = ref.store().reshape(ws, p.n_glwe(), -1)
    if not np.array_equal(mine[:, rank::world], full[:, rank::world]):
        fails.append("RAM limbs after write_plain")
    if not np.array_equal(lib.read_plain(addrs, keys), ref.read_plain(addrs, keys)):
        fails.append("read_plain after write_plain")
    lib.close()
    Path(f"{out_dir}/r{rank}.txt").write_text("\n".join(fails))
    dist.barrier()
    dist.destroy_process_group()


def test_plain_access_over_nccl(built, tmp_path):
    import torch
    import torch.multiprocessing as mp
    world = 2
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs >= {world} GPUs")
    sock = socket.socket(); sock.bind(("127.0.0.1", 0)); port = sock.getsockname()[1]; sock.close()
    mp.spawn(_nccl_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        fails = (tmp_path / f"r{r}.txt").read_text()
        assert fails == "", f"rank {r}: {fails}"
