"""-m gpu: RAMs whose polynomial count m = ceil(max_addr / N) is not a power of two, limb for limb against the CPU oracle.

The packer tree of such a RAM keeps only its m present inputs and runs one mixed level (DESIGN.md §1): pairs whose
second operand exists take the two-sided combine, the others the one-sided one, in one launch (MODE_MIXED).  Under the
default launch-width rule on a 148-SM B200 that launch, of H = 2^(ceil(log2 m) - 1) items for a single pack, lands on
k_ks8<8> for n = 3, 5 (H = 2, 4), k_ks8<4> for n = 20 (H = 16), k_ks6 for n = 100 (H = 64), k_ks5 for n = 200 (H = 128)
and k_ks4 for n = 300, 4095 (H = 256, 2048).  The subprocess sweep at the end forces every combine kernel.
"""
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
SIZES = [(3 * 4096, 2, 8), (5 * 4096 + 17, 1, 8), (3 << 16, 4, 9)]


def _rand_glwe(rng, params, n):
    return rng.integers(-(1 << 16), 1 << 16, size=(n, params.glwe_len()), dtype=np.int64)


def _feed(params, cts):
    N, log_n = params.n(), params.log_n()
    feed = []
    for j in range(N):
        h = int(format(j, f"0{log_n}b")[::-1], 2)
        feed.append(cts[h] if h < len(cts) else None)
    return feed


@pytest.mark.parametrize("n", [3, 5, 20, 100, 200, 300, 4095])
def test_pack_any_width(scenario, gpu_keys, n):
    from fhe_ram_b200 import api
    s = scenario()
    keys = gpu_keys(s)
    cts = _rand_glwe(np.random.default_rng(500 + n), s.params, n)
    s.params.profile(True)
    got = api.glwe_pack(s.params, keys, cts)
    recs = s.params.profile_records(64)
    s.params.profile(False)
    want = s.orc.pack(s.okeys, _feed(s.params, cts))
    assert np.array_equal(got, want), np.count_nonzero(got != want)
    # launches: one trace chain over the n inputs (none when log2 n rounds up to 12), the mixed level over H pairs,
    # then the two-sided levels H/2 ... 1
    L = (n - 1).bit_length()
    H = 1 << (L - 1)
    ks = [(c, items, steps) for c, _, items, steps in recs if c in ("trace", "combine2")]
    chain = [(n, 12 - L)] if L < 12 else []
    assert [(i, st) for c, i, st in ks if c == "trace"] == chain
    assert [i for c, i, _ in ks if c == "combine2"] == [H >> k for k in range(L)]


def _oracle_ram(s):
    s.orc.set_ram_threads(8)
    return s.orc.ram_new(s.cts.copy())


@pytest.mark.parametrize("max_addr,word_size,k_pt", SIZES)
def test_read_rpw_write_any_size(scenario, gpu_keys, max_addr, word_size, k_pt):
    s = scenario(max_addr, word_size, k_pt)
    fr, p = s.fr, s.params
    assert p.n_glwe() & (p.n_glwe() - 1)
    keys = gpu_keys(s)
    ram = fr.Ram.new(p)
    ram.load(s.cts)
    oram = _oracle_ram(s)
    idx = max_addr - 2
    addr = s.address(idx)

    got = ram.read(addr, keys)
    rc, want = s.orc.ram_read(oram, addr.data, s.okeys)
    assert rc == 0 and np.array_equal(got, want), np.count_nonzero(got != want)
    s.check_decrypt(got, idx)

    got = ram.read_prepare_write(addr, keys)
    rc, want = s.orc.ram_read_prepare_write(oram, addr.data, s.okeys)
    assert rc == 0 and np.array_equal(got, want)
    s.check_decrypt(got, idx)
    assert ram.state() and np.array_equal(ram.store(), s.orc.ram_store(oram))
    assert np.array_equal(ram.tree_store(), s.orc.ram_tree_store(oram))

    value = np.array([(37 * i + 5) % 256 for i in range(word_size)], dtype=np.uint8)
    w = np.stack([fr.encrypt_glwe(p, int(v), s.sk) for v in value])
    ram.write(w, addr, keys)
    assert s.orc.ram_write(oram, w.reshape(-1), addr.data, s.okeys) == 0
    assert not ram.state()
    assert np.array_equal(ram.store(), s.orc.ram_store(oram)), "RAM limbs differ after write"
    assert np.array_equal(ram.tree_store(), s.orc.ram_tree_store(oram))

    data2 = s.data.copy()
    data2[idx * word_size:(idx + 1) * word_size] = value
    got = ram.read(addr, keys)
    rc, want = s.orc.ram_read(oram, addr.data, s.okeys)
    assert np.array_equal(got, want)
    s.check_decrypt(got, idx, data2)
    for other in (0, idx - p.n(), idx + 1):
        s.check_decrypt(ram.read(s.address(other), keys), other, data2)
    ram.close()


def test_batched_reads_any_size(scenario, gpu_keys, monkeypatch):
    from fhe_ram_b200 import api
    monkeypatch.setenv("FHERAM_CHUNK", "3")  # several chunks in every batched path
    s = scenario(3 * 4096, 2, 8)
    fr, p = s.fr, s.params
    keys = gpu_keys(s)
    ram = fr.Ram.new(p)
    ram.load(s.cts)
    idxs = [0, 1, 4095, 4096, 8191, 8192, 3 * 4096 - 1, 5000]
    addrs = [s.address(i) for i in idxs]
    n = len(idxs)
    batch = fr.Address.batch(p, addrs)
    singles = np.stack([ram.read(a, keys) for a in addrs])
    oram = _oracle_ram(s)
    rc, want = s.orc.ram_read_many(oram, np.concatenate([a.data for a in addrs]), n, s.okeys, 8)
    assert rc == 0 and np.array_equal(singles, want)
    for b, i in enumerate(idxs):
        s.check_decrypt(singles[b], i)

    assert np.array_equal(ram.read_batch(batch, keys), want)
    d = ram.read_batch_device(batch, keys)
    dev = np.zeros(n * p.word_size() * p.glwe_len(), dtype=np.int64)
    api._check(api.lib().fheram_download_glwe(p.module(), C.c_void_p(d), n * p.word_size(), api._p(dev)))
    assert np.array_equal(dev.reshape(want.shape), want)
    limbs = np.stack([a.data for a in addrs])
    assert np.array_equal(ram.read_batch_host(limbs, n, keys), want)
    got32 = ram.read_batch_host_i32(limbs.astype(np.int32), n, keys)
    assert np.array_equal(got32.astype(np.int64), want)
    assert np.array_equal(ram.read_batch_host_p17(api.pack17(limbs), n, keys), got32)
    ram.close()


def test_device_encrypt_and_decrypt_any_size(scenario):
    s = scenario(3 * 4096, 2, 8)
    fr, p = s.fr, s.params
    ram = fr.Ram.new(p)
    ram.encrypt_sk_gpu(s.data, s.sk, fr.Source(11), fr.Source(12))  # the Sources Scenario encrypted s.cts with
    assert np.array_equal(ram.store(), s.cts)
    values, err = ram.decrypt_sk(s.sk)
    want_v, want_e = fr.decrypt_ram(p, s.cts, s.sk)
    assert np.array_equal(values, want_v) and np.array_equal(err, want_e)
    w = min(8, p.k_glwe_pt())
    plain = np.array([fr.cast_u8_to_signed(int(b), w) for b in s.data], dtype=np.int16).reshape(values.shape)
    assert np.array_equal(values, plain)
    ram.close()


def test_sharded_create_is_refused(scenario):
    s = scenario(3 * 4096, 2, 8)
    fr = s.fr
    with pytest.raises(fr.FheRamError) as e:
        fr.Ram(s.params, shard=0, n_shards=2)
    assert e.value.code == -1 and "power of two" in str(e.value)


@pytest.mark.parametrize("name", ["ks4", "ks5", "ks6", "ks8", "ks8c4"])
def test_mixed_level_on_every_combine_kernel(built, name):
    """the pack and the small read cases of this file with FHERAM_KERNEL forcing each combine kernel"""
    env = dict(os.environ)
    env["FHERAM_KERNEL"] = name
    sel = "test_pack_any_width or (test_read_rpw_write_any_size and not 196608)"
    r = subprocess.run([sys.executable, "-m", "pytest", str(ROOT / "tests" / "test_gpu_any_size.py"), "-m", "gpu",
                        "-x", "-q", "-k", sel], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, f"FHERAM_KERNEL={name}:\n{r.stdout[-3000:]}\n{r.stderr[-1000:]}"
    assert " passed" in r.stdout
