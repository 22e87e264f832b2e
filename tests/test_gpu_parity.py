"""-m gpu: parity of the CUDA path (through the C ABI) against the CPU oracle on identical inputs.
Bit-exact on every ciphertext limb; decrypt-level acceptance as examples/fhe-ram.rs:104-176."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _rand_glwe(rng, params, n):
    # normalised base-2^17 limbs, BASELINE.json config 2 distribution
    return rng.integers(-(1 << 16), 1 << 16, size=(n, params.glwe_len()), dtype=np.int64)


def test_external_product_matches_oracle(scenario):
    from fhe_ram_b200 import api
    s = scenario()
    rng = np.random.default_rng(1)
    n = 5
    cts = _rand_glwe(rng, s.params, n)
    addr = s.address(1234)
    ggsw = addr.data[: s.params.ggsw_len()]
    got = api.external_product_batch(s.params, cts, ggsw)
    for i in range(n):
        want = s.orc.external_product(cts[i], ggsw)
        assert np.array_equal(got[i], want), f"ct {i}: {np.count_nonzero(got[i] != want)} limbs differ"


def test_external_product_adversarial_limbs(scenario):
    """extreme digits (all -2^16 / 2^16-1) stress the f64 exactness margin (SURVEY.md 7)."""
    from fhe_ram_b200 import api
    s = scenario()
    p = s.params
    cts = np.full((2, p.glwe_len()), -(1 << 16), dtype=np.int64)
    cts[1, :] = (1 << 16) - 1
    ggsw = np.full(p.ggsw_len(), -(1 << 16), dtype=np.int64)
    got = api.external_product_batch(p, cts, ggsw)
    for i in range(2):
        assert np.array_equal(got[i], s.orc.external_product(cts[i], ggsw))


def test_coordinate_product_chain(scenario):
    from fhe_ram_b200 import api
    s = scenario()
    rng = np.random.default_rng(2)
    cts = _rand_glwe(rng, s.params, 3)
    addr = s.address(4321)
    nd = len(s.params.base2d()[0])
    ggsws = addr.data[: nd * s.params.ggsw_len()]
    got = api.coordinate_product(s.params, cts, ggsws, nd)
    for i in range(3):
        assert np.array_equal(got[i], s.orc.coordinate_product(cts[i], ggsws, nd))


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_automorphism_variants(scenario, gpu_keys, mode):
    from fhe_ram_b200 import api
    s = scenario()
    keys = gpu_keys(s)
    rng = np.random.default_rng(3 + mode)
    cts = _rand_glwe(rng, s.params, 2)
    for gi in (0, 1, 7, 11):
        got = api.glwe_automorphism(s.params, keys, gi, mode, cts)
        for i in range(2):
            x = cts[i] if mode == 0 else s.orc.glwe_rsh(1, cts[i])
            want = s.orc.automorphism(s.okeys, gi, mode, x)
            assert np.array_equal(got[i], want), (mode, gi, i, np.count_nonzero(got[i] != want))


def test_trace_matches_oracle(scenario, gpu_keys):
    from fhe_ram_b200 import api
    s = scenario()
    keys = gpu_keys(s)
    rng = np.random.default_rng(5)
    cts = _rand_glwe(rng, s.params, 3)
    got = api.glwe_trace(s.params, keys, cts)
    for i in range(3):
        assert np.array_equal(got[i], s.orc.trace(s.okeys, cts[i]))
    got = api.glwe_trace(s.params, keys, cts, 3, 9)
    assert np.array_equal(got[0], s.orc.trace(s.okeys, cts[0], 3, 9))


def _extreme_glwe(rng, params, n):
    """ciphertexts whose digits sit on the edges of the balanced range: the word-domain kernels
    (kernels_ks3.cuh) replace digit carry chains by arithmetic mod 2^51 on biased words, so the cases to
    pin are -2^16 (whose negation under a rotation / automorphism is the non-canonical +2^16), 2^16 - 1,
    and values whose top digit wraps"""
    L = params.glwe_len()
    cts = np.empty((n, L), dtype=np.int64)
    cts[0, :] = -(1 << 16)
    cts[1 % n, :] = (1 << 16) - 1
    for i in range(2, n):
        cts[i] = rng.choice(np.array([-(1 << 16), -(1 << 16) + 1, -1, 0, 1, (1 << 16) - 2, (1 << 16) - 1], dtype=np.int64), size=L)
    return cts


def test_trace_adversarial_limbs(scenario, gpu_keys):
    from fhe_ram_b200 import api
    s = scenario()
    keys = gpu_keys(s)
    cts = _extreme_glwe(np.random.default_rng(15), s.params, 4)
    got = api.glwe_trace(s.params, keys, cts)
    for i in range(4):
        want = s.orc.trace(s.okeys, cts[i])
        assert np.array_equal(got[i], want), (i, np.count_nonzero(got[i] != want))


def test_packer_adversarial_limbs(scenario, gpu_keys):
    from fhe_ram_b200 import api
    s = scenario()
    keys = gpu_keys(s)
    n = 4
    cts = _extreme_glwe(np.random.default_rng(16), s.params, n)
    got = api.glwe_pack(s.params, keys, cts)
    N, log_n = s.params.n(), s.params.log_n()
    feed = []
    for j in range(N):
        jr = int(format(j, f"0{log_n}b")[::-1], 2)
        feed.append(cts[jr] if jr < n else None)
    want = s.orc.pack(s.okeys, feed)
    assert np.array_equal(got, want), np.count_nonzero(got != want)


@pytest.mark.parametrize("n", [1, 2, 8])
def test_packer_matches_oracle(scenario, gpu_keys, n):
    """GLWEPacker fed as src/ram.rs:424-449 does (bit-reversed order, None elsewhere)."""
    from fhe_ram_b200 import api
    s = scenario()
    keys = gpu_keys(s)
    rng = np.random.default_rng(6 + n)
    cts = _rand_glwe(rng, s.params, n)
    got = api.glwe_pack(s.params, keys, cts)
    N, log_n = s.params.n(), s.params.log_n()
    feed = []
    for j in range(N):
        jr = int(format(j, f"0{log_n}b")[::-1], 2)
        feed.append(cts[jr] if jr < n else None)
    want = s.orc.pack(s.okeys, feed)
    assert np.array_equal(got, want), np.count_nonzero(got != want)


def test_ggsw_invert_matches_oracle(scenario, gpu_keys):
    from fhe_ram_b200 import api
    s = scenario()
    keys = gpu_keys(s)
    addr = s.address(777)
    L = s.params.ggsw_len()
    got = api.ggsw_invert(s.params, keys, addr.data[: 2 * L])
    for i in range(2):
        want = s.orc.ggsw_automorphism_inv(s.okeys, addr.data[i * L:(i + 1) * L])
        assert np.array_equal(got[i * L:(i + 1) * L], want), np.count_nonzero(got[i * L:(i + 1) * L] != want)


@pytest.mark.parametrize("max_addr,word_size", [(1 << 13, 2), (1 << 12, 1), (1 << 10, 1), (1 << 14, 4)])
def test_read_rpw_write_bit_exact(scenario, gpu_keys, max_addr, word_size):
    """The acceptance scenario of examples/fhe-ram.rs:97-176, limb-for-limb against the oracle."""
    s = scenario(max_addr, word_size)
    fr, p = s.fr, s.params
    keys = gpu_keys(s)
    ram = fr.Ram.new(p)
    ram.load(s.cts)
    oram = s.orc.ram_new(s.cts.copy())
    idx = s.src.next_u32() % max_addr
    addr = s.address(idx)

    got = ram.read(addr, keys)
    rc, want = s.orc.ram_read(oram, addr.data, s.okeys)
    assert rc == 0 and np.array_equal(got, want), np.count_nonzero(got != want)
    s.check_decrypt(got, idx)

    got = ram.read_prepare_write(addr, keys)
    rc, want = s.orc.ram_read_prepare_write(oram, addr.data, s.okeys)
    assert rc == 0 and np.array_equal(got, want)
    assert ram.state() and np.array_equal(ram.store(), s.orc.ram_store(oram))
    if len(p.base2d()) > 1:
        assert np.array_equal(ram.tree_store(), s.orc.ram_tree_store(oram))

    value = s.src.fill_bytes(word_size)
    w = np.stack([fr.encrypt_glwe(p, int(v), s.sk) for v in value])
    ram.write(w, addr, keys)
    assert s.orc.ram_write(oram, w.reshape(-1), addr.data, s.okeys) == 0
    assert not ram.state()
    assert np.array_equal(ram.store(), s.orc.ram_store(oram)), "RAM limbs differ after write"
    if len(p.base2d()) > 1:
        assert np.array_equal(ram.tree_store(), s.orc.ram_tree_store(oram))

    data2 = s.data.copy()
    data2[idx * word_size:(idx + 1) * word_size] = value
    got = ram.read(addr, keys)
    rc, want = s.orc.ram_read(oram, addr.data, s.okeys)
    assert np.array_equal(got, want)
    s.check_decrypt(got, idx, data2)
    other = (idx + p.n() + 1) % max_addr
    got = ram.read(s.address(other), keys)
    s.check_decrypt(got, other, data2)
    ram.close()


def test_batched_reads_equal_single_reads(scenario, gpu_keys):
    s = scenario()
    fr, p = s.fr, s.params
    keys = gpu_keys(s)
    ram = fr.Ram.new(p)
    ram.load(s.cts)
    idxs = [0, 1, p.n() - 1, p.n(), p.max_addr() - 1, 4242 % p.max_addr(), 77]
    addrs = [s.address(i) for i in idxs]
    batch = fr.Address.batch(p, addrs)
    got = ram.read_batch(batch, keys)
    oram = s.orc.ram_new(s.cts.copy())
    for b, (i, a) in enumerate(zip(idxs, addrs)):
        rc, want = s.orc.ram_read(oram, a.data, s.okeys)
        assert np.array_equal(got[b], want), (b, i)
        s.check_decrypt(got[b], i)
        assert np.array_equal(ram.read(a, keys), want)
    ram.close()


def test_host_buffer_batch_pipeline(scenario, gpu_keys):
    """fheram_ram_read_batch_host (chunked, double-buffered) == one read per address."""
    s = scenario(1 << 13, 2)
    fr, p = s.fr, s.params
    keys = gpu_keys(s)
    ram = fr.Ram.new(p)
    ram.load(s.cts)
    idxs = [(37 * i + 11) % p.max_addr() for i in range(70)]      # > 2 chunks of 32
    addrs = [s.address(i) for i in idxs]
    limbs = np.stack([a.data for a in addrs])
    got = ram.read_batch_host(limbs, len(idxs), keys)
    for b in (0, 1, 31, 32, 63, 64, 69):
        assert np.array_equal(got[b], ram.read(addrs[b], keys)), b
        s.check_decrypt(got[b], idxs[b])
    # compact host format (int32 limbs in and out): the same limbs
    got32 = ram.read_batch_host_i32(limbs.astype(np.int32), len(idxs), keys)
    assert got32.dtype == np.int32 and np.array_equal(got32.astype(np.int64), got)
    # packed host format (17-bit fields)
    from fhe_ram_b200 import api
    got17 = ram.read_batch_host_p17(api.pack17(limbs), len(idxs), keys)
    assert np.array_equal(got17, got32)
    bad = limbs.copy()
    bad[3, 5] = 1 << 40
    with pytest.raises(fr.FheRamError) as e:
        ram.read_batch_host(bad, len(idxs), keys)
    assert e.value.code == -6
    ram.close()


def test_state_machine_and_errors(scenario, gpu_keys):
    """assert!s of src/ram.rs:182-185,243,393-396,555-558 become error codes."""
    s = scenario()
    fr, p = s.fr, s.params
    keys = gpu_keys(s)
    ram = fr.Ram.new(p)
    addr = s.address(3)
    with pytest.raises(fr.FheRamError) as e:
        ram.read(addr, keys)
    assert e.value.code == -4
    ram.load(s.cts)
    w = np.stack([fr.encrypt_glwe(p, 1, s.sk) for _ in range(p.word_size())])
    with pytest.raises(fr.FheRamError) as e:
        ram.write(w, addr, keys)
    assert e.value.code == -3
    ram.read_prepare_write(addr, keys)
    with pytest.raises(fr.FheRamError) as e:
        ram.read(addr, keys)
    assert e.value.code == -2
    with pytest.raises(fr.FheRamError):
        ram.write(w[:1], addr, keys)
    ram.write(w, addr, keys)
    ram.read(addr, keys)
    with pytest.raises(fr.FheRamError):
        ram.encrypt_sk(s.data[:-1], s.sk, s.xa, s.xe)
    ram.close()


def test_full_size_2pow18_properties(scenario, gpu_keys):
    """BASELINE.json size (2^18 x 4 B): size-independent properties -- every read decrypts to the
    plaintext word, write/read-back round trip, untouched words survive a write."""
    s = scenario(1 << 18, 4, 9)
    fr, p = s.fr, s.params
    keys = gpu_keys(s)
    ram = fr.Ram.new(p)
    ram.load(s.cts)
    idxs = [0, 4095, 4096, (1 << 18) - 1, 123457]
    batch = fr.Address.batch(p, [s.address(i) for i in idxs])
    got = ram.read_batch(batch, keys)
    for b, i in enumerate(idxs):
        s.check_decrypt(got[b], i)
    addr = s.address(200001)
    s.check_decrypt(ram.read_prepare_write(addr, keys), 200001)
    value = np.array([1, 2, 100, 127], dtype=np.uint8)
    w = np.stack([fr.encrypt_glwe(p, int(v), s.sk) for v in value])
    ram.write(w, addr, keys)
    data2 = s.data.copy()
    data2[200001 * 4:200001 * 4 + 4] = value
    s.check_decrypt(ram.read(addr, keys), 200001, data2)
    for i in (200000, 200002, 200001 - 4096, 5):
        s.check_decrypt(ram.read(s.address(i), keys), i, data2)
    ram.close()


def test_wide_kernels_repeatable_and_equal_to_narrow(scenario, gpu_keys):
    """2^18 x 4 B: a batch (wide launches: k_ext8 / k_ks7 / k_ks4, in-place word accumulation) must give, limb
    for limb, what single reads (narrow launches: k_ext9 / k_ks8 / k_ks6 / k_ks5) give, and the
    same limbs on every repetition (compute-sanitizer is not available on the GPU pool: races would show up here)."""
    s = scenario(1 << 18, 4, 9)
    fr, p = s.fr, s.params
    keys = gpu_keys(s)
    ram = fr.Ram.new(p)
    ram.load(s.cts)
    idxs = [3, 4097, 77777, (1 << 18) - 2]
    addrs = [s.address(i) for i in idxs]
    batch = fr.Address.batch(p, addrs)
    first = ram.read_batch(batch, keys)
    for _ in range(4):
        again = ram.read_batch(batch, keys)
        assert np.array_equal(first, again), np.count_nonzero(first != again)
    for b, a in enumerate(addrs):
        single = ram.read(a, keys)
        assert np.array_equal(single, first[b]), (b, np.count_nonzero(single != first[b]))
        s.check_decrypt(first[b], idxs[b])
    ram.close()


@pytest.mark.parametrize("n_shards", [2, 4])
def test_sharded_stages_on_one_gpu(scenario, gpu_keys, n_shards):
    """The sharded path of the C ABI (SURVEY.md 8e) with every shard emulated on one GPU: local
    stages per shard, partials concatenated rank-major (what the NCCL exchange produces), finish.
    Must equal the unsharded read / read_prepare_write / write limb for limb."""
    import ctypes as C
    from fhe_ram_b200 import api
    s = scenario(1 << 14, 2)
    fr, p = s.fr, s.params
    keys = gpu_keys(s)
    L = p.word_size() * p.glwe_len()
    idxs = [5, 4096 + 9, (1 << 14) - 1]
    addrs = [s.address(i) for i in idxs]
    batch = fr.Address.batch(p, addrs)
    ref = fr.Ram.new(p)
    ref.load(s.cts)
    want = ref.read_batch(batch, keys)
    shards = [fr.Ram(p, shard=g, n_shards=n_shards) for g in range(n_shards)]
    for r in shards:
        r.load(s.cts)

    def gather(fn):
        parts = []
        for r in shards:
            d = C.c_void_p()
            api._check(fn(r, C.byref(d)))
            n = (batch.count if fn is local_read else 1) * p.word_size()
            host = np.zeros(n * p.glwe_len(), dtype=np.int64)
            api._check(api.lib().fheram_download_glwe(p.module(), d, n, api._p(host)))
            parts.append(host)
        return np.concatenate(parts)

    def upload(limbs):
        # park the gathered partials in a device buffer via a scratch RAM-less route: an Address-free
        # upload helper does not exist in the ABI, so reuse torch for the device buffer
        import torch
        t = torch.from_numpy(limbs.astype(np.int32)).cuda()
        return t

    local_read = lambda r, d: api.lib().fheram_ram_read_local_device(r.h, batch.device(), keys.h, d)
    g = upload(gather(local_read))
    for r in shards[:2]:
        d = C.c_void_p()
        api._check(api.lib().fheram_ram_read_finish_device(r.h, C.c_void_p(g.data_ptr()), batch.count, 0,
                                                           batch.count, batch.device(), 0, keys.h, C.byref(d)))
        got = np.zeros(batch.count * L, dtype=np.int64)
        api._check(api.lib().fheram_download_glwe(p.module(), d, batch.count * p.word_size(), api._p(got)))
        assert np.array_equal(got.reshape(want.shape), want)

    # read_prepare_write + write, replicated finish, no communication for the write
    a = addrs[1]
    want_rpw = ref.read_prepare_write(a, keys)
    local_rpw = lambda r, d: api.lib().fheram_ram_rpw_local_device(r.h, a.device(), keys.h, d)
    g = upload(gather(local_rpw))
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


def test_cpp_host_layer_runs_the_example_scenario(built):
    """fhe_ram_b200/cpp/example_fhe_ram = examples/fhe-ram.rs:34-177 through fheram.hpp (the
    compiled-language mirror of the Rust API): exits 0 only if every decrypt/noise assert holds."""
    import subprocess
    from pathlib import Path
    exe = Path(__file__).resolve().parent.parent / "fhe_ram_b200" / "cpp" / "example_fhe_ram"
    r = subprocess.run([str(exe), "14"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "READ Elapsed time" in r.stdout and "WRITE Elapsed time" in r.stdout and r.stdout.strip().endswith("OK")


def test_scaled_ram_2pow22_properties(scenario, gpu_keys):
    """BASELINE.json config 5 size (2^22 entries; one byte lane to keep the oracle-free check fast):
    coordinate 1 has four digits [3,3,3,1]; reads decrypt to the plaintext, write round trip."""
    s = scenario(1 << 22, 1, 8)
    fr, p = s.fr, s.params
    assert p.base2d() == [[3, 3, 3, 3], [3, 3, 3, 1]] and p.n_glwe() == 1024
    keys = gpu_keys(s)
    ram = fr.Ram.new(p)
    ram.load(s.cts)
    idxs = [0, (1 << 22) - 1, 4096 * 513 + 77, 1234567]
    got = ram.read_batch(fr.Address.batch(p, [s.address(i) for i in idxs]), keys)
    for b, i in enumerate(idxs):
        s.check_decrypt(got[b], i)
    a = s.address(3000001)
    s.check_decrypt(ram.read_prepare_write(a, keys), 3000001)
    ram.write(np.stack([fr.encrypt_glwe(p, 99, s.sk)]), a, keys)
    d2 = s.data.copy()
    d2[3000001] = 99
    s.check_decrypt(ram.read(a, keys), 3000001, d2)
    s.check_decrypt(ram.read(s.address(3000002), keys), 3000002, d2)
    ram.close()


def test_external_product_microbench_shape(scenario):
    """BASELINE.json config 2 at reduced batch: n GLWE x one GGSW, random 17-bit limbs, bit-exact."""
    from fhe_ram_b200 import api
    s = scenario()
    rng = np.random.default_rng(42)
    n = 300          # > 2 waves of 148 CTAs
    cts = _rand_glwe(rng, s.params, n)
    ggsw = rng.integers(-(1 << 16), 1 << 16, size=s.params.ggsw_len(), dtype=np.int64)
    got = api.external_product_batch(s.params, cts, ggsw)
    for i in (0, 147, 148, 299):
        assert np.array_equal(got[i], s.orc.external_product(cts[i], ggsw)), i


def test_noise_stays_within_budget_over_write_cycles(built):
    """§8(f).3 noise instrumentation: ten rpw/write cycles at random addresses; an untouched word and
    every freshly written word keep decrypting with noise below the example's bound 2^-(k_pt+1), and
    the growth per cycle is sub-bit (README.md:36: tens of millions of accesses before refresh)."""
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tools"))
    import noise_growth
    rows = noise_growth.run(max_addr_log2=13, word_size=1, cycles=10, verbose=False)
    assert all(r[1] < -9 for r in rows)
    assert all(r[2] < -9 for r in rows[1:])
    assert rows[-1][1] - rows[1][1] < 6.0       # after the first write the noise floor moves slowly
