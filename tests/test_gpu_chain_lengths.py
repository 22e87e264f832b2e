"""-m gpu: external-product and trace chains of every length the C ABI accepts, limb for limb against the CPU oracle.

The chain kernels carry state from one step to the next: k_ext9 alternates its contribution slabs by step parity and
fills its matrix ring one step ahead, k_ext8 keeps the ciphertext on chip between steps, the key-switch kernels run
the trace steps back to back.  A read at the default decomposition only runs external-product chains of 1..4 steps;
the address decomposition `decomp_n` makes them up to 8 long ([1]*7+[5]), fheram_coordinate_product accepts 12, and a
one-sided packer chain has 12 - ceil(log2 G) steps for any G up to 4096.  So every length 1..12 is run here, at widths
that the launch-width rule (DESIGN.md 3.4) sends to each kernel class, and test_kernel_forced_chains repeats the lot
with each kernel forced by FHERAM_KERNEL, adding a width at which the forced cluster kernels and k_ks5 take several
ciphertexts per cluster or CTA."""
import os
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent

LENGTHS = list(range(1, 13))
# default rule on a 148-SM B200: k_ext9<8>, k_ext9<4>, k_ext8
EXT_WIDTHS = [2, 24, 160]
# default rule on a 148-SM B200: k_ks8<8>, k_ks8<4>, k_ks6, k_ks5, k_ks7
TRACE_WIDTHS = [2, 24, 70, 100, 160]


def _widths(base):
    """under a forced kernel, also 2 S + 3: more than one item per cluster of the forced cluster kernels and per CTA of
    k_ks5 (k_ks6 keeps its own rule above 2 n > S, the default one)"""
    if not os.environ.get("FHERAM_KERNEL"):
        return base
    import torch
    return base + [2 * torch.cuda.get_device_properties(0).multi_processor_count + 3]


def _rand_glwe(rng, params, n):
    return rng.integers(-(1 << 16), 1 << 16, size=(n, params.glwe_len()), dtype=np.int64)


def _sample(n):
    return sorted({0, n // 2, n - 1})


@pytest.fixture(scope="module")
def ggsw_sets(scenario):
    """16 real GGSWs (the address 0xB5A5C at 2^20 with decomp_n [1]*7+[5]: coordinates [1]*7+[5] and [1]*8) and 16 of
    random limbs in [-2^16, 2^16)"""
    s = scenario()
    fr = s.fr
    p = fr.Parameters.new(max_addr=1 << 20, word_size=1, k_pt=8, decomp_n=[1] * 7 + [5])
    assert p.n_ggsw() == 16 and p.ggsw_len() == s.params.ggsw_len()
    real = fr.Address.alloc(p).encrypt_sk(p, 0xB5A5C, s.sk, fr.Source(61), fr.Source(62)).data
    rand = np.random.default_rng(63).integers(-(1 << 16), 1 << 16, size=real.size, dtype=np.int64)
    return {"real": real, "random": rand}


@pytest.mark.parametrize("kind", ["real", "random"])
@pytest.mark.parametrize("k", LENGTHS)
def test_external_product_chain_of_every_length(scenario, ggsw_sets, k, kind):
    from fhe_ram_b200 import api
    s = scenario()
    L = s.params.ggsw_len()
    # the chain starts at a different GGSW for each length, so that the real set's sixteen all take part
    first = (3 * k) % (16 - k + 1)
    ggsws = ggsw_sets[kind][first * L:(first + k) * L]
    for n in _widths(EXT_WIDTHS):
        cts = _rand_glwe(np.random.default_rng(1000 * k + n), s.params, n)
        got = api.coordinate_product(s.params, cts, ggsws, k)
        for i in _sample(n):
            want = s.orc.coordinate_product(cts[i], ggsws, k)
            assert np.array_equal(got[i], want), \
                f"{kind} k={k} n={n} ct {i}: {np.count_nonzero(got[i] != want)} limbs differ"


def test_external_product_chain_of_13_is_refused(scenario, ggsw_sets):
    from fhe_ram_b200 import api
    s = scenario()
    fr = s.fr
    cts = _rand_glwe(np.random.default_rng(13), s.params, 2)
    ggsws = ggsw_sets["random"][: 13 * s.params.ggsw_len()]
    with pytest.raises(fr.FheRamError) as e:
        api.coordinate_product(s.params, cts, ggsws, 13)
    assert e.value.code == -1


@pytest.mark.parametrize("window", ["head", "tail"])
@pytest.mark.parametrize("k", LENGTHS)
def test_trace_chain_of_every_length(scenario, gpu_keys, k, window):
    """[0, k): the one-sided packer levels of a RAM of 2^(12-k) polynomials; [12 - k, 12): the end of the final trace"""
    from fhe_ram_b200 import api
    s = scenario()
    keys = gpu_keys(s)
    g0, g1 = (0, k) if window == "head" else (12 - k, 12)
    for n in _widths(TRACE_WIDTHS):
        cts = _rand_glwe(np.random.default_rng(2000 * k + n + (0 if window == "head" else 500)), s.params, n)
        got = api.glwe_trace(s.params, keys, cts, g0, g1)
        for i in _sample(n):
            want = s.orc.trace(s.okeys, cts[i], g0, g1)
            assert np.array_equal(got[i], want), \
                f"[{g0}, {g1}) n={n} ct {i}: {np.count_nonzero(got[i] != want)} limbs differ"


# FHERAM_KERNEL values.  Forcing an external-product kernel leaves every trace launch on the default rule and the other
# way round, so each name runs the chains of its own class.  ks4 serves only two-sided combines, which no chain here
# runs; test_gpu_kernel_variants.py forces it through the packer.
FORCED = {
    "ext8": "external_product_chain_of_every_length",
    "ext9": "external_product_chain_of_every_length",
    "ext9c4": "external_product_chain_of_every_length",
    "ks8": "trace_chain_of_every_length",
    "ks8c4": "trace_chain_of_every_length",
    "ks7": "trace_chain_of_every_length",
    "ks6": "trace_chain_of_every_length",
    "ks5": "trace_chain_of_every_length",
}


@pytest.mark.parametrize("name", sorted(FORCED))
def test_kernel_forced_chains(built, name):
    env = dict(os.environ)
    env["FHERAM_KERNEL"] = name
    r = subprocess.run([sys.executable, "-m", "pytest", str(Path(__file__)), "-m", "gpu", "-x", "-q", "-k", FORCED[name]],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"FHERAM_KERNEL={name}:\n{r.stdout[-3000:]}\n{r.stderr[-1000:]}"
    assert re.search(r"\b24 passed\b", r.stdout), r.stdout[-500:]
