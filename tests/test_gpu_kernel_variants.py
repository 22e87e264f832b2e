"""Every kernel generation behind the same C ABI must give the same limbs as the oracle.

The library picks a kernel per launch from the launch width (DESIGN.md 3.4; the default selection is what
test_gpu_parity.py itself runs, test_gpu_launch_widths.py pins the rule, and the wide kernels are checked at BASELINE
sizes in test_gpu_baseline_sizes.py).  The small parity cases of test_gpu_parity.py only produce narrow launches, so
each kernel is forced with FHERAM_KERNEL through the whole limb-level parity set (external product, chains, trace,
packer, read / read_prepare_write / write at four parameter sets, batched, sharded) in a subprocess.
"""
import os
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent

SELECT = ("test_external_product_matches_oracle or test_external_product_adversarial_limbs or "
          "test_coordinate_product_chain or test_trace_matches_oracle or test_packer_matches_oracle or "
          "test_trace_adversarial_limbs or test_packer_adversarial_limbs or "
          "test_read_rpw_write_bit_exact or test_batched_reads_equal_single_reads or "
          "test_sharded_stages_on_one_gpu")

# FHERAM_KERNEL values
VARIANTS = (
    # word-domain key switch with in-place accumulation and two tiles in flight (k_ks4) for every two-sided combine
    "ks4",
    # 16-point-per-thread transform with two exchanges, two polynomials per CTA (k_ks7) for every trace chain
    "ks7",
    # one operation per SM, 512 threads, tiles parked in tensor memory (k_ks5), trace and combine
    "ks5",
    # the two-SM cluster kernel (k_ks6) for every narrow trace / combine (the default hands the narrowest ones to k_ks8)
    "ks6",
    # one key-switch chain per cluster of eight (or, beyond one wave of those, four) SMs, contributions exchanged
    # through L2 (k_ks8), for every trace / combine launch
    "ks8",
    # the four-SM cluster variant of k_ks8 (two output polynomials per CTA) for every trace / combine launch
    "ks8c4",
    # one-SM-per-ciphertext external product (k_ext8) for the narrow launches too (the default hands them to k_ext9)
    "ext8",
    # one external-product chain per cluster of eight / four SMs (k_ext9) for every launch
    "ext9",
    "ext9c4",
)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_kernel_variant_is_bit_exact(built, name):
    env = dict(os.environ)
    env["FHERAM_KERNEL"] = name
    r = subprocess.run([sys.executable, "-m", "pytest", str(ROOT / "tests" / "test_gpu_parity.py"), "-m", "gpu",
                        "-x", "-q", "-k", SELECT], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"FHERAM_KERNEL={name}:\n{r.stdout[-3000:]}\n{r.stderr[-1000:]}"
    assert " passed" in r.stdout


@pytest.mark.parametrize("spec", ["bogus", "ks5,ks6", "ext8,ext9", "ks6,"])
def test_unknown_kernel_name_fails_context_creation(built, monkeypatch, spec):
    """FHERAM_KERNEL is read by every context creation: an unknown name, or two of one class, is an error that lists
    the valid names (checked before the device, so this runs anywhere)."""
    import fhe_ram_b200 as fr
    monkeypatch.setenv("FHERAM_KERNEL", spec)
    with pytest.raises(fr.FheRamError) as e:
        fr.Parameters.new().module()
    assert e.value.code == -1, str(e.value)
    assert f"FHERAM_KERNEL={spec}" in str(e.value) and "ext9c4" in str(e.value) and "ks8c4" in str(e.value)
