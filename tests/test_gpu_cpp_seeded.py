"""-m gpu: the seeded calls of the C++ host layer (fhe_ram_b200/cpp/fheram.hpp) through tests/cpp_seeded.cpp: one
Address object reused with seeded and full encryptions in turn must read the address it was last encrypted with,
and a seeded RAM and a batch of seeded addresses from host buffers must decrypt to the stored bytes.  The program is
compiled into the test's temporary directory."""
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.gpu
def test_cpp_seeded_calls(built, tmp_path):
    exe = tmp_path / "cpp_seeded"
    pkg = ROOT / "fhe_ram_b200"
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-I", str(ROOT / "include"), "-I", str(pkg / "cpp"),
                           str(ROOT / "tests" / "cpp_seeded.cpp"), "-o", str(exe), "-L", str(pkg), "-lfheram_cuda",
                           f"-Wl,-rpath,{pkg}"])
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr
