"""Per-kernel machine-code comparison of the library against a git revision (default HEAD), without a GPU.

Both trees are compiled to an sm_100a cubin with the flags of __graft_entry__.py plus -cubin -Xptxas -v.  For every
__global__ function the SASS of `cuobjdump -sass` is reduced to its instruction text and branch targets (addresses and
encodings dropped) and compared, together with the function's ptxas lines (registers, barriers, stack, spills, shared
memory).  A refactor that must not change the generated code prints "same" for every entry point.

    python tools/sass_compare.py [--rev REV] [--out DIR]

Exit code 0 when every function is the same, 1 otherwise; the per-function report is printed and written to
DIR/sass_compare.txt (DIR defaults to a temporary directory).
"""
from __future__ import annotations

import argparse
import hashlib
import re
import subprocess
import sys
import tarfile
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from __graft_entry__ import NVCC_FLAGS  # noqa: E402

CUDA = Path("/usr/local/cuda/bin")


def build(tree: Path, out: Path) -> tuple[dict, dict]:
    """cubin of tree's library -> ({function: sass digest}, {function: [ptxas lines]})"""
    out.mkdir(parents=True, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f not in ("-shared", "-Xcompiler", "-fPIC")]
    cubin = out / "lib.cubin"
    ptx = subprocess.run([str(CUDA / "nvcc"), *flags, "-ccbin", "/usr/bin/g++", "-cubin", "-Xptxas", "-v",
                          "-o", str(cubin), str(tree / "fhe_ram_b200" / "csrc" / "fheram_cuda.cu")],
                         capture_output=True, text=True, check=True).stderr
    sass = subprocess.run([str(CUDA / "cuobjdump"), "-sass", str(cubin)], capture_output=True, text=True,
                          check=True).stdout
    funcs, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if cur and m:
            funcs[cur].append(re.sub(r"\s+", " ", m.group(1)).strip())
    digests = {f: hashlib.sha1("\n".join(v).encode()).hexdigest()[:12] for f, v in funcs.items()}
    props, cur = {}, None
    for line in ptx.splitlines():
        m = re.search(r"(?:Compiling entry function|Function properties for) '?([^' ]+)'?", line)
        if m:
            cur = m.group(1)
            props.setdefault(cur, [])
        elif cur and ("stack frame" in line or "Used" in line):
            props[cur].append(line.split(":", 1)[-1].strip() if "Used" in line else line.strip())
    return digests, props


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rev", default="HEAD", help="git revision to compare against (default HEAD)")
    ap.add_argument("--out", type=Path, default=None, help="directory for the cubins and the report")
    args = ap.parse_args()
    out = args.out or Path(tempfile.mkdtemp(prefix="sass_compare_"))
    ref = out / "ref_tree"
    ref.mkdir(parents=True, exist_ok=True)
    archive = subprocess.run(["git", "-C", str(ROOT), "archive", args.rev, "fhe_ram_b200/csrc", "include"],
                             capture_output=True, check=True).stdout
    (out / "ref.tar").write_bytes(archive)
    with tarfile.open(out / "ref.tar") as t:
        t.extractall(ref)
    old_s, old_p = build(ref, out / "ref")
    new_s, new_p = build(ROOT, out / "new")
    lines, differing = [], 0
    for f in sorted(set(old_s) | set(new_s)):
        same = old_s.get(f) == new_s.get(f) and old_p.get(f) == new_p.get(f)
        differing += not same
        lines.append(f"{'same' if same else 'DIFF'} {f}  sass {old_s.get(f)} -> {new_s.get(f)}  ptxas {new_p.get(f)}")
        if old_p.get(f) != new_p.get(f):
            lines.append(f"    ptxas was {old_p.get(f)}")
    lines.append(f"{differing} of {len(set(old_s) | set(new_s))} functions differ from {args.rev}")
    report = "\n".join(lines) + "\n"
    (out / "sass_compare.txt").write_text(report)
    print(report, end="")
    return 1 if differing else 0


if __name__ == "__main__":
    sys.exit(main())
