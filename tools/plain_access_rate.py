"""Rates of the plaintext-address calls (DESIGN.md 3.8) against the oblivious ones, at 2^18 x 4 B (k_pt = 9) on one GPU.
Every step is timed with a host clock around the call and a device synchronise, after two warm-up steps; the median
of --reps steps is reported.  The GPU name and power limit are read in the same run.

  1 024 addresses: fheram_ram_read_plain_device against fheram_ram_read_batch_device, in reads/s
  one address:     fheram_ram_read_plain against fheram_ram_read (host results), in ms
  one word:        fheram_ram_write_plain against fheram_ram_read_prepare_write + fheram_ram_write, in ms

  python tools/plain_access_rate.py [--out profiles/plain_access_rate.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, sync, reps, warm=2):
    for _ in range(warm):
        fn()
    sync()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        sync()
        ts.append(time.perf_counter() - t0)
    return {"median_ms": 1e3 * statistics.median(ts), "min_ms": 1e3 * min(ts), "max_ms": 1e3 * max(ts), "steps": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--reads", type=int, default=1024)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "plain_access_rate.json"))
    a = ap.parse_args()
    import fhe_ram_b200 as fr
    out = {"tool": "tools/plain_access_rate.py", **gpu_info(), "reps": a.reps, "max_addr": 1 << 18, "word_size": 4,
           "k_pt": 9}
    p = fr.Parameters.readme(max_addr=1 << 18, word_size=4)
    ws = p.word_size()
    sk = fr.GLWESecret.fill_ternary_prob(p, 0.5, fr.Source(7))
    data = fr.Source(5).fill_bytes(p.max_addr() * ws)
    plain = data.view(np.int8).reshape(-1, ws)
    keys = fr.EvaluationKeysPrepared.encrypt_sk_gpu(p, sk, fr.Source(3), fr.Source(4))
    ram = fr.Ram.new(p)
    ram.encrypt_sk_gpu(data, sk, fr.Source(21), fr.Source(22))
    sync = p.synchronize

    # batches of reads, results left on the device
    idxs = np.random.default_rng(1).integers(0, p.max_addr(), size=a.reads).astype(np.uint32)
    addrs = fr.Address.encrypt_sk_gpu(p, idxs, sk, fr.Source(41), fr.Source(42))
    n = a.reads
    for name, fn in (("read_plain_device", lambda: ram.read_plain_device(idxs, keys)),
                     ("read_batch_device", lambda: ram.read_batch_device(addrs, keys))):
        r = timed(fn, sync, a.reps)
        r["reads"] = n
        r["reads_per_s"] = n / (r["median_ms"] * 1e-3)
        values, _ = fr.decrypt_words_device(p, fn(), n * ws, sk)
        assert np.array_equal(values.reshape(n, ws), plain[idxs]), name
        out[f"{name}_{n}"] = r
    out["batch_speedup"] = out[f"read_plain_device_{n}"]["reads_per_s"] / out[f"read_batch_device_{n}"]["reads_per_s"]

    # one read, results on the host
    i0 = int(idxs[0])
    addr = fr.Address.alloc(p).encrypt_sk(p, i0, sk, fr.Source(43), fr.Source(44))
    out["read_plain_1"] = timed(lambda: ram.read_plain([i0], keys), sync, a.reps)
    out["read_1"] = timed(lambda: ram.read(addr, keys), sync, a.reps)
    out["read_speedup"] = out["read_1"]["median_ms"] / out["read_plain_1"]["median_ms"]

    # one write (the same word again each step)
    new = [1, 2, 3, 4]
    w = np.stack([fr.encrypt_glwe(p, v, sk) for v in new])

    def pair():
        ram.read_prepare_write(addr, keys)
        ram.write(w, addr, keys)
    out["write_plain_1"] = timed(lambda: ram.write_plain(i0, w, keys), sync, a.reps)
    out["rpw_write_pair_1"] = timed(pair, sync, a.reps)
    out["write_speedup"] = out["rpw_write_pair_1"]["median_ms"] / out["write_plain_1"]["median_ms"]
    values, _ = ram.decrypt_sk(sk)
    want = plain.copy()
    want[i0] = new
    assert np.array_equal(values, want)

    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(out, indent=1) + "\n")
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
