"""Rates of the decryption entry points (DESIGN.md 3.7).  Every call is timed with a host clock around the call and a
device synchronise, after two warm-up calls; the median of --reps calls is reported.

  whole RAM on the device (fheram_ram_decrypt_sk) at 2^18 x 4 B and 2^22 x 4 B, download of values and errors included
  whole RAM on the CPU (fheram_decrypt_ram, all host threads) at 2^18 x 4 B
  fheram_decrypt_words_device on the result arena of a 1 024-read batch (4 096 GLWEs), and that batched read itself
  a loop of fheram_decrypt_word over the same 4 096 words (CPU, one thread)

  python tools/decrypt_rate.py > profiles/decrypt_rate.json
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
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
    return {"median_ms": 1e3 * statistics.median(ts), "min_ms": 1e3 * min(ts), "max_ms": 1e3 * max(ts), "calls": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--word-reps", type=int, default=5)
    a = ap.parse_args()
    import fhe_ram_b200 as fr
    from fhe_ram_b200 import api
    out = {"tool": "tools/decrypt_rate.py", **gpu_info(), "host_threads": os.cpu_count(), "reps": a.reps}

    for log2 in (18, 22):
        p = fr.Parameters.readme(max_addr=1 << log2, word_size=4)
        sk = fr.GLWESecret.fill_ternary_prob(p, 0.5, fr.Source(7))
        data = fr.Source(5).fill_bytes(p.max_addr() * 4)
        ram = fr.Ram.new(p)
        ram.encrypt_sk_gpu(data, sk, fr.Source(21), fr.Source(22))
        values = np.zeros((p.max_addr(), 4), dtype=np.int16)
        err = np.zeros((p.max_addr(), 4), dtype=np.int64)
        r = timed(lambda: ram.decrypt_sk(sk, values, err), p.synchronize, a.reps)
        r["bytes_decrypted"] = p.max_addr() * 4
        r["glwe"] = 4 * p.n_glwe()
        r["bytes_per_s"] = r["bytes_decrypted"] / (r["median_ms"] * 1e-3)
        out[f"ram_decrypt_sk_2^{log2}x4"] = r
        plain = data.view(np.int8).reshape(-1, 4)
        assert np.array_equal(values, plain)
        if log2 == 18:
            cts = ram.store()
            r = timed(lambda: fr.decrypt_ram(p, cts, sk), lambda: None, a.word_reps, warm=1)
            r["bytes_decrypted"] = p.max_addr() * 4
            r["bytes_per_s"] = r["bytes_decrypted"] / (r["median_ms"] * 1e-3)
            out["decrypt_ram_cpu_2^18x4"] = r
            assert np.array_equal(fr.decrypt_ram(p, cts, sk)[0], plain)

            keys = fr.EvaluationKeysPrepared.encrypt_sk_gpu(p, sk, fr.Source(3), fr.Source(4))
            idxs = np.random.default_rng(1).integers(0, p.max_addr(), size=1024).astype(np.uint32)
            addrs = fr.Address.encrypt_sk_gpu(p, idxs, sk, fr.Source(41), fr.Source(42))
            out["read_batch_device_1024"] = timed(lambda: ram.read_batch_device(addrs, keys), p.synchronize, a.reps)
            d = ram.read_batch_device(addrs, keys)
            n = 1024 * 4
            r = timed(lambda: fr.decrypt_words_device(p, d, n, sk), p.synchronize, a.reps)
            r["words"] = n
            out["decrypt_words_device_4096"] = r
            vals, _ = fr.decrypt_words_device(p, d, n, sk)
            assert np.array_equal(vals, plain[idxs].reshape(-1))
            limbs = np.zeros(n * p.glwe_len(), dtype=np.int64)
            api._check(api.lib().fheram_download_glwe(p.module(), C.c_void_p(d), n, api._p(limbs)))
            limbs = limbs.reshape(n, -1)

            def word_loop():
                for j in range(n):
                    fr.decrypt_glwe(p, limbs[j], 0, sk)
            r = timed(word_loop, lambda: None, a.word_reps, warm=1)
            r["words"] = n
            out["decrypt_word_loop_cpu_4096"] = r
            addrs.close(); keys.close()
        ram.close()
        p.close()
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
