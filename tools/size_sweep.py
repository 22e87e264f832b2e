"""Cost of a RAM size whose polynomial count is not a power of two (DESIGN.md §1, the mixed packer level), against
the powers of two around it: max_addr = 2^17, 3 * 2^16 and 2^18 entries of 4 bytes, README parameters (k_pt = 9).

Per size: single read, read_prepare_write and write (host clock around the call and a device synchronise, median of
--reps calls after two warm-up calls; every write follows its read_prepare_write), and the rate of a device-resident
batch of --batch reads (fheram_ram_read_batch_device).  Read results are decoded on the device and checked against the
plaintext.  The card's name and power limit are read in the same run.

  python tools/size_sweep.py > profiles/size_sweep.json
"""
import argparse
import json
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


def median_ms(ts):
    return {"median_ms": 1e3 * statistics.median(ts), "min_ms": 1e3 * min(ts), "max_ms": 1e3 * max(ts), "calls": len(ts)}


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
    return median_ms(ts)


def run_size(fr, max_addr, batch, reps):
    ws = 4
    p = fr.Parameters.readme(max_addr=max_addr, word_size=ws)
    sk = fr.GLWESecret.fill_ternary_prob(p, 0.5, fr.Source(7))
    data = fr.Source(5).fill_bytes(max_addr * ws)
    plain = data.view(np.int8).reshape(-1, ws)
    keys = fr.EvaluationKeysPrepared.encrypt_sk_gpu(p, sk, fr.Source(3), fr.Source(4))
    ram = fr.Ram.new(p)
    ram.encrypt_sk_gpu(data, sk, fr.Source(21), fr.Source(22))
    rng = np.random.default_rng(max_addr)
    one = fr.Address.encrypt_sk_gpu(p, np.array([max_addr - 3], dtype=np.uint32), sk, fr.Source(31), fr.Source(32))
    out = {"max_addr": max_addr, "word_size": ws, "n_glwe": p.n_glwe()}

    out["read"] = timed(lambda: ram.read(one, keys), p.synchronize, reps)
    got = ram.read(one, keys)
    for i in range(ws):
        v, _ = fr.decrypt_glwe(p, got[i], int(plain[max_addr - 3, i]), sk)
        assert v == plain[max_addr - 3, i], (max_addr, i, v)

    words = np.stack([fr.encrypt_glwe(p, int(v), sk) for v in plain[max_addr - 3].view(np.uint8)])
    t_rpw, t_write = [], []
    for r in range(reps + 2):
        t0 = time.perf_counter()
        ram.read_prepare_write(one, keys)
        p.synchronize()
        t1 = time.perf_counter()
        ram.write(words, one, keys)   # writes back the word it holds: the plaintext stays as it was
        p.synchronize()
        t2 = time.perf_counter()
        if r >= 2:
            t_rpw.append(t1 - t0)
            t_write.append(t2 - t1)
    out["read_prepare_write"] = median_ms(t_rpw)
    out["write"] = median_ms(t_write)

    idxs = rng.integers(0, max_addr, size=batch).astype(np.uint32)
    addrs = fr.Address.encrypt_sk_gpu(p, idxs, sk, fr.Source(41), fr.Source(42))
    r = timed(lambda: ram.read_batch_device(addrs, keys), p.synchronize, reps)
    r["batch"] = batch
    r["reads_per_s"] = batch / (r["median_ms"] * 1e-3)
    out["read_batch_device"] = r
    d = ram.read_batch_device(addrs, keys)
    vals, _ = fr.decrypt_words_device(p, d, batch * ws, sk)
    assert np.array_equal(vals, plain[idxs].reshape(-1)), max_addr
    addrs.close(); one.close(); ram.close(); keys.close(); p.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--batch", type=int, default=1024)
    a = ap.parse_args()
    import fhe_ram_b200 as fr
    out = {"tool": "tools/size_sweep.py", **gpu_info(), "reps": a.reps, "sizes": []}
    for max_addr in (1 << 17, 3 << 16, 1 << 18):
        out["sizes"].append(run_size(fr, max_addr, a.batch, a.reps))
    by = {s["max_addr"]: s for s in out["sizes"]}
    mid, top = by[3 << 16], by[1 << 18]
    out["ratio_3x2^16_over_2^18"] = {
        "read": mid["read"]["median_ms"] / top["read"]["median_ms"],
        "read_prepare_write": mid["read_prepare_write"]["median_ms"] / top["read_prepare_write"]["median_ms"],
        "write": mid["write"]["median_ms"] / top["write"]["median_ms"],
        "batch_time": top["read_batch_device"]["reads_per_s"] / mid["read_batch_device"]["reads_per_s"],
    }
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
