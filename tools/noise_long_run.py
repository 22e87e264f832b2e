"""Long-run noise growth of the RAM under read_prepare_write / write cycles at the README parameter set (2^18 x 4 B,
k_pt = 9), against README.md:36 ("at least ~40 mio read/write without having to refresh the RAM").

Every cycle writes a random word at a random address (addresses encrypted on the device, fheram_address_encrypt_sk);
every `--sample-every` cycles a batch of 64 probe addresses that are never written is read and the decryption error of
every probe byte is recorded.  A write re-injects coefficient h of the packed polynomial into EVERY RAM polynomial
(src/ram.rs:612-630), so untouched words collect fresh key-switch noise at every cycle: the error variance grows
linearly, var(c) = var_0 + c * var_w.  The script fits var_w and extrapolates the number of cycles after which the error
standard deviation reaches 1/8 of the rounding margin 2^-(k_pt+1) (failure probability ~ 10^-15 per decryption).

At every sample point the whole RAM is also decrypted on the device (fheram_ram_decrypt_sk): every cell must equal the
model, written cells included, and the rms / max of the exact error (as a fraction of the torus) is recorded separately
for written and never-written cells, with the same fit on the never-written cells of the whole RAM.

  gpurun --timeout 900 -- python tools/noise_long_run.py --cycles 20000 > gpurun_out/noise_long_run.json
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import __graft_entry__ as g


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cycles", type=int, default=20000)
    ap.add_argument("--sample-every", type=int, default=1000)
    ap.add_argument("--max-addr-log2", type=int, default=18)
    ap.add_argument("--word-size", type=int, default=4)
    a = ap.parse_args()
    g.build()
    import fhe_ram_b200 as fr
    k_pt, ws = 9, a.word_size
    p = fr.Parameters.readme(max_addr=1 << a.max_addr_log2, word_size=ws, k_pt=k_pt)
    sk, evk = fr.gen_keys(p)
    keys = fr.EvaluationKeysPrepared.alloc(p).prepare(evk)
    data = fr.Source(5).fill_bytes(p.max_addr() * ws)
    ram = fr.Ram.new(p)
    ram.encrypt_sk_gpu(data, sk, fr.Source(11), fr.Source(12))
    rng = np.random.default_rng(7)
    n_probe = 64
    probes = rng.choice(p.max_addr(), size=n_probe, replace=False)
    probe_set = set(int(x) for x in probes)
    a_probe = fr.Address.encrypt_sk_gpu(p, probes.astype(np.uint32), sk, [fr.Source(100 + i) for i in range(n_probe)],
                                        [fr.Source(300 + i) for i in range(n_probe)])
    xa, xe = fr.Source(21), fr.Source(22)
    written = np.zeros(p.max_addr(), dtype=bool)
    values = np.zeros((p.max_addr(), ws), dtype=np.int16)
    err = np.zeros((p.max_addr(), ws), dtype=np.int64)

    def whole_ram():
        ram.decrypt_sk(sk, values, err)
        model = data.view(np.int8).reshape(-1, ws)  # cast_u8_to_signed(b, 8) of every byte
        bad = int(np.count_nonzero(values != model))
        assert bad == 0, ("decrypted RAM differs from the model in", bad, "cells")
        e = err.astype(np.float64) * 2.0 ** -p.k_glwe_ct()
        row = {}
        for name, sel in (("written", written), ("never_written", ~written)):
            x = e[sel]
            if x.size:
                row[f"ram_{name}_cells"] = int(x.size)
                row[f"ram_{name}_rms_log2"] = float(0.5 * np.log2(np.mean(x * x)))
                row[f"ram_{name}_max_log2"] = float(np.log2(np.abs(x).max()))
        return row

    def sample():
        got = ram.read_batch(a_probe, keys)
        errs = []
        for b, idx in enumerate(probes):
            for i in range(ws):
                want = fr.cast_u8_to_signed(int(data[int(idx) * ws + i]), 8)
                v, noise = fr.decrypt_glwe(p, got[b, i], want, sk)
                assert v == want, ("probe word corrupted", int(idx), i, v, want)
                errs.append(2.0 ** noise)          # |error| as a fraction of the torus
        e = np.array(errs)
        return float(np.sqrt(np.mean(e * e))), float(e.max())

    rows = []
    t0 = time.time()
    rms, mx = sample()
    rows.append({"cycle": 0, "rms_log2": float(np.log2(rms)), "max_log2": float(np.log2(mx)), **whole_ram()})
    for c in range(1, a.cycles + 1):
        idx = int(rng.integers(0, p.max_addr()))
        while idx in probe_set:
            idx = int(rng.integers(0, p.max_addr()))
        addr = fr.Address.encrypt_sk_gpu(p, np.array([idx], dtype=np.uint32), sk, xa, xe)
        ram.read_prepare_write(addr, keys)
        val = rng.integers(0, 128, size=ws)
        ram.write(np.stack([fr.encrypt_glwe(p, int(v), sk) for v in val]), addr, keys)
        data[idx * ws:(idx + 1) * ws] = val
        written[idx] = True
        addr.close()
        if c % a.sample_every == 0:
            rms, mx = sample()
            rows.append({"cycle": c, "rms_log2": float(np.log2(rms)), "max_log2": float(np.log2(mx)), **whole_ram()})
            r = rows[-1]
            print(f"cycle {c}: rms 2^{np.log2(rms):.2f} max 2^{np.log2(mx):.2f}; whole RAM never written rms "
                  f"2^{r['ram_never_written_rms_log2']:.2f} max 2^{r['ram_never_written_max_log2']:.2f}, written max "
                  f"2^{r.get('ram_written_max_log2', float('nan')):.2f} ({time.time() - t0:.0f} s)", file=sys.stderr)
    margin = 2.0 ** -(k_pt + 1)
    target_var = (margin / 8.0) ** 2

    def fit(key):  # linear fit of the variance
        cs = np.array([r["cycle"] for r in rows], dtype=float)
        var = np.array([4.0 ** r[key] for r in rows])
        A = np.vstack([np.ones_like(cs), cs]).T
        (v0, vw), *_ = np.linalg.lstsq(A, var, rcond=None)
        return v0, vw, (target_var - v0) / vw if vw > 0 else float("inf")

    v0, vw, cycles_to_refresh = fit("rms_log2")
    rv0, rvw, ram_cycles = fit("ram_never_written_rms_log2")
    last = rows[-1]
    out = {"parameters": {"max_addr_log2": a.max_addr_log2, "word_size": ws, "k_pt": k_pt}, "cycles": a.cycles,
           "probes": n_probe * ws, "samples": rows,
           "fit": {"var0_log2": float(np.log2(max(v0, 1e-300))), "var_per_cycle_log2": float(np.log2(max(vw, 1e-300))),
                   "std_after_fit_cycles_log2": float(0.5 * np.log2(v0 + vw * a.cycles))},
           "margin_log2": -(k_pt + 1),
           "cycles_until_std_is_margin_over_8": float(cycles_to_refresh),
           "readme_claim": "at least ~40 mio read/write without refresh (README.md:36)",
           "whole_ram": {"cells": p.max_addr() * ws, "written_words_at_end": int(written.sum()),
                         "fit_never_written": {"var0_log2": float(np.log2(max(rv0, 1e-300))),
                                               "var_per_cycle_log2": float(np.log2(max(rvw, 1e-300)))},
                         "cycles_until_std_is_margin_over_8": float(ram_cycles),
                         "max_log2_at_end_all_cells": max(last.get("ram_written_max_log2", -np.inf),
                                                          last["ram_never_written_max_log2"])},
           **gpu_info(),
           "seconds": time.time() - t0}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
