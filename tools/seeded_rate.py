"""What seeded addresses and a seeded RAM buy at the host boundary (DESIGN.md 3.6, 5.2).

1. End to end from host buffers: a batch of --batch reads at 2^18 x 4 B (README parameters) through
   fheram_ram_read_batch_host_p17 (addresses as packed 17-bit limbs) and fheram_ram_read_batch_host_seeded (packed
   bodies + one seed per address), the two arms alternating step by step; host clock around each call (the call ends
   in a device synchronise), medians of --steps steps after --warmup, and the host -> device bytes of one step.  Both
   host buffers are pinned (fheram_host_register).  The addresses are --distinct seeded addresses encrypted on the
   CPU, repeated to fill the batch; the _p17 arm gets their expanded limbs, so both arms compute the same results,
   which are compared.
2. Device time of k_glwe_expand per address (and of k_unpack17, what the _p17 path runs in its place), from
   torch.profiler over one step of each arm, run after the timed steps.
3. fheram_ram_load against fheram_ram_load_seeded of a 2^22 x 4 B RAM from pageable host memory (host clock, medians
   of --reps alternating calls); the seeded load is checked limb for limb against the plain one.

Multi-GPU (torchrun --nproc-per-node G): the RAM is sharded over the G ranks, every rank passes its share of the batch
(fheram.h: the contract of the _p17 call), a step is timed from a barrier to the slowest rank; parts 2 and 3 run on
one GPU only.  The multi-GPU path has not been run yet.

  python tools/seeded_rate.py > profiles/seeded_rate.json
  torchrun --nproc-per-node 8 tools/seeded_rate.py > profiles/seeded_rate_8gpu.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader",
                        "-i", str(index)], capture_output=True, text=True, check=True).stdout.strip()
    name, power, max_clock, clock = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": max_clock, "sm_clock_at_start": clock}


def stats(ts):
    return {"median_ms": 1e3 * statistics.median(ts), "min_ms": 1e3 * min(ts), "max_ms": 1e3 * max(ts), "steps": len(ts)}


def seeded_addresses(fr, api, p, sk, distinct, batch):
    """--distinct seeded addresses (CPU), repeated to `batch`: their packed expanded limbs (the _p17 arm), packed
    bodies and seeds (the seeded arm) and the address values, [batch] each"""
    xa, xe = fr.Source(21), fr.Source(22)
    values = np.array([(104729 * i + 17) % p.max_addr() for i in range(distinct)])
    enc = [fr.Address.encrypt_sk_seeded(p, int(v), sk, xa, xe) for v in values]
    bodies = np.stack([b for b, _ in enc])
    seeds = np.concatenate([s for _, s in enc])
    p17 = api.pack17(fr.Address.expand(p, bodies, seeds, distinct).data).reshape(distinct, -1)
    s17 = api.pack17(bodies).reshape(distinct, -1)
    pick = np.arange(batch) % distinct
    return p17[pick], s17[pick], seeds[pick], values[pick]


def batch_rates(fr, api, p, ram, keys, p17, s17, seeds, values, plain, a, dist=None):
    """part 1 on this rank's share; returns the timings and the arms' buffers"""
    n = p17.shape[0]
    p17, s17, seeds = (np.ascontiguousarray(x) for x in (p17, s17, seeds))
    for buf in (p17, s17):
        api.host_register(buf)
    out_a = np.zeros((n, p.word_size(), p.glwe_len()), dtype=np.int32)
    out_b = np.zeros_like(out_a)
    api.host_register(out_a); api.host_register(out_b)
    arms = {"p17": lambda: ram.read_batch_host_p17(p17, n, keys, out_a),
            "seeded": lambda: ram.read_batch_host_seeded(s17, seeds, n, keys, out_b)}
    ts = {k: [] for k in arms}
    for step in range(a.warmup + a.steps):
        for k, fn in arms.items():
            if dist is not None:
                dist.barrier()
            t0 = time.perf_counter()
            fn()
            dt = time.perf_counter() - t0
            if dist is not None:
                import torch
                t = torch.tensor([dt], dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t[0])
            if step >= a.warmup:
                ts[k].append(dt)
    assert np.array_equal(out_a, out_b), "the two arms computed different results"
    if dist is None:
        vals, _ = fr.decrypt_words_device(p, ram.read_batch_device(fr.Address.from_limbs(
            p, api.unpack17(p17[:8], 8 * p17.shape[1] * 32 // 17), 8), keys), 8 * p.word_size(), fr.GLWESecret(p, a.sk))
        assert np.array_equal(vals, plain[values[:8]].reshape(-1)), "seeded reads do not decrypt to the RAM's bytes"
    return ts, (p17, s17, out_a, out_b)


def profile_kernels(p, ram, keys, n, arms):
    """device time per address of the kernels that turn uploaded bytes into raw limbs, one step per arm"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for name, fn in arms.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        for e in prof.key_averages():
            if "k_glwe_expand" in e.key or "k_unpack17" in e.key:
                us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                out[f"{name}:{'k_glwe_expand' if 'expand' in e.key else 'k_unpack17'}"] = {
                    "launches": e.count, "total_ms": us / 1e3, "us_per_address": us / n}
    return out


def ram_loads(fr, reps):
    p = fr.Parameters.readme(max_addr=1 << 22, word_size=4)
    sk = fr.GLWESecret.fill_ternary_prob(p, 0.5, fr.Source(7))
    data = fr.Source(5).fill_bytes(p.max_addr() * p.word_size())
    xa = fr.Source(61)
    seed = xa.seed()
    ram = fr.Ram.new(p)
    ram.encrypt_sk_gpu(data, sk, xa, fr.Source(62))
    cts = ram.store()
    S, n = -(-p.k_glwe_ct() // p.basek()), p.n()
    bodies = np.ascontiguousarray(cts.reshape(-1, S, 2, n)[:, :, 0, :]).reshape(-1)
    ts = {"ram_load": [], "ram_load_seeded": []}
    for r in range(reps + 1):
        for k, fn in (("ram_load", lambda: ram.load(cts)), ("ram_load_seeded", lambda: ram.load_seeded(bodies, seed))):
            t0 = time.perf_counter()
            fn()
            p.synchronize()
            if r:
                ts[k].append(time.perf_counter() - t0)
    assert np.array_equal(ram.store(), cts), "ram_load_seeded != ram_load"
    res = {"max_addr": p.max_addr(), "word_size": p.word_size(), "host_memory": "pageable",
           "ram_load": {**stats(ts["ram_load"]), "bytes": int(cts.nbytes)},
           "ram_load_seeded": {**stats(ts["ram_load_seeded"]), "bytes": int(bodies.nbytes) + 40}}
    res["speedup"] = res["ram_load"]["median_ms"] / res["ram_load_seeded"]["median_ms"]
    ram.close(); p.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--distinct", type=int, default=64)
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import fhe_ram_b200 as fr
    from fhe_ram_b200 import api
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(rank)
        dist.init_process_group("gloo")
    p = fr.Parameters.readme(device=rank, word_size=4)
    sk = fr.GLWESecret.fill_ternary_prob(p, 0.5, fr.Source(7))
    a.sk = sk.data
    data = fr.Source(5).fill_bytes(p.max_addr() * p.word_size())
    plain = data.view(np.int8).reshape(-1, p.word_size())
    keys = fr.EvaluationKeysPrepared.encrypt_sk_gpu(p, sk, fr.Source(3), fr.Source(4))
    if world > 1:
        from fhe_ram_b200.sharded import ShardedRamLib
        ram = ShardedRamLib(p, rank, world).ram
    else:
        ram = fr.Ram.new(p)
    ram.encrypt_sk_gpu(data, sk, fr.Source(11), fr.Source(12))
    p17, s17, seeds, values = seeded_addresses(fr, api, p, sk, a.distinct, a.batch)
    mine = slice(rank * (a.batch // world), (rank + 1) * (a.batch // world))
    ts, bufs = batch_rates(fr, api, p, ram, keys, p17[mine], s17[mine], seeds[mine], values[mine], plain, a, dist)
    del p17, s17
    per_addr = p.n_ggsw() * p.ggsw_len()
    out = {"tool": "tools/seeded_rate.py", **gpu_info(rank), "gpus": world, "batch": a.batch,
           "distinct_addresses": a.distinct, "max_addr": p.max_addr(), "word_size": p.word_size(), "arms": {}}
    for k, host_bytes in (("p17", per_addr * 17 // 8), ("seeded", per_addr // 2 * 17 // 8 + 40)):
        s = stats(ts[k])
        s["reads_per_s"] = a.batch / (s["median_ms"] * 1e-3)
        s["h2d_bytes_per_step"] = a.batch * host_bytes
        out["arms"][k] = s
    out["seeded_over_p17_rate"] = out["arms"]["seeded"]["reads_per_s"] / out["arms"]["p17"]["reads_per_s"]
    if world == 1:
        p17, s17, out_a, out_b = bufs
        seeds = np.ascontiguousarray(seeds)
        n = a.batch
        out["kernels"] = profile_kernels(p, ram, keys, n, {
            "p17": lambda: ram.read_batch_host_p17(p17, n, keys, out_a),
            "seeded": lambda: ram.read_batch_host_seeded(s17, seeds, n, keys, out_b)})
        for buf in bufs:
            api.host_unregister(buf)
        out["ram_load_2^22x4"] = ram_loads(fr, a.reps)
    else:
        for buf in bufs:
            api.host_unregister(buf)
    if rank == 0:
        print(json.dumps(out, indent=1))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
