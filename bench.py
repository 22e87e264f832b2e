#!/usr/bin/env python
"""bench.py -- FHE-RAM hot-path benchmark (BASELINE.json metric: batched reads/s at 2^18 x 4 B,
plus single read / read_prepare_write / write latency).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

A "step" is one batch of B independent encrypted-address reads (BASELINE.json config 3, B = 1024)
against a RAM of max_addr = 2^18 words x 4 bytes (README.md:17-34 parameters).  `value` is measured
with keys, RAM and prepared addresses resident in HBM; `e2e` runs the same batch through the C ABI
with HOST buffers (address upload + on-device prepare + read + result download in the timed
region; host limb format --host-format i32 (default: the compact format of the C ABI) or i64).  N > 1: the RAM
is sharded by polynomial index mod N (SURVEY.md 8e), one process per GPU, every exchange step inside
libfheram_cuda.so on its own NCCL communicator; the global batch stays B ("strong" scaling, also the label at N = 1).
--impl reference times the CPU restatement of the reference's FFT64 path (oracle/, kind "port": the reference
itself cannot be built here -- no Rust toolchain, Poulpy un-vendored) on inputs made by the oracle's own client side;
that arm imports nothing of fhe_ram_b200.
The GPU arm runs from the tree as __graft_entry__.build() left it and writes nothing there.  --dump-outputs DIR writes
what the last timed step computed (see dump_outputs) so that two builds can be compared output for output: every input
comes from fixed seeds, so the same arguments give the same inputs on every run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# algorithmic work per operation (SURVEY.md 8d / BASELINE.md 4)
F_EXT = 2_363_392   # flop per external product (6 fwd + 8 inv FFT of 2048 pts, 6x8 contraction)
F_KS = 1_632_256    # flop per key-switch automorphism (3 + 8 FFT, 3x8 contraction)
B_EXT = 1.5 * 2**20 + 2 * 96 * 2**10   # bytes per ext product: prepared GGSW + ct in + ct out (int32)
B_KS = 0.75 * 2**20                    # bytes per key-switch: prepared key (ct stays in shared memory)
DUMP_BYTES = 48 << 20                  # --dump-outputs budget: a whole batch at 2^18 x 4 B is 805 MB of float64


def op_model(max_addr, word_size, base2d, n=4096):
    """(ext, ks) per read (src/ram.rs:382-459) and per write (:226-294, GGSW inversions excluded)."""
    g = max(1, max_addr // n)
    d0 = len(base2d[0])
    d1 = len(base2d[1]) if len(base2d) > 1 else 0
    lg = (g - 1).bit_length() if g > 1 else 0
    pack = 0 if g == 1 else g * (12 - lg) + (g - 1)
    read = (word_size * (g * d0 + d1), word_size * (pack + 12))
    write = (word_size * (g * d0 + d1), word_size * (12 + (2 * g * 12 if g > 1 else 0)))
    return read, write


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None   # timed window (time.time()); rows carry their arrival time

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index),
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            self.proc.wait()
        # samples taken inside the timed window; a window shorter than the sampling period falls back to
        # the samples of the warm-up + timed span (same kernels, same load) and says so
        window = "timed region"
        rows = [r for t, r in self.rows if self.t0 is None or (self.t0 - 0.05 <= t <= (self.t1 or t) + 0.05)]
        if not rows:
            rows, window = [r for _, r in self.rows], "warm-up + timed region (timed region shorter than the sampling period)"
        self.rows = rows
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for i, nm in enumerate(names):
                if len(r) > 3 + i and r[3 + i].lower().startswith("active"):
                    reasons.add(nm)
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


def make_addresses(fr, params, sk, idxs, threads, first=0):
    """Address::encrypt_sk (client side, CPU) for every index, on `threads` host threads; address j of the batch
    draws from Source(1000 + first + j) / Source(5000 + first + j)."""
    out = np.zeros((len(idxs), params.n_ggsw() * params.ggsw_len()), dtype=np.int64)

    def one(j):
        a = fr.Address.alloc(params)
        a.data = out[j]
        a.encrypt_sk(params, int(idxs[j]), sk, fr.Source(1000 + first + j), fr.Source(5000 + first + j))

    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(one, range(len(idxs))))
    return out


def dump_outputs(out_dir, res, first):
    """Writes the results of the last timed step: `read_limbs.npy` [n][word_size][glwe_len], the ciphertexts a caller of
    the batched read receives (float64 holds every limb exactly), for a fixed, seeded sample of n reads that fits
    DUMP_BYTES, and `read_positions.npy` [n], their positions in the batch."""
    n = min(len(res), DUMP_BYTES // (res[0].size * 8))
    pick = np.sort(np.random.default_rng(0).choice(len(res), size=n, replace=False))
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "read_limbs.npy", res[pick].astype(np.float64))
    np.save(out_dir / "read_positions.npy", (first + pick).astype(np.float64))


def bench_config(args, world):
    """the workload-defining keys, identical in both arms"""
    return {"workload": f"{args.batch} independent encrypted-address reads, RAM 2^{args.max_addr_log2} x {args.word_size} B "
                        "(N=4096, base2k=17)",
            "max_addr": 1 << args.max_addr_log2, "word_size": args.word_size, "k_pt": 9, "batch": args.batch,
            "n_gpus": args.gpus, "host_format": args.host_format}


def cpu_measure(orc, keys, ram, addr_limbs, n_reads, threads, samples, check=None):
    """Warm, repeated timing of the oracle's FFT64 restatement of Ram::read (the CPU port): `samples` runs of n_reads
    reads on `threads` threads after one warm-up run, and single reads on ONE thread (the shape of README.md:36)."""
    addrs = np.ascontiguousarray(addr_limbs[:n_reads]).reshape(-1)
    rc, out = orc.ram_read_many(ram, addrs, n_reads, keys, threads)  # warm-up (page faults, caches, thread pool)
    assert rc == 0
    if check is not None:
        check(out)
    ts = []
    for _ in range(samples):
        t0 = time.perf_counter()
        rc, out = orc.ram_read_many(ram, addrs, n_reads, keys, threads)
        ts.append(time.perf_counter() - t0)
        assert rc == 0
    one = []
    orc.set_ram_threads(1)
    for _ in range(2):
        t0 = time.perf_counter()
        rc, _ = orc.ram_read(ram, addrs[: addrs.size // n_reads], keys)
        one.append(time.perf_counter() - t0)
        assert rc == 0
    return {"reads_per_s": n_reads / float(np.median(ts)), "step_s": float(np.median(ts)),
            "spread": [n_reads / max(ts), n_reads / min(ts)], "one_thread_read_s": float(min(one)), "samples": samples}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--max-addr-log2", type=int, default=18)
    ap.add_argument("--word-size", type=int, default=4)
    ap.add_argument("--cpu-reads", type=int, default=0, help="reads in the cpu_baseline sample (0: auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--host-format", default="p17", choices=["p17", "i32", "i64"],
                    help="host limb format of the e2e call: packed 17-bit fields, int32, or int64 (Poulpy's containers)")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write a seeded sample of the last timed step's read results to DIR as .npy (GPU arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    max_addr, ws, k_pt = 1 << args.max_addr_log2, args.word_size, 9
    from oracle.oracle import host_threads
    threads = host_threads()
    config = bench_config(args, world)

    if args.impl == "reference":
        if rank != 0:
            return
        # inputs from the oracle's OWN client side (keygen, Ram::encrypt_sk, Address::encrypt_sk restated in
        # oracle/fheram_oracle.c): nothing of fhe_ram_b200 is imported or loaded in this arm
        from oracle.oracle import Oracle, build as build_oracle
        build_oracle()
        orc = Oracle(backend="fft64", max_addr=max_addr, word_size=ws, k_pt=k_pt)
        sk = orc.secret_gen(orc.source(0))
        atk, tsk, inv = orc.keygen(sk, orc.source(0), orc.source(0))
        keys = orc.keys_prepare(atk, tsk, inv)
        data = orc.source_bytes(orc.source(5), max_addr * ws)
        ram = orc.ram_new(orc.ram_encrypt(data, sk, orc.source(11), orc.source(12)))
        n_reads = args.cpu_reads or max(1, 4 * threads // ws)  # 4 tasks (read x sub-RAM) per thread: ~1 s of host time per sample
        idxs = np.random.default_rng(7).integers(0, max_addr, size=n_reads)
        addrs = np.stack([orc.address_encrypt(int(i), sk, orc.source(100 + j), orc.source(200 + j)) for j, i in enumerate(idxs)])

        def check(out):  # the port must decrypt correctly too
            for b in range(n_reads):
                for i in range(ws):
                    want = orc.cast_u8_to_signed(int(data[i + ws * idxs[b]]), min(8, k_pt))
                    v, noise = orc.decrypt_glwe(out[b, i], sk, want)
                    assert v == want, "cpu port decrypt mismatch"

        flat = addrs.reshape(-1)
        n_warm = max(2, args.warmup)  # the first passes fault the keys and the RAM in and spin the thread pool up
        for _ in range(n_warm):
            rc, out = orc.ram_read_many(ram, flat, n_reads, keys, threads)
            assert rc == 0
        check(out)
        ts = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            rc, out = orc.ram_read_many(ram, flat, n_reads, keys, threads)
            ts.append(time.perf_counter() - t0)
            assert rc == 0
        one_t = []
        orc.set_ram_threads(1)
        for _ in range(2):
            t0 = time.perf_counter()
            rc, _ = orc.ram_read(ram, flat[: flat.size // n_reads], keys)
            one_t.append(time.perf_counter() - t0)
        one = float(min(one_t))
        v = n_reads / float(np.median(ts))  # median: one descheduled step of a short sample must not set the rate
        sample = (f"{n_reads} Ram::read per step ({n_warm} warm-up + {args.steps} timed steps, median), oracle FFT64 port, "
                  f"{threads} threads; one read on one thread: {one:.2f} s")
        print(json.dumps({
            "impl": "reference", "metric": "batched_reads_per_s", "value": v, "unit": "reads/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.median(ts)) * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config,
            "cpu_baseline": {"value": v, "unit": "reads/s", "cores": threads, "kind": "port", "sample": sample,
                             "one_thread_read_s": one,
                             "readme_reference": "450 ms/read, 1200 ms/write, i9-12900K 1 thread (README.md:36)"},
            "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "the reference binary cannot be built offline (no cargo/rustc; Poulpy path dependency "
                    "absent, Cargo.toml:7-10); each step is a bounded sample of the workload (sample_reads reads of the "
                    f"{args.batch}-read batch)", "sample_reads_per_step": n_reads,
        }))
        return

    import torch
    import hashlib
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    import fhe_ram_b200 as fr
    from fhe_ram_b200 import api

    device = local_rank if world > 1 else 0
    torch.cuda.set_device(device)
    params = fr.Parameters.readme(device=device, max_addr=max_addr, word_size=ws, k_pt=k_pt)
    sk, evk = fr.gen_keys(params)                       # same seeds on every rank: identical keys
    keys = fr.EvaluationKeysPrepared.alloc(params).prepare(evk)
    data = fr.Source(5).fill_bytes(max_addr * ws)
    import ctypes as C
    cts, t_ram_cpu = None, None
    if world == 1:
        # the client side on the CPU (also the RAM of the cpu_baseline); N > 1: every rank encrypts its own shard on
        # its GPU (Ram::encrypt_sk on the device: the same limbs from the same Sources, tests/test_gpu_encrypt.py)
        cts = np.zeros(ws * params.n_glwe() * params.glwe_len(), dtype=np.int64)
        xa, xe = fr.Source(11), fr.Source(12)
        t0 = time.perf_counter()
        api._check(api.lib().fheram_encrypt_ram(C.byref(params.c), data.ctypes.data_as(api._PU8), api._p(sk.data),
                                                xa.h, xe.h, api._p(cts)))
        t_ram_cpu = time.perf_counter() - t0
    B = args.batch
    assert B % world == 0, "--batch must be a multiple of the number of GPUs"
    mine = B // world                                   # reads this rank finishes: [first, first + mine)
    first = rank * mine
    rng = np.random.default_rng(7)
    idxs = rng.integers(0, max_addr, size=B)
    # host buffers: every rank makes (and pins) only ITS addresses, with the client side on the CPU
    t0 = time.perf_counter()
    my_limbs64 = make_addresses(fr, params, sk, idxs[first:first + mine], threads, first)
    t_addr = time.perf_counter() - t0
    fmt = args.host_format
    i32 = fmt != "i64"                                  # results come back as int32 limbs unless the host format is int64
    my_limbs = {"p17": lambda: api.pack17(my_limbs64), "i32": lambda: my_limbs64.astype(np.int32), "i64": lambda: my_limbs64}[fmt]()
    api.host_register(my_limbs)
    stream = torch.cuda.ExternalStream(params.stream(), device=device)
    L = params.glwe_len()
    out_host = np.zeros((mine, ws, L), dtype=np.int32 if i32 else np.int64)
    api.host_register(out_host)
    # device-resident addresses of the whole batch: Address::encrypt_sk on the device (the same limbs as the CPU
    # client side from the same Sources: checked below against this rank's host slice)
    addr_res = fr.Address.encrypt_sk_gpu(params, idxs.astype(np.uint32), sk, [fr.Source(1000 + j) for j in range(B)],
                                         [fr.Source(5000 + j) for j in range(B)], prepare=False)
    per = params.n_ggsw() * params.ggsw_len()
    assert np.array_equal(addr_res.download_raw().reshape(B, per)[first:first + min(mine, 4)], my_limbs64[:min(mine, 4)]), \
        "device Address::encrypt_sk != client side"
    addr_res.prepare()

    if world > 1:
        from fhe_ram_b200.sharded import ShardedRamLib
        ram = ShardedRamLib(params, rank, world)
        ram.ram.encrypt_sk_gpu(data, sk, fr.Source(11), fr.Source(12))
    else:
        ram = fr.Ram.new(params)
        ram.load(cts)

    last_out = [None]   # device pointer of the result arena the latest resident step wrote

    def run_resident():
        last_out[0] = ram.read_batch_device(addr_res, keys)
        return last_out[0]

    def run_e2e():
        # this rank's host address limbs -> device, prepare, read (all exchange steps), results back on the host
        if world > 1:
            return ram.read_batch_host(my_limbs, mine, keys, out_host, fmt=fmt)
        return {"p17": ram.read_batch_host_p17, "i32": ram.read_batch_host_i32, "i64": ram.read_batch_host}[fmt](my_limbs, mine, keys, out_host)

    def check(out):
        """decrypt a sample of this rank's results (examples/fhe-ram.rs:104-115)"""
        for b in (0, mine // 2, mine - 1):
            for i in range(ws):
                want = fr.cast_u8_to_signed(int(data[i + ws * idxs[first + b]]), 8)
                v, noise = fr.decrypt_glwe(params, out[b, i].astype(np.int64), want, sk)
                assert v == want and noise < -(k_pt + 1), (b, i, v, want, noise)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        params.synchronize()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps):
                fn()
            e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=f"cuda:{device}")
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- warm-up, then the device-resident timed region --------------------------------
    sampler = ClockSampler(device)
    sampler.start()
    try:  # the sampler's nvidia-smi must not outlive a failed run
        for _ in range(args.warmup):
            run_resident()
        params.profile(True)
        l0 = params.launch_count()
        sampler.mark_start()
        ms_total = timed(run_resident, args.steps)
        sampler.mark_end()
        launches = params.launch_count() - l0
        prof = params.profile_get()
        params.profile(False)
    finally:
        clocks = sampler.stop()
    ms_step = ms_total / args.steps
    value = B / (ms_step * 1e-3)

    # correctness of what was timed: this rank's slice of the last timed step, decrypted, and -- N > 1 -- compared LIMB
    # FOR LIMB with what ONE GPU computes for the same reads (an unsharded RAM on this rank's GPU, outside every timed region)
    res = np.zeros((mine, ws, L), dtype=np.int64)
    api._check(api.lib().fheram_download_glwe(params.module(), last_out[0], mine * ws, api._p(res)))
    check(res)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, first)
    digest = hashlib.sha256(res.tobytes()).hexdigest()
    parity = None
    if world > 1:
        single = fr.Ram.new(params)
        single.encrypt_sk_gpu(data, sk, fr.Source(11), fr.Source(12))
        own = fr.Address.from_limbs(params, my_limbs64, mine)
        want = single.read_batch(own, keys)
        same = bool(np.array_equal(want, res))
        single.close()
        own._drop()
        flags = [None] * world
        torch.distributed.all_gather_object(flags, (same, digest, hashlib.sha256(want.tobytes()).hexdigest()))
        parity = {"every_rank_equals_one_gpu_limbs": all(f[0] for f in flags),
                  "sha256_sharded": [f[1][:16] for f in flags], "sha256_one_gpu": [f[2][:16] for f in flags]}
        assert parity["every_rank_equals_one_gpu_limbs"], parity

    # ---- end-to-end through the C ABI with host buffers --------------------------------
    e2e = None
    if not args.no_e2e:
        for _ in range(min(args.warmup, 2)):
            run_e2e()
        barrier()
        t0 = time.perf_counter()
        ms_e2e = timed(run_e2e, args.steps)
        wall = (time.perf_counter() - t0) * 1e3
        out = run_e2e()
        check(out)
        assert np.array_equal(out.astype(np.int64), res), "host-buffer path != device-resident path"
        h2d = int(my_limbs.nbytes) * world
        e2e = {"value": B / (ms_e2e / args.steps * 1e-3), "unit": "reads/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(out_host.nbytes) * world,
               "ms_per_step": ms_e2e / args.steps, "wall_ms_per_step": wall / args.steps,
               "host_format": {"p17": "addresses as packed 17-bit fields (fheram_pack17), results as int32 limbs",
                               "i32": "int32 limbs in and out", "i64": "int64 limbs (Poulpy's VecZnx containers) in and out"}[fmt],
               "h2d_gb_per_s_per_gpu": h2d / world / (ms_e2e / args.steps * 1e-3) / 1e9,
               "call": {"p17": "fheram_ram_read_batch_host_p17", "i32": "fheram_ram_read_batch_host_i32",
                        "i64": "fheram_ram_read_batch_host"}[fmt] + ": every rank passes its own batch / n_gpus addresses"}
        if world == 1 and fmt != "i64":   # the other host formats once, for the record (same pipeline, more PCIe bytes)
            l64 = my_limbs64
            api.host_register(l64)
            o64 = np.zeros((mine, ws, L), dtype=np.int64)
            ram.read_batch_host(l64, mine, keys, o64)
            ms64 = timed(lambda: ram.read_batch_host(l64, mine, keys, o64), 1)
            assert np.array_equal(o64, res)
            e2e["i64_value"] = B / (ms64 * 1e-3)
            e2e["i64_h2d_bytes_per_step"] = int(B * per * 8)

    # ---- BASELINE config 4: interleaved read_prepare_write / write stream on the sharded RAM ----
    pair_ms = None
    if world > 1:
        a1 = fr.Address.from_limbs(params, my_limbs64[0] if rank == 0 else np.zeros(per, dtype=np.int64), 1)
        # every rank needs the same address: rank 0's first one
        box = [my_limbs64[0].copy() if rank == 0 else None]
        torch.distributed.broadcast_object_list(box, src=0)
        a1 = fr.Address.from_limbs(params, box[0], 1)
        wv = np.stack([fr.encrypt_glwe(params, int(v), sk) for v in (1, 2, 3, 4)[:ws]])
        ram.read_prepare_write(a1, keys)
        ram.write(wv if rank == 0 else None, a1, keys)
        barrier()
        t0 = time.perf_counter()
        n_pairs = 5
        for _ in range(n_pairs):
            ram.read_prepare_write(a1, keys)
            ram.write(wv if rank == 0 else None, a1, keys)
        barrier()
        t = torch.tensor([(time.perf_counter() - t0) * 1e3 / n_pairs], device=f"cuda:{device}")
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        pair_ms = float(t.item())

    if rank != 0:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
        return

    # ---- single-op latencies (BASELINE metric: read / write ms at 2^18 x 4 B, 1 GPU) ----
    lat = {}
    if world == 1:
        a1 = fr.Address.from_limbs(params, my_limbs64[0], 1)
        a1.device()
        one = np.zeros((1, ws, L), dtype=np.int64)

        def t_call(fn, reps=5):
            ts = []
            for _ in range(reps):
                params.synchronize()
                t0 = time.perf_counter()
                fn()
                params.synchronize()
                ts.append((time.perf_counter() - t0) * 1e3)
            return float(np.median(ts))

        lat["read_ms"] = t_call(lambda: api._check(api.lib().fheram_ram_read(ram.h, a1.device(), keys.h, api._p(one))))
        wv = np.stack([fr.encrypt_glwe(params, int(v), sk) for v in (1, 2, 3, 4)[:ws]])
        rpw, wr = [], []
        for _ in range(3):
            params.synchronize(); t0 = time.perf_counter()
            ram.read_prepare_write(a1, keys)
            params.synchronize(); rpw.append((time.perf_counter() - t0) * 1e3)
            t0 = time.perf_counter()
            ram.write(wv, a1, keys)
            params.synchronize(); wr.append((time.perf_counter() - t0) * 1e3)
        lat["read_prepare_write_ms"] = float(np.median(rpw))
        lat["write_ms"] = float(np.median(wr))

    # ---- SURVEY.md 8(f).1: Ram::encrypt_sk / Address::encrypt_sk on the device (k_glwe_encrypt), set-up path,
    #      outside every timed region above; checked limb for limb against the CPU client side ----
    if world == 1:
        r2 = fr.Ram.new(params)
        r2.encrypt_sk_gpu(data, sk, fr.Source(11), fr.Source(12))  # first call: allocations
        params.synchronize(); t0 = time.perf_counter()
        r2.encrypt_sk_gpu(data, sk, fr.Source(11), fr.Source(12))
        params.synchronize(); t_ram_gpu = time.perf_counter() - t0
        assert np.array_equal(r2.store(), cts), "device Ram::encrypt_sk != client side"
        r2.close()
        na = min(B, 256)
        vals = np.ascontiguousarray(idxs[:na], dtype=np.uint32)
        stages = None
        for rep in range(2):  # second pass: kernels loaded, allocator warm
            xas, xes = [fr.Source(1000 + j) for j in range(na)], [fr.Source(5000 + j) for j in range(na)]
            ha = (C.c_void_p * na)(*[x.h for x in xas])
            he = (C.c_void_p * na)(*[x.h for x in xes])
            params.synchronize(); t0 = time.perf_counter()
            dev = fr.Address.device_alloc(params, na)
            params.synchronize(); t1 = time.perf_counter()
            api._check(api.lib().fheram_address_encrypt_sk(dev.h, 0, na, vals.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                           api._p(sk.data), ha, he, na))
            params.synchronize(); t2 = time.perf_counter()
            dev.prepare()
            params.synchronize(); t3 = time.perf_counter()
            stages = (t1 - t0, t2 - t1, t3 - t2)
            if rep == 0:
                assert np.array_equal(dev.download_raw().reshape(na, -1), my_limbs64[:na]), \
                    "device Address::encrypt_sk != client side"
            dev.close()
        t_addr_gpu = stages[1]
        lat["client_side_encrypt"] = {
            "ram_glwe": int(ws * params.n_glwe()), "ram_cpu_s": round(t_ram_cpu, 3), "ram_gpu_s": round(t_ram_gpu, 4),
            "addresses": na, "address_cpu_per_s": round(B / t_addr, 1), "address_cpu_threads": threads,
            "address_gpu_per_s": round(na / t_addr_gpu, 1),
            "address_gpu_stage_ms": {"device_alloc": round(stages[0] * 1e3, 2), "encrypt": round(stages[1] * 1e3, 2),
                                     "prepare": round(stages[2] * 1e3, 2)},
            "noise": params.encrypt_stats(),
            "note": "GPU path: mask (ChaCha20), noise (Box-Muller on the same stream; the host re-draws the samples "
                    "whose rounding could depend on libm's last bit), product with the secret and normalization on "
                    "the device; limbs equal to the CPU client side (asserted)"}

    # ---- BASELINE config 2: external-product microbenchmark (4096 GLWE x one prepared GGSW) ----
    micro = None
    if world == 1:
        nb = 4096
        rngm = np.random.default_rng(3)
        g_in = rngm.integers(-(1 << 16), 1 << 16, size=(nb, params.glwe_len()), dtype=np.int64)
        ggsw = rngm.integers(-(1 << 16), 1 << 16, size=params.ggsw_len(), dtype=np.int64)
        api.external_product_batch(params, g_in[:296], ggsw)           # warm-up
        params.profile(True)
        api.external_product_batch(params, g_in, ggsw)
        pm = params.profile_get()["ext"]
        params.profile(False)
        micro = {"workload": "4096 GLWE(k=51) x 1 prepared GGSW(k=68), N=4096", "kernel_ms": pm["ms"],
                 "ext_products_per_s": nb / (pm["ms"] * 1e-3), "tflops": nb * F_EXT / (pm["ms"] * 1e-3) / 1e12,
                 "gbs_algorithmic": nb * B_EXT / (pm["ms"] * 1e-3) / 1e9}

    # ---- roofline of the dominant kernel (CUDA events over the timed region) -------------
    (r_ext, r_ks), _ = op_model(max_addr, ws, params.base2d())
    fp64_peak = params.fp64_peak_tflops()
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    cls_flop = {"ext": F_EXT, "trace": F_KS, "combine2": F_KS}
    dom = max(("ext", "trace", "combine2"), key=lambda k: prof[k]["ms"])
    pd = prof[dom]
    ach_tf = pd["ops"] * cls_flop[dom] / (pd["ms"] * 1e-3) / 1e12 if pd["ms"] > 0 else 0.0
    shares = {k: round(prof[k]["ms"] / max(1e-9, sum(prof[c]["ms"] for c in prof)), 4) for k in prof}
    traffic, traffic_src, l1tex_view = None, None, None
    try:  # DRAM bytes per op from the committed ncu --set full capture, scaled to this launch size
        captured = json.loads((ROOT / "profiles" / "ncu_dram_per_op.json").read_text())
        per_op = captured[dom]
        traffic = per_op["dram_bytes_per_op"] * pd["ops"] / max(1, pd["launches"])
        traffic_src = per_op["capture"]
        # the unit ncu shows closest to saturation (not a number measured in this run)
        l1tex_view = {"unit": "l1tex data pipe (shared-memory exchanges + matrix loads)",
                      "pct_of_peak_in_capture": captured["l1tex_data_pipe_pct"][dom], "source": per_op["capture"]}
    except Exception:
        pass
    roofline = {
        "bound": "fp64", "kernel": {"ext": "k_ext8", "trace": "k_ks7", "combine2": "k_ks4<COMBINE2>"}[dom],
        "achieved": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s",
        "frac": ach_tf / fp64_peak if fp64_peak else None, "traffic": traffic, "traffic_source": traffic_src,
        "peak_source": "fp64 FMA probe kernel run in this process (MEASURED_PEAKS.json has no FP64 entry; "
                       "nominal 37.2 TFLOP/s = 148 SM x 64 FMA x 2 x 1.965 GHz)",
        "avg_launch_ms": pd["ms"] / max(1, pd["launches"]), "launches": pd["launches"],
        "ops_per_launch": pd["ops"] / max(1, pd["launches"]), "flop_per_op": cls_flop[dom],
        "kernel_time_share": shares,
        "l1tex_view": l1tex_view,
        "hbm_note": "not the bound: measured DRAM traffic per launch is `traffic` (tens of KB per operation; the prepared "
                    "matrices stream from L2), against %.0f GB/s of measured copy bandwidth" % peaks.get("hbm_gbs", 6650.0),
        "whole_read": {"flop_per_read": r_ext * F_EXT + r_ks * F_KS,
                       "achieved_tflops": value * (r_ext * F_EXT + r_ks * F_KS) / 1e12,
                       "frac_of_fp64_peak": value * (r_ext * F_EXT + r_ks * F_KS) / 1e12 / (fp64_peak * world) if fp64_peak else None},
    }

    # ---- CPU baseline (oracle port) on a bounded sample: warm, repeated, all threads and one thread ----------
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        from oracle.oracle import Oracle
        orc = Oracle(backend="fft64", max_addr=max_addr, word_size=ws, k_pt=k_pt)
        okeys = orc.keys_prepare(evk.atk_glwe, evk.gglwe_to_ggsw_key, evk.atk_ggsw_inv)
        oram = orc.ram_new(cts)
        n_reads = args.cpu_reads or max(1, 4 * threads // ws)  # 4 tasks (read x sub-RAM) per thread: ~1 s of host time per sample

        def cpu_check(out):
            assert np.array_equal(out, res[:n_reads]), "cpu port limbs != CUDA path limbs"

        m = cpu_measure(orc, okeys, oram, my_limbs64, n_reads, threads, 5, cpu_check)
        cpu = {"value": m["reads_per_s"], "unit": "reads/s", "cores": threads, "kind": "port",
               "sample": f"{n_reads} Ram::read of the same workload per run, 1 warm-up + {m['samples']} timed runs (median; "
                         f"{m['spread'][0]:.1f} .. {m['spread'][1]:.1f} reads/s), oracle FFT64 restatement (not the reference "
                         f"binary), {threads} threads; its limbs equal the CUDA path's",
               "one_thread_read_s": m["one_thread_read_s"],
               "readme_reference": "450 ms/read, 1200 ms/write, i9-12900K 1 thread (README.md:36)"}

    line = {
        "metric": "batched_reads_per_s", "value": value, "unit": "reads/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config,
        "parallelism": f"ram sharded by polynomial index mod {world}, exchange steps inside libfheram_cuda.so (NCCL)" if world > 1 else "single gpu",
        "l2": "inputs larger than L2: prepared addresses %.1f GiB + work arenas" % (B * params.n_ggsw() * 1.5 / 1024),
        "address_gen_s": round(t_addr, 2), "result_sha256_rank0": digest, "sharded_parity": parity,
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
        "cpu_baseline": cpu, "ext_product_microbench": micro, **lat,
    }
    if pair_ms is not None:
        line["sharded_rpw_write_pair_ms"] = pair_ms
    if "read_ms" in lat:
        line["vs_readme_read"] = 450.0 / lat["read_ms"]
        line["vs_readme_write"] = 1200.0 / lat["write_ms"]
    print(json.dumps(line))
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
