"""Sharded multi-GPU FHE-RAM (SURVEY.md 8e): one process per GPU.

Two layers:
  * ShardedRamLib -- the product path: the exchange steps (all-gather of prepared GGSWs, all-to-all of packed
    partials, all-gather for read_prepare_write, broadcast of the written word) run INSIDE libfheram_cuda.so on its
    own NCCL communicator (fheram_comm_init); Python only hands the 128-byte communicator id from rank 0 to the
    other ranks (torch.distributed object broadcast) and calls the same entry points as on one GPU.
  * ShardedRam -- the same schedule with the exchange done by torch.distributed around an `engine` object
    (GpuEngine = the *_local_device / *_finish_device halves of the C ABI; tests substitute an oracle-backed engine to
    exercise the host logic with gloo on CPU).

Partition: rank g keeps the polynomials h == g (mod G) of every sub-RAM.  The packer feeds its
inputs in bit-reversed order (src/ram.rs:426,512), so the polynomials of one rank form one
contiguous block of the packing tree and everything below the top log2(G) levels is local
(rotation by the first coordinate, one-sided levels, local two-sided levels).  One exchange step
per batch of reads: every rank ends with one partial ciphertext per (read, sub-RAM); an
all-to-all hands read q's G partials to rank q*G/B, which finishes it (top log2 G levels, second
coordinate, trace).  Never a floating-point reduction: each combine runs exactly once, on integer
limbs, so the result is bit-identical to the single-GPU / reference order.

read_prepare_write all-gathers instead (one read) and finishes on every rank, so every rank
holds tree[0][0]; Ram::write then needs no communication at all (each rank rebuilds the new
packed polynomial redundantly and updates its own slice).

The arithmetic lives behind an `engine` object (GpuEngine = the C ABI; tests substitute an
oracle-backed engine to exercise this host logic with gloo on CPU).
"""
from __future__ import annotations

import ctypes as C

import numpy as np


def shard_of_read(q: int, n_reads: int, world: int) -> int:
    """rank that finishes read q (reads are split into `world` equal contiguous slices)"""
    return q // (n_reads // world)


class _DevView:
    """exposes a raw device pointer to torch through __cuda_array_interface__ (no copy)"""

    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (ptr, False), "version": 2}


class GpuEngine:
    """Local / finishing stages through libfheram_cuda.so (include/fheram.h).

    Stream contract: the library queues its kernels on the context's private stream while torch's collectives order
    against torch's CURRENT stream, so every method of ShardedRam that touches this engine runs inside
    `self.stream_ctx()` (the context stream as torch's current stream): partials are complete before NCCL reads
    them and are not overwritten while it still does."""

    def __init__(self, params, rank: int, world: int, cts_full: np.ndarray):
        from . import api
        self.api, self.params, self.rank, self.world = api, params, rank, world
        self.ram = api.Ram(params, shard=rank, n_shards=world)
        self.ram.load(cts_full)
        self.L = params.word_size() * params.glwe_len()     # int32 limbs per read result / partial

    def stream_ctx(self):
        import torch
        return torch.cuda.stream(torch.cuda.ExternalStream(self.params.stream(), device=self.params.device))

    def _tensor(self, ptr, n):
        import torch
        return torch.as_tensor(_DevView(int(ptr), n), device=f"cuda:{self.params.device}")

    def read_local(self, addrs, keys):
        d = C.c_void_p()
        self.api._check(self.api.lib().fheram_ram_read_local_device(self.ram.h, addrs.device(), keys.h, C.byref(d)))
        return self._tensor(d.value, addrs.count * self.L)

    def read_finish(self, gathered, n_entries, addrs, addr_first, keys):
        d = C.c_void_p()
        self.api._check(self.api.lib().fheram_ram_read_finish_device(
            self.ram.h, C.c_void_p(gathered.data_ptr()), n_entries, 0, n_entries, addrs.device(), addr_first,
            keys.h, C.byref(d)))
        return self._tensor(d.value, n_entries * self.L)

    def rpw_local(self, addr, keys):
        d = C.c_void_p()
        self.api._check(self.api.lib().fheram_ram_rpw_local_device(self.ram.h, addr.device(), keys.h, C.byref(d)))
        return self._tensor(d.value, self.L)

    def rpw_finish(self, gathered, addr, keys):
        d = C.c_void_p()
        self.api._check(self.api.lib().fheram_ram_rpw_finish_device(
            self.ram.h, C.c_void_p(gathered.data_ptr()), addr.device(), keys.h, C.byref(d)))
        return self._tensor(d.value, self.L)

    def write(self, w, addr, keys):
        self.ram.write(w, addr, keys)

    def empty(self, n):
        import torch
        return torch.empty(n, dtype=torch.int32, device=f"cuda:{self.params.device}")

    def to_host(self, t):
        return t.cpu().numpy().astype(np.int64)

    def store(self):
        return self.ram.store()


class ShardedRam:
    """Ram (src/ram.rs:25-29) sharded over the ranks of the default process group."""

    def __init__(self, engine, rank: int, world: int):
        assert world & (world - 1) == 0, "world size must be a power of two"
        self.e, self.rank, self.world = engine, rank, world

    def _ctx(self):
        """the engine's stream as torch's current stream (GpuEngine); engines without one run as they are"""
        import contextlib
        return self.e.stream_ctx() if hasattr(self.e, "stream_ctx") else contextlib.nullcontext()

    # ---- batched reads ------------------------------------------------------------------
    def read_batch_local_slice(self, addrs, keys):
        """B = addrs.count independent reads.  Returns this rank's slice of the results:
        reads [rank*B/G, (rank+1)*B/G), as a flat int32 tensor [B/G][word_size][glwe limbs]."""
        import torch.distributed as dist
        B, G = addrs.count, self.world
        assert B % G == 0, "batch must be a multiple of the world size"
        with self._ctx():
            part = self.e.read_local(addrs, keys)                  # [B][ws] partials of the local slice
            if G == 1:
                return self.e.read_finish(part, B, addrs, 0, keys)
            recv = self.e.empty(part.numel())                      # [G shards][B/G][ws]
            dist.all_to_all_single(recv, part)                     # chunk r of `part` = reads of rank r
            return self.e.read_finish(recv, B // G, addrs, self.rank * (B // G), keys)

    def read_batch(self, addrs, keys):
        """all B results on every rank ([B][word_size][limbs] int64 numpy), for tests"""
        import torch.distributed as dist
        with self._ctx():
            mine = self.read_batch_local_slice(addrs, keys)
            if self.world == 1:
                return self.e.to_host(mine)
            full = self.e.empty(mine.numel() * self.world)
            dist.all_gather_into_tensor(full, mine.contiguous())
            return self.e.to_host(full)

    # ---- read_prepare_write / write -----------------------------------------------------
    def read_prepare_write(self, addr, keys):
        import torch.distributed as dist
        with self._ctx():
            part = self.e.rpw_local(addr, keys)
            if self.world > 1:
                gathered = self.e.empty(part.numel() * self.world)  # [G][1][ws]
                dist.all_gather_into_tensor(gathered, part.contiguous())
            else:
                gathered = part
            return self.e.to_host(self.e.rpw_finish(gathered, addr, keys))

    def write(self, w, addr, keys):
        """Ram::write (src/ram.rs:226-294): no communication (see module docstring)."""
        self.e.write(w, addr, keys)


class ShardedRamLib:
    """Ram (src/ram.rs:25-29) sharded over the ranks of the default process group, every exchange step inside the
    library (include/fheram.h, fheram_comm_*).  The calls are the single-GPU ones; what differs is what they mean on
    a sharded RAM (see the header): batches are split over the ranks, read_prepare_write returns the same result on
    every rank, write takes rank 0's word."""

    def __init__(self, params, rank: int, world: int, cts_full: np.ndarray | None = None):
        from . import api
        assert world & (world - 1) == 0, "world size must be a power of two"
        self.api, self.params, self.rank, self.world = api, params, rank, world
        if world > 1:
            import torch.distributed as dist
            box = [api.Parameters.comm_unique_id().tobytes() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            params.comm_init(world, rank, np.frombuffer(box[0], dtype=np.uint8))
        self.ram = api.Ram(params, shard=rank, n_shards=world)
        if cts_full is not None:
            self.ram.load(cts_full)

    def read_batch(self, addrs, keys) -> np.ndarray:
        """addrs = the whole batch (the same on every rank); returns this rank's slice of the results"""
        return self.ram.read_batch(addrs, keys)

    def read_batch_device(self, addrs, keys) -> int:
        return self.ram.read_batch_device(addrs, keys)

    def read_batch_host(self, my_addr_limbs, n, keys, out=None, fmt="i64"):
        """my_addr_limbs = THIS rank's n addresses in host format `fmt` (i64 / i32 limbs, p17 packed); returns this
        rank's n results"""
        fn = {"i64": self.ram.read_batch_host, "i32": self.ram.read_batch_host_i32, "p17": self.ram.read_batch_host_p17}[fmt]
        return fn(my_addr_limbs, n, keys, out)

    def read_batch_host_seeded(self, my_bodies_p17, my_seeds, n, keys, out=None):
        """THIS rank's n seeded addresses (packed bodies + one seed each); returns this rank's n results"""
        return self.ram.read_batch_host_seeded(my_bodies_p17, my_seeds, n, keys, out)

    def read_prepare_write(self, addr, keys) -> np.ndarray:
        return self.ram.read_prepare_write(addr, keys)

    def write(self, w, addr, keys) -> None:
        self.ram.write(w, addr, keys)

    def read_plain(self, addrs, keys, out=None) -> np.ndarray:
        """addrs = the same plaintext addresses on every rank; returns all n results on every rank"""
        return self.ram.read_plain(addrs, keys, out)

    def read_plain_device(self, addrs, keys) -> int:
        return self.ram.read_plain_device(addrs, keys)

    def write_plain(self, addr, w, keys) -> None:
        """rank 0's word is written (the other ranks may pass None)"""
        self.ram.write_plain(addr, w, keys)

    def store(self) -> np.ndarray:
        return self.ram.store()

    def close(self):
        self.ram.close()
        if self.world > 1:
            self.params.comm_destroy()
