"""Launches every live kernel of the library at least once, the throughput kernels with WIDE launches (a batch of 64
reads at 2^18 x 4 B): input of the per-kernel ncu table (tools/ncu_per_kernel.sh -> profiles/r2_per_kernel.md)."""
import sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import __graft_entry__ as g
g.build()
import fhe_ram_b200 as fr
from fhe_ram_b200 import api
p = fr.Parameters.readme()
sk, evk = fr.gen_keys(p)
keys = fr.EvaluationKeysPrepared.alloc(p).prepare(evk)              # k_prepare, k_prepare7, k_i64_to_i32
data = fr.Source(5).fill_bytes(p.max_addr() * 4)
ram = fr.Ram.new(p)
ram.encrypt_sk_gpu(data, sk, fr.Source(1), fr.Source(2))            # k_noise_sample, k_glwe_encrypt
B = 64
idxs = np.arange(B, dtype=np.uint32) * 4001 + 7
addrs = fr.Address.encrypt_sk_gpu(p, idxs, sk, [fr.Source(100 + i) for i in range(B)], [fr.Source(300 + i) for i in range(B)])
ram.read_batch_device(addrs, keys)                                  # wide: k_ext8, k_ks7, k_ks4; narrow tails
limbs = addrs.download_raw().reshape(B, -1)
ram.read_batch_host_p17(api.pack17(limbs[:16]), 16, keys)           # k_unpack17 (+ the pipeline)
ram.read_batch_host(limbs[:16], 16, keys)                           # k_i64_to_i32, k_i32_to_i64
one = fr.Address.from_limbs(p, limbs[0], 1)
ram.read(one, keys)                                                 # narrow: k_ext9<8>, k_ks8<8, ...>, k_ks6, k_ks5
ram.read_prepare_write(one, keys)
w = np.stack([fr.encrypt_glwe(p, v, sk) for v in (1, 2, 3, 4)])
ram.write(w, one, keys)                                             # k_vmp<AUTO / EXPAND> (GGSW inversion), k_sub_add_normalize, k_rotate
# launch shapes of a RAM sharded over 8 GPUs (32 ciphertexts per rank): the four-SM cluster variants k_ks8<4, ...>, k_ext9<4>
rng = np.random.default_rng(0)
cts32 = rng.integers(-(1 << 16), 1 << 16, size=(32, p.glwe_len()), dtype=np.int64)
api.glwe_trace(p, keys, cts32)
api.glwe_pack(p, keys, cts32)
api.coordinate_product(p, cts32, limbs[0][: 4 * p.ggsw_len()], 4)
p.synchronize()
print("done", p.launch_count(), "launches")
