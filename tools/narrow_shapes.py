"""Device time of the narrow launch shapes of a RAM sharded over 8 GPUs (32 ciphertexts per rank) and of the tail of a read
(4 ciphertexts), under the current kernel selection (FHERAM_KERNEL=ks6,ext8 gives the one- and two-SM kernels)."""
import json, os, sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import __graft_entry__ as g
g.build()
import fhe_ram_b200 as fr
from fhe_ram_b200 import api
p = fr.Parameters.readme()
sk, evk = fr.gen_keys(p)
keys = fr.EvaluationKeysPrepared.alloc(p).prepare(evk)
rng = np.random.default_rng(0)
L, GL = p.glwe_len(), p.ggsw_len()
ggsws = rng.integers(-(1 << 16), 1 << 16, size=4 * GL, dtype=np.int64)
out = {"kernel": os.environ.get("FHERAM_KERNEL", "")}
for n in (4, 16, 32, 64):
    cts = rng.integers(-(1 << 16), 1 << 16, size=(n, L), dtype=np.int64)
    api.glwe_trace(p, keys, cts); api.coordinate_product(p, cts, ggsws, 4)
    p.profile(True); api.glwe_trace(p, keys, cts); t = p.profile_get()["trace"]["ms"] * 1e3; p.profile(False)
    p.profile(True); api.coordinate_product(p, cts, ggsws, 4); e = p.profile_get()["ext"]["ms"] * 1e3; p.profile(False)
    out[f"trace12_x{n}_us"] = round(t, 1); out[f"ext4_x{n}_us"] = round(e, 1)
    if n >= 8:
        api.glwe_pack(p, keys, cts)
        p.profile(True); api.glwe_pack(p, keys, cts); pm = p.profile_get(); p.profile(False)
        out[f"pack_x{n}_us"] = {k: round(v["ms"] * 1e3, 1) for k, v in pm.items() if v["launches"]}
print(json.dumps(out))
