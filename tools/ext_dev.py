"""Development loop of the external-product kernel (run on the B200 box):
  parity of a 4-step coordinate chain against the CPU oracle on random + extreme inputs,
  then device time of BASELINE config 2 (4096 x 1) and of a 4-step chain over 4096 ciphertexts.
  FHERAM_KERNEL=ext8 / ext9 / ext9c4 forces one external-product kernel for the same run."""
import json
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import fhe_ram_b200 as fr  # noqa: E402
from fhe_ram_b200 import api  # noqa: E402
from oracle.oracle import Oracle  # noqa: E402

F_EXT = 2363392


def main():
    params = fr.Parameters.readme()
    rng = np.random.default_rng(7)
    L, GL = params.glwe_len(), params.ggsw_len()
    out = {"kernel": os.environ.get("FHERAM_KERNEL", "")}
    if "--no-parity" not in sys.argv:
        orc = Oracle(backend="fft64", max_addr=1 << 18, word_size=4, k_pt=9)
        cts = rng.integers(-(1 << 16), 1 << 16, size=(5, L), dtype=np.int64)
        cts[3, :] = -(1 << 16)
        cts[4, :] = (1 << 16) - 1
        ggsws = rng.integers(-(1 << 16), 1 << 16, size=4 * GL, dtype=np.int64)
        ggsws[3 * GL:] = -(1 << 16)
        for nd in (1, 4):
            got = api.coordinate_product(params, cts, ggsws[: nd * GL], nd)
            bad = 0
            for i in range(len(cts)):
                want = orc.coordinate_product(cts[i], ggsws[: nd * GL], nd)
                bad += int(np.count_nonzero(got[i] != want))
            out[f"parity_mismatches_nd{nd}"] = bad
        # more items than SMs (the item loop) against the oracle on a few of them
        n = 300
        cts = rng.integers(-(1 << 16), 1 << 16, size=(n, L), dtype=np.int64)
        got = api.coordinate_product(params, cts, ggsws[: 2 * GL], 2)
        bad = 0
        for i in (0, 147, 148, 299):
            bad += int(np.count_nonzero(got[i] != orc.coordinate_product(cts[i], ggsws[: 2 * GL], 2)))
        out["parity_mismatches_n300"] = bad
    nb = 4096
    g_in = rng.integers(-(1 << 16), 1 << 16, size=(nb, L), dtype=np.int64)
    ggsws = rng.integers(-(1 << 16), 1 << 16, size=4 * GL, dtype=np.int64)
    api.coordinate_product(params, g_in[:296], ggsws[:GL], 1)
    for nd in (1, 4):
        best = None
        for _ in range(3):
            params.profile(True)
            api.coordinate_product(params, g_in, ggsws[: nd * GL], nd)
            pm = params.profile_get()["ext"]
            params.profile(False)
            best = pm["ms"] if best is None else min(best, pm["ms"])
        out[f"ms_4096x{nd}"] = best
        out[f"tflops_4096x{nd}"] = nb * nd * F_EXT / (best * 1e-3) / 1e12
        out[f"cycles_per_ext_per_sm_x{nd}"] = best * 1e-3 * 1.965e9 * 148 / (nb * nd)
    # narrow launch (latency): 4 ciphertexts x 2 steps, as the end of a single read
    api.coordinate_product(params, g_in[:4], ggsws[: 2 * GL], 2)
    params.profile(True)
    api.coordinate_product(params, g_in[:4], ggsws[: 2 * GL], 2)
    out["us_4x2"] = params.profile_get()["ext"]["ms"] * 1e3
    params.profile(False)
    if "--phases" in sys.argv:
        import ctypes as C
        n = 148 * 8
        names = ["pre", "fwd_load", "forward16", "contract", "inverse", "epilogue", "output", "fwd_store_sync"]
        fn = lambda: api.coordinate_product(params, g_in[:n], ggsws, 4)
        fn()
        ph = (C.c_longlong * 8)()
        api._check(api.lib().fheram_debug_phase_cycles(params.module(), 1, ph))
        fn()
        api._check(api.lib().fheram_debug_phase_cycles(params.module(), 0, ph))
        out["phase_cycles_per_ext"] = {nm: round(ph[i] / (n * 4)) for i, nm in enumerate(names)}
        out["phase_total"] = round(sum(ph) / (n * 4))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
