#!/usr/bin/env python3
"""Write shape of the expand kernels on compressible witness slots (TUNING build).  The 2-CTAs-per-SM shared-memory cap of
k_expand_round was chosen for DRAM row locality of uncompressed writes (profiles/r01_expand_sweep.md); with compressed lines the
trade-off may move.  Prints generation throughput of a staged 512-instance batch for each (slots, shared-memory cap, round-kernel
threads, streaming stores, expand group) case; the whole list runs twice, so every case is measured in two alternated passes."""
import os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "proof-of-burn_b200"))
import numpy as np
import pob_b200
from pob_b200 import synth

pob_b200.LIB_PATH = os.path.join(ROOT, "proof-of-burn_b200", "pob_b200", "libpob_b200_tuning.so")
shape = (16, 4, 16, 50, 31, 2, 10 ** 19, 10 ** 20)
N = 512
packed = synth.pack_instances(synth.make_batch(N, shape, seed=5), shape)
ref = None
# (plain slots, expand smem cap KB, round threads, streaming stores, expand group; 0 = default)
CASES = [(1, 85, 256, 0, 0), (0, 85, 256, 0, 0), (0, 120, 256, 0, 0), (0, 70, 256, 0, 0), (0, 50, 256, 0, 0), (0, 0, 256, 0, 0),
         (0, 85, 512, 0, 0), (0, 85, 128, 0, 0), (0, 85, 256, 1, 0), (0, 85, 256, 0, 8), (0, 85, 256, 0, 21)]
for plain, smem_kb, threads, cs, group in CASES * 2:
    env = {"POB_PLAIN_SLOTS": str(plain), "POB_EXPAND_SMEM_KB": str(smem_kb), "POB_EXPAND_THREADS": str(threads), "POB_EXPAND_CS": str(cs)}
    os.environ.update(env)
    if group:
        os.environ["POB_EXPAND_GROUP"] = str(group)
    else:
        os.environ.pop("POB_EXPAND_GROUP", None)
    case = {"plain_slots": plain, "expand_smem_kb": smem_kb, "round_threads": threads, "streaming_stores": cs, "expand_group": group}
    try:
        c = pob_b200.Circuit(pob_b200.MAIN_PROOF_OF_BURN)
        c.stage(packed)
        c.run_packed(None, n=N, staged=True, discard=True)
        t = [c.run_packed(None, n=N, staged=True, discard=True).timing for _ in range(3)]
        best = min(t, key=lambda q: q["total_ms"])
        dg = c.run_packed(packed[:3], digest=True)
        if ref is None:
            ref = dg.digests.copy()
        print(json.dumps({**case, "wit_s": round(N / (best["total_ms"] / 1e3), 1), "wit_s_all": [round(N / (q["total_ms"] / 1e3), 1) for q in t],
                          "expand_gbs": round(32.0 * c.n_signals * N / (best["expand_ms"] / 1e3) / 1e9, 1), "slots": c.desc["n_slots"],
                          "digests_ok": bool(np.array_equal(dg.digests, ref))}), flush=True)
        c.close()
    except Exception as e:
        print(json.dumps({**case, "error": str(e)}), flush=True)
