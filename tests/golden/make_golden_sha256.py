#!/usr/bin/env python3
"""Regenerates tests/golden/golden_sha256_po2_<P>_w256.json from the CPU oracle: the headline configuration of bench.py
(W = 256 = code 16 + data 192 + accum 48, trace seed 0x48595046, blind seed 1) proved with the SHA-256 hash suite
(hashfn = "sha-256", oracle/sha_suite.py).  The file pins every transcript checkpoint, the (Poseidon2) hash of the whole seal, the seal length
and its first / last 64 words, in the format of make_golden_large.py, so the GPU test compares the CUDA path with the
oracle at full size without re-running the oracle.  Self-generated regression pins of the oracle, like the Poseidon2 ones.

usage: python tests/golden/make_golden_sha256.py [po2 ...]   (default: 20)"""
import json
import os
import sys
import time
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from oracle import sha_suite  # noqa: E402

W = (16, 192, 48)
TRACE_SEED = 0x48595046
BLIND_SEED = 1


def make(po2):
    cir = oracle.Circuit(*W)
    t0 = time.time()
    code = cir.gen_code(po2)
    g = cir.gen_globals(TRACE_SEED)
    data = cir.gen_data(po2, code, g, TRACE_SEED, BLIND_SEED)
    t1 = time.time()
    sha_cir = sha_suite.Circuit(*W)
    seal, cps = sha_cir.prove(po2, g, code, data, BLIND_SEED)
    t2 = time.time()
    out = {"widths": list(W), "po2": po2, "trace_seed": TRACE_SEED, "blind_seed": BLIND_SEED, "hashfn": "sha-256",
           "control_id": sha_cir.control_id(po2).tolist(),
           "seal_words": int(len(seal)),
           "seal_hash": oracle.hash_elems(seal % oracle.P).tolist(),
           "seal_head": seal[:64].tolist(), "seal_tail": seal[-64:].tolist(),
           "seal_sum_u64": int(seal.astype(np.uint64).sum()),
           "checkpoints": {k: v.tolist() for k, v in cps.items()},
           "oracle_seconds": {"witgen": round(t1 - t0, 2), "prove": round(t2 - t1, 2), "threads": os.cpu_count()}}
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_sha256_po2_%d_w256.json" % po2)
    with open(path, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print("wrote %s (prove %.1f s)" % (path, t2 - t1), flush=True)


if __name__ == "__main__":
    oracle.build()
    for p in ([int(a) for a in sys.argv[1:]] or [20]):
        make(p)
