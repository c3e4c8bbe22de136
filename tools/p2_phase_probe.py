"""Cycles per permutation of each phase of the tensor-core Poseidon2 permutation (p2_mix_tc), from clock64.

Needs a build with the phase probe compiled in, e.g.
    tools/build_variant.sh probe3 -ldl -DP2_PHASE_PROBE=1 -DP2TC_BLOCKS=3
    python tools/p2_phase_probe.py variants/libhfb200_probe3.so [--rows 65536]
It runs one 192-column Merkle build (HashRowsKernel, then HashFoldKernel on the levels above 4096 nodes) after a warm-up
build, and prints, per phase, the cycles lane 0 of warp 1 of every CTA spent in it, averaged over the permutations it ran.
The sampled warp does not issue the MMAs, so a round trip is what every waiting warp sees: A row stores, CTA barrier,
MMA issue and commit by thread 0, mbarrier wait.
"""
import argparse
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def phase_names(n_blocks):
    names = ["full rounds (first 4 + external layer)"]
    for b in range(n_blocks):
        names += ["GEMM 1 round trip (v row stores + MMA)" if b == 0 else "block GEMM %d round trip (delta row stores + MMA)" % b,
                  "block %d loads + recombination" % b, "block %d S-box chain" % b]
    names += ["GEMM 2 round trip (delta row stores + MMA)", "GEMM 2 loads + recombination", "full rounds (last 4)"]
    return names


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("lib", help="a libhfb200 build with -DP2_PHASE_PROBE=1")
    ap.add_argument("--rows", type=int, default=1 << 16)
    ap.add_argument("--cols", type=int, default=192)
    a = ap.parse_args()
    import hfb200_loader
    pkg = hfb200_loader.load()
    lib = pkg.load_library(os.path.abspath(a.lib))
    fn = lib.hfb200_p2_probe_read
    fn.restype = C.c_char_p
    fn.argtypes = [C.c_void_p, C.POINTER(C.c_ulonglong), C.POINTER(C.c_uint32)]
    m = np.random.default_rng(1).integers(0, 2013265921, (a.cols, a.rows), dtype=np.uint32)
    out = (C.c_ulonglong * 32)()
    n = C.c_uint32()
    with pkg.Context(0, 12, (8, 16, 8), lib=lib) as c:
        c.op_merkle(m)  # warm-up: module load, first launches
        err = fn(c._h, out, C.byref(n))
        if err:
            raise RuntimeError(err.decode())
        c.op_merkle(m)
        err = fn(c._h, out, C.byref(n))
        if err:
            raise RuntimeError(err.decode())
    n_ph = n.value
    perms = out[n_ph]
    n_blocks = (n_ph - 4) // 3
    print("p2_mix_tc phases, P2TC_BLOCKS = %d, Merkle %d rows x %d columns, %d sampled permutations (one lane per CTA)"
          % (n_blocks, a.rows, a.cols, perms))
    total = 0.0
    for i, name in enumerate(phase_names(n_blocks)):
        cyc = out[i] / max(perms, 1)
        total += cyc
        print("  %2d  %-52s %8.1f cycles" % (i, name, cyc))
    print("      %-52s %8.1f cycles" % ("sum", total))


if __name__ == "__main__":
    main()
