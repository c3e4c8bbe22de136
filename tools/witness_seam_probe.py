"""What the device witness seam saves per segment when the witness is generated on the GPU.

Two comparisons, each on one GPU and on all visible GPUs (pools with 2 contexts per device, every job of a run at po2 20), each
with a `host` leg and a `witgen` leg (the key prefixes of the JSON):
  stand-in circuit, W = 256 (16 / 192 / 48), runs "standin_w256_gpus_<n>":
    host     jobs carry their data columns in pinned host memory (uploaded by the library)
    witgen   jobs carry data = NULL; the witgen callback of tools/witness_seam_cb.cu copies one 64-bit seed per column into
             hfb200_segment_scratch and expands it on the device, hfb200_segment_data_blind writes the blinding rows
  build_scaled(560), W = 400 (24 / 320 / 56), with the accum callback of tools/accum_seam_cb.cu in both legs, runs
  "scaled560_w400_gpus_<n>":
    host     jobs carry their data columns in pageable host memory (the configuration of profiles/accum_seam_probe.json)
    witgen   data = NULL through the witgen callback, then the accum callback
Both legs of a comparison run in the same pool, on the same columns (the host columns are the numpy expansion of the callback's
seeds with the key's blinding rows) and give the same seals, which the probe checks.  Every job uses a shared control group
(hfb200_pool_load_control), so the legs differ only in where the data columns come from.  Timing: host wall clock around
hfb200_pool_prove, which returns with every seal on the host; median of `--reps` runs, the legs alternating.  Prints one JSON
line, with the card name and power limit; writes nothing into the tree (the callbacks are compiled into a temporary directory).

    python tools/witness_seam_probe.py [--reps 3] [--jobs-per-device 8]
"""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import hfb200_loader  # noqa: E402
import oracle  # noqa: E402  (control columns and globals of the stand-in)
from oracle import synth_ir  # noqa: E402
from test_device_witness_seam import PinnedSeeds, column_seeds, expand_columns  # noqa: E402

PO2 = 20


def build_callbacks(pkg, tmp):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    libdir = os.path.dirname(pkg.LIB_PATH)
    out = {}
    for name in ("witness_seam_cb", "accum_seam_cb"):
        so = os.path.join(tmp, "lib%s.so" % name)
        subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-Xcompiler", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"),
                               "-o", so, os.path.join(ROOT, "tools", name + ".cu"), "-L", libdir, "-l:libhfb200.so", "-Xlinker", "-rpath," + libdir])
        out[name] = C.CDLL(so)
    return C.cast(out["witness_seam_cb"].seam_witgen, C.c_void_p).value, C.cast(out["accum_seam_cb"].seam_accum, C.c_void_p).value


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True, timeout=60)
        return [l.strip() for l in out.strip().splitlines()]
    except Exception as e:  # the numbers stand without it, but say so
        return ["unknown (%s)" % type(e).__name__]


def compare(pkg, lib, devices, widths, ir, host_data, seeds, jobs_per_device, reps, wfn, afn):
    """Alternating runs of the host-data leg and the witgen leg in one pool; returns the timings and whether the seals agree."""
    cir = oracle.Circuit(*widths)
    code, g = cir.gen_code(PO2), cir.gen_globals(PO2)
    n_jobs = jobs_per_device * len(devices)
    pinned = PinnedSeeds(pkg, lib, [seeds] * n_jobs)
    try:
        with pkg.Pool(devices=devices, contexts_per_device=2, max_po2=PO2, circuit=widths, lib=lib, ir=ir, deterministic=True) as pool:
            pool.set_witgen(wfn, C.addressof(pinned.input))
            if afn:
                pool.set_accum(afn)
            pool.load_control(PO2, code)
            legs = {"host": [(PO2, g, None, host_data, 1)] * n_jobs, "witgen": [(PO2, g, None, None, 1)] * n_jobs}
            cap = 1 << 22
            seals = {k: pool.prove(v[:2 * len(devices)], cap)[0][0] for k, v in legs.items()}  # warm-up of every worker context
            ts = {k: [] for k in legs}
            for _ in range(reps):
                for k, v in legs.items():
                    t0 = time.perf_counter()
                    pool.prove(v, cap)
                    ts[k].append((time.perf_counter() - t0) * 1e3 / n_jobs)
    finally:
        pinned.close()
    r = {"jobs": n_jobs, "seals_equal": bool(len(seals["host"]) == len(seals["witgen"]) and (seals["host"] == seals["witgen"]).all())}
    for k, v in ts.items():
        med = float(np.median(v))
        r[k + "_ms_per_segment"] = round(med, 2)
        r[k + "_ms_all"] = [round(t, 2) for t in v]
        r[k + "_segments_per_s"] = round(1e3 / med, 2)
    r["saved_ms_per_segment"] = round(r["host_ms_per_segment"] - r["witgen_ms_per_segment"], 2)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--jobs-per-device", type=int, default=8)
    args = ap.parse_args()
    pkg = hfb200_loader.load()
    lib = pkg.load_library()
    ndev = pkg.device_count(lib)
    if ndev < 1:
        raise SystemExit("witness_seam_probe: no CUDA device (the measurement has no CPU fallback)")
    device_sets = [(0,)] + ([tuple(range(ndev))] if ndev > 1 else [])
    tmp = tempfile.mkdtemp(prefix="witness_seam_probe_")
    result = {"probe": "witness_seam", "po2": PO2, "devices": ndev, "gpu": gpu_info(), "reps": args.reps,
              "contexts_per_device": 2, "jobs_per_device": args.jobs_per_device, "runs": {}}
    try:
        wfn, afn = build_callbacks(pkg, tmp)
        # stand-in circuit, pinned host data against the witgen callback
        widths = (16, 192, 48)
        seeds = column_seeds(1, widths[1])
        cols = expand_columns(seeds, PO2, 1)
        ctx = pkg.Context(0, 12, (8, 16, 8), lib=lib)
        pinned = ctx.host_alloc(cols.shape)
        pinned[...] = cols
        del cols
        for devs in device_sets:
            result["runs"]["standin_w256_gpus_%d" % len(devs)] = compare(pkg, lib, devs, widths, None, pinned, seeds, args.jobs_per_device,
                                                                         args.reps, wfn, None)
        ctx.host_free(pinned)
        ctx.close()
        # rv32im-scale data-defined circuit, pageable host data + accum callback against witgen + accum callbacks
        ir = synth_ir.build_scaled(n_groups=560)
        W = ir["widths"]
        seeds = column_seeds(2, W[1])
        cols = expand_columns(seeds, PO2, 1)
        result["data_upload_mb_w400"] = round(cols.nbytes / 1e6, 1)
        for devs in device_sets:
            result["runs"]["scaled560_w400_gpus_%d" % len(devs)] = compare(pkg, lib, devs, W, ir, cols, seeds, max(2, args.jobs_per_device // 2),
                                                                           args.reps, wfn, afn)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
