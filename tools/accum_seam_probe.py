"""What the device step_accum seam saves per segment of a data-defined circuit at rv32im scale.

Circuit: oracle/synth_ir.build_scaled(n_groups=560): ~51 k PolyExtSteps, W = 400 (24 / 320 / 56), 14 accum chains.  For po2 18 and
20, ms per segment (host wall clock, every path ends in its seal on the host) of
  host_two_phase   hfb200_segment_begin -> CPU step_accum (the oracle's, OpenMP) -> hfb200_segment_finish(accum): today's path,
                   w_accum * N * 4 bytes uploaded per segment
  device_seam      hfb200_segment_begin_dev -> term kernel + hfb200_segment_accum_scan + _accum_blind (tools/accum_seam_cb.cu,
                   a callback outside libhfb200) -> hfb200_segment_finish_dev
  pool_seam        the same through hfb200_pool_prove with hfb200_pool_set_accum, 2 contexts per device (wall time / jobs)
plus the device time of one hfb200_segment_accum_scan over the 56 columns (CUDA events on the context's stream, mean of
`--scan-iters`), next to the built-in stand-in's ms_accum (its own step_accum, 48 columns) at the same po2.  Trace inputs are
host arrays in every path.  Seals of the three paths are compared for equal seeds.  Prints one JSON line; writes nothing into
the tree (the callback is compiled into a temporary directory).

    python tools/accum_seam_probe.py [--po2 18 20] [--reps 3] [--pool-jobs 4]
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
import hfb200_loader  # noqa: E402
import oracle  # noqa: E402  (CPU step_accum of the host path, and the circuit tables)
from oracle import synth_ir  # noqa: E402

P = 2013265921


def build_callback(pkg, tmp):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    so = os.path.join(tmp, "libseam_cb.so")
    libdir = os.path.dirname(pkg.LIB_PATH)
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-Xcompiler", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"),
                           "-o", so, os.path.join(ROOT, "tools", "accum_seam_cb.cu"), "-L", libdir, "-l:libhfb200.so", "-Xlinker", "-rpath," + libdir])
    lib = C.CDLL(so)
    lib.seam_accum.restype = C.c_int
    lib.seam_accum.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(pkg.SegmentDev), C.c_size_t]
    return lib


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True, timeout=60)
        return [l.strip() for l in out.strip().splitlines()]
    except Exception as e:  # the numbers stand without it, but say so
        return ["unknown (%s)" % type(e).__name__]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--po2", type=int, nargs="+", default=[18, 20])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--pool-jobs", type=int, default=4, help="jobs per device and po2 in the pool leg")
    ap.add_argument("--scan-iters", type=int, default=20)
    args = ap.parse_args()
    pkg = hfb200_loader.load()
    lib = pkg.load_library()
    ndev = pkg.device_count(lib)
    if ndev < 1:
        raise SystemExit("accum_seam_probe: no CUDA device (the measurement has no CPU fallback)")
    ir = synth_ir.build_scaled(n_groups=560)
    W = ir["widths"]
    chains = W[2] // 4
    cir = oracle.Circuit(*W)
    max_po2 = max(args.po2)
    tmp = tempfile.mkdtemp(prefix="accum_seam_probe_")
    result = {"probe": "accum_seam", "circuit": "build_scaled(560)", "widths": list(W), "steps": int(len(ir["steps"])), "devices": ndev,
              "gpu": gpu_info(), "reps": args.reps, "po2": {}}
    try:
        cb = build_callback(pkg, tmp)
        fn = C.cast(cb.seam_accum, C.c_void_p).value
        with pkg.Context(0, max_po2, W, lib=lib, ir=ir, deterministic=True) as c, \
             pkg.Context(0, max_po2, lib=lib, deterministic=True) as builtin:
            for po2 in args.po2:
                n = 1 << po2
                code = cir.gen_code(po2)
                g = cir.gen_globals(po2)
                data = np.random.default_rng(po2).integers(0, P, size=(W[1], n), dtype=np.uint32)
                r = {}

                def host_path(seed):
                    mix = c.segment_begin(po2, g, code, data, seed)
                    return c.segment_finish(cir.step_accum(po2, data, mix, seed))

                def dev_path(seed):
                    seg = c.segment_begin_dev(po2, g, code, data, seed)
                    if cb.seam_accum(None, c._h, C.byref(seg), 0) != 0:
                        raise RuntimeError("callback failed")
                    return c.segment_finish_dev()

                ref = {}
                for name, path in (("host_two_phase", host_path), ("device_seam", dev_path)):
                    ref[name] = path(1)  # warm-up (NVRTC specialisation for this po2, module loads), and the seal to compare
                    ts, acc = [], []
                    for k in range(args.reps):
                        t0 = time.perf_counter()
                        path(2 + k)
                        ts.append((time.perf_counter() - t0) * 1e3)
                        acc.append(c.last_stats()["ms_accum"])
                    r[name + "_ms"] = round(float(np.median(ts)), 2)
                    r[name + "_ms_all"] = [round(t, 2) for t in ts]
                    r[name + "_ms_accum_stat"] = round(float(np.median(acc)), 3)
                r["accum_upload_mb"] = round(W[2] * n * 4 / 1e6, 1)
                # scan kernel alone: 14 chains = 56 columns over N - zk rows, repeated on the segment's accum columns
                seg = c.segment_begin_dev(po2, g, code, data, 1)
                rows = n - seg.zk_rows
                c.segment_accum_scan(0, 0, chains, rows)  # warm-up
                c.mark(0)
                for _ in range(args.scan_iters):
                    c.segment_accum_scan(0, 0, chains, rows)
                c.mark(1)
                r["scan_ms_56_columns"] = round(c.mark_elapsed(0, c, 1) / args.scan_iters, 4)
                r["scan_bytes_moved_mb"] = round(3 * W[2] * rows * 4 / 1e6, 1)  # two reads (block totals, scan) and one write
                r["scan_gbs"] = round(r["scan_bytes_moved_mb"] / 1e3 / (r["scan_ms_56_columns"] / 1e3), 1)
                c.segment_finish_dev()
                # the built-in stand-in's own step_accum (48 columns) at this po2
                builtin.witgen_synth(po2, 7, 1)
                ms = []
                for k in range(args.reps + 1):
                    builtin.prove_resident(1)
                    ms.append(builtin.last_stats()["ms_accum"])
                r["builtin_ms_accum_48_columns"] = round(float(np.median(ms[1:])), 4)
                # pool: 2 contexts per device, the C callback on every worker
                jobs = [(po2, g, code, data, 100 + k) for k in range(args.pool_jobs * ndev)]
                with pkg.Pool(devices=tuple(range(ndev)), contexts_per_device=2, max_po2=po2, circuit=W, lib=lib, ir=ir, deterministic=True) as pool:
                    pool.set_accum(fn)
                    cap = c.seal_words(po2)
                    pool.prove(jobs[:2 * ndev], cap)  # warm-up of every worker context
                    t0 = time.perf_counter()
                    seals, _, _ = pool.prove(jobs, cap)
                    r["pool_seam_ms_per_segment"] = round((time.perf_counter() - t0) * 1e3 / len(jobs), 2)
                    r["pool_jobs"] = len(jobs)
                r["seals_equal"] = bool((ref["host_two_phase"] == ref["device_seam"]).all())
                # the pool's seal for seed 100 against the single-context device path
                r["pool_seal_equal"] = bool((seals[0] == dev_path(100)).all())
                r["saved_ms_per_segment"] = round(r["host_two_phase_ms"] - r["device_seam_ms"], 2)
                result["po2"][str(po2)] = r
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
