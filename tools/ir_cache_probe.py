#!/usr/bin/env python3
"""What the process-wide eval_check kernel cache and kernel bundles change for a data-defined circuit at rv32im scale
(oracle/synth_ir.build_scaled(560): ~51 k PolyExtSteps, W = 400), pools at max_po2 = 20 on every visible GPU.

  ir_cache_probe.py [--old-lib PATH] [--out FILE]

Each phase runs in a fresh process, since the cache belongs to the process:
  cold    empty cache: pool creation, the first proof of an unseen size (po2 18), then a bundle for po2 18 and 20 (no compile)
  bundle  after hfb200_ir_load_kernels: pool creation, the first po2 18 proof, a context re-created after an injected device
          fault, and the creation of one context
  check   context init and ms_check at po2 = 20 from one context of this build with the bundle loaded and with an empty cache,
          and, with --old-lib, of the previous build (which compiles in every context); alternated, two processes of each
The estimated pool creation before the cache is contexts x the previous build's measured per-context init.
Writes JSON (default profiles/ir_cache_probe.json) with the GPU name and power limit read in the same run."""
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

MAX_PO2, SMALL_PO2 = 20, 18


class _Absent:
    """Stands in for an entry a previous build does not export (the binding sets restype / argtypes of every entry)."""


def _pkg(lib_path=None):
    import hfb200_loader
    pkg = hfb200_loader.load()
    if not lib_path:
        return pkg, pkg.load_library()
    # a previous build lacks the kernel-cache entries: bind what it exports
    real = C.CDLL

    class Tolerant(real):
        def __getattr__(self, name):
            try:
                return real.__getattr__(self, name)
            except AttributeError:
                return _Absent()
    pkg.binding.C.CDLL = Tolerant
    try:
        return pkg, pkg.load_library(lib_path)
    finally:
        pkg.binding.C.CDLL = real


def _ir():
    from oracle import synth_ir   # test infrastructure: only builds the tables
    ir = synth_ir.build_scaled(n_groups=560)
    return ir, tuple(ir["widths"])


def _job(pkg, W, po2, seed):
    rng = np.random.default_rng(seed)
    n = 1 << po2
    code = rng.integers(0, pkg.P, size=(W[0], n), dtype=np.uint32)
    data = rng.integers(0, pkg.P, size=(W[1], n), dtype=np.uint32)
    g = rng.integers(0, pkg.P, size=32, dtype=np.uint32)
    return (po2, g, code, data, seed)


def _pool(pkg, lib, ir, W, cb):
    ndev = pkg.device_count(lib)
    t0 = time.time()
    pool = pkg.Pool(devices=tuple(range(ndev)), contexts_per_device=2, max_po2=MAX_PO2, circuit=W, lib=lib, ir=ir, deterministic=True)
    create_s = time.time() - t0
    pool.set_accum(C.cast(cb.seam_accum, C.c_void_p).value, None)
    return pool, create_s, ndev


def _timed_prove(pool, jobs, cap):
    t0 = time.time()
    pool.prove(jobs, cap)
    return time.time() - t0


def phase_cold(cb_path, bundle_path):
    pkg, lib = _pkg()
    ir, W = _ir()
    cb = C.CDLL(cb_path)
    cap = 1 << 22
    n0 = pkg.ir_nvrtc_programs(lib)
    pool, create_s, ndev = _pool(pkg, lib, ir, W, cb)
    out = {"devices": ndev, "contexts": 2 * ndev, "pool_create_s": round(create_s, 2), "programs_create": pkg.ir_nvrtc_programs(lib) - n0}
    job = _job(pkg, W, SMALL_PO2, 1)
    n1 = pkg.ir_nvrtc_programs(lib)
    out["first_po2_18_proof_s"] = round(_timed_prove(pool, [job], cap), 2)
    out["programs_first_po2_18"] = pkg.ir_nvrtc_programs(lib) - n1
    out["second_po2_18_proof_s"] = round(_timed_prove(pool, [job], cap), 2)
    pool.close()
    t0 = time.time()
    b = pkg.ir_compile(ir, W, [SMALL_PO2, MAX_PO2], lib=lib)
    out["bundle_from_cache_s"] = round(time.time() - t0, 2)
    out["bundle_bytes"] = len(b)
    with open(bundle_path, "wb") as f:
        f.write(b)
    return out


def phase_bundle(cb_path, bundle_path):
    pkg, lib = _pkg()
    ir, W = _ir()
    cb = C.CDLL(cb_path)
    cap = 1 << 22
    t0 = time.time()
    specs = pkg.ir_load_kernels(open(bundle_path, "rb").read(), lib=lib)
    out = {"load_kernels_s": round(time.time() - t0, 2), "specialisations": specs}
    n0 = pkg.ir_nvrtc_programs(lib)
    pool, create_s, ndev = _pool(pkg, lib, ir, W, cb)
    out["pool_create_s"] = round(create_s, 2)
    job = _job(pkg, W, SMALL_PO2, 1)
    out["first_po2_18_proof_s"] = round(_timed_prove(pool, [job], cap), 2)
    out["second_po2_18_proof_s"] = round(_timed_prove(pool, [job], cap), 2)
    pool.inject_fault(0, 0, 0)
    out["po2_18_proof_with_recreated_context_s"] = round(_timed_prove(pool, [job], cap), 2)
    out["contexts_recreated"] = pool.stats()["contexts_recreated"]
    pool.close()
    t0 = time.time()
    with pkg.Context(0, MAX_PO2, W, lib=lib, ir=ir, deterministic=True) as c:
        out["context_init_s"] = round(time.time() - t0, 2)
        out["compile_ms"] = round(c.ir_jit_active()[1], 1)
    out["programs"] = pkg.ir_nvrtc_programs(lib) - n0
    return out


def phase_check(lib_path, bundle_path):
    """Context init and ms_check at po2 = 20 (median of 3 segments after one warm-up) from the build at lib_path."""
    pkg, lib = _pkg(lib_path or None)
    ir, W = _ir()
    if bundle_path:
        pkg.ir_load_kernels(open(bundle_path, "rb").read(), lib=lib)
    po2, g, code, data, seed = _job(pkg, W, MAX_PO2, 7)
    accum = np.random.default_rng(8).integers(0, pkg.P, size=(W[2], 1 << po2), dtype=np.uint32)
    t0 = time.time()
    with pkg.Context(0, MAX_PO2, W, lib=lib, ir=ir, deterministic=True) as c:
        init_s = time.time() - t0
        active, compile_ms = c.ir_jit_active()
        assert active
        ms, seal = [], None
        for i in range(4):
            c.segment_begin(po2, g, code, data, seed)
            seal = c.segment_finish(accum)
            if i:
                ms.append(c.last_stats()["ms_check"])
    import hashlib
    return {"init_s": round(init_s, 2), "compile_ms": round(compile_ms, 1), "ms_check": [round(x, 3) for x in ms],
            "seal_sha256": hashlib.sha256(seal.tobytes()).hexdigest()}


def _child(*args):
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--phase", *[str(a) for a in args]], cwd=ROOT, capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit("phase %s failed:\n%s" % (args[0], r.stderr[-4000:]))
    return json.loads(r.stdout.strip().splitlines()[-1])


def _gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return [ln.strip() for ln in q.stdout.strip().splitlines()]


def main():
    args = sys.argv[1:]
    if args and args[0] == "--phase":
        fn = {"cold": phase_cold, "bundle": phase_bundle, "check": phase_check}[args[1]]
        print(json.dumps(fn(*[a if a != "-" else None for a in args[2:]])))
        return
    old_lib = args[args.index("--old-lib") + 1] if "--old-lib" in args else None
    out_path = args[args.index("--out") + 1] if "--out" in args else os.path.join(ROOT, "profiles", "ir_cache_probe.json")
    tmp = tempfile.mkdtemp(prefix="ir_cache_probe_")
    try:
        import hfb200_loader
        pkg = hfb200_loader.load()
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        cb = os.path.join(tmp, "libseam_cb.so")
        libdir = os.path.dirname(pkg.LIB_PATH)
        subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-Xcompiler", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"),
                               "-o", cb, os.path.join(ROOT, "tools", "accum_seam_cb.cu"), "-L", libdir, "-l:libhfb200.so", "-Xlinker", "-rpath," + libdir])
        bundle = os.path.join(tmp, "rv32im.bundle")
        res = {"what": "eval_check kernel cache and bundles, rv32im-scale data-defined circuit (synth_ir.build_scaled(560)), pools of 2 "
                       "contexts per GPU at max_po2 = 20 (tools/ir_cache_probe.py)",
               "gpus": _gpu_info()}
        def save():
            with open(out_path, "w") as f:
                json.dump(res, f, indent=1)
        res["cold"] = _child("cold", cb, bundle)
        save()
        res["bundle"] = _child("bundle", cb, bundle)
        save()
        checks = {"new_bundle": [], "new_empty_cache": []}
        if old_lib:
            checks["old"] = []
        for _ in range(2):
            if old_lib:
                checks["old"].append(_child("check", old_lib, "-"))
            checks["new_empty_cache"].append(_child("check", "-", "-"))
            checks["new_bundle"].append(_child("check", "-", bundle))
            res["check_po2_20"] = checks
            save()
        res["check_po2_20"] = checks
        res["ms_check_r2_ir_scale"] = 134.173
        if old_lib:
            per_ctx = float(np.median([c["init_s"] for c in checks["old"]]))
            res["previous_build_context_init_s"] = round(per_ctx, 2)
            res["estimated_pool_create_before_s"] = round(per_ctx * res["cold"]["contexts"], 1)
            res["seals_equal_old_new"] = len({c["seal_sha256"] for v in checks.values() for c in v}) == 1
        res["gpus_after"] = _gpu_info()
        save()
        print(json.dumps(res))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
