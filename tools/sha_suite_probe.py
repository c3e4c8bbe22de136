"""The SHA-256 hash suite against Poseidon2 on one GPU: segment throughput, stage times, the SHA-256 Merkle kernels against
their instruction-issue bound, and host verification.

For each suite and po2 in --po2s (W = 256 = 16 / 192 / 48, deterministic blinding), in one process:
  * resident segments/s with F contexts in flight, F chosen as bench.py chooses it (8, fewer when the arenas would not fit in
    80 % of the free HBM): every context proves its own synthetic segment --steps times after --warmup steps, one host thread
    per context; device time from the earliest start mark to the latest end mark (hfb200_mark, CUDA events on the library's
    streams);
  * ms_hash_main and ms_fri from hfb200_last_stats, mean over --steps segments on ONE context (kernel durations undisturbed);
  * host verification: ms per seal of hfb200_verify_segment_suite, and every seal of the timed run verified against the control
    id of its suite; the SHA-256 seal of the fixed seed (trace seed 0x48595046, blind seed 1) is recorded at po2 = 20.
The SHA-256 Merkle kernels alone (hfb200_hal_sha_rows / _sha_fold on torch tensors, CUDA events on the HAL stream, inputs larger
than the 126 MB L2): leaves of 4 * 2^20 rows x 192 columns (3.2 GB read), the fold of the 2^21-node level and all folds of that
tree, beside Poseidon2's hash_rows of the same matrix.  The issue bound of each kernel: SASS instructions per compression
(cuobjdump -sass of the built library) x compressions / 32 threads per warp-instruction / (148 SMs x 4 schedulers x SM clock);
the kernel's share of that bound is bound / measured time.  Records the card name, power limit and SM clocks.

    python tools/sha_suite_probe.py [--po2s 16 18 20 22] [--steps 4] [--warmup 2] [--out profiles/sha_suite_probe.json]
"""
import argparse
import hashlib
import json
import os
import re
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hfb200_loader  # noqa: E402

W = (16, 192, 48)
TRACE_SEED = 0x48595046
SUITES = ("poseidon2", "sha-256")
SMS, SCHEDULERS_PER_SM = 148, 4


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.check_output(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], text=True, timeout=60)
    vals = [v.strip() for v in out.strip().splitlines()[0].split(",")]
    return dict(zip(q.split(","), vals))


def sass_counts(lib_path):
    """SASS instructions (NOPs excluded) of every SHA-256 kernel in the library, from cuobjdump -sass."""
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    dump = subprocess.check_output([exe, "-sass", lib_path], text=True, timeout=600)
    out = {}
    for part in dump.split("Function : ")[1:]:
        name = part.split("\n", 1)[0].strip()
        m = re.search(r"INS_(\d+)(Sha\w+?Kernel)E", name)
        if not m:
            continue
        ins = re.findall(r"/\*[0-9a-f]{4,}\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)", part)
        ops = [op for _, op in ins if not op.startswith("NOP")]
        out[m.group(2)] = {"instructions": len(ops), "shf": sum(o.startswith("SHF") for o in ops), "lop3": sum(o.startswith("LOP3") for o in ops),
                           "iadd3": sum(o.startswith("IADD3") for o in ops), "prmt": sum(o.startswith("PRMT") for o in ops),
                           "ldg": sum(o.startswith("LDG") for o in ops)}
    return out


def contexts_in_flight(torch, po2):
    """bench.py's choice: 8, fewer when the arenas would not fit in 80 % of the free HBM"""
    free_dev = torch.cuda.mem_get_info(0)[0]
    return max(1, min(8, int(0.8 * free_dev / (7.4e9 * 2.0 ** (po2 - 20)))))


def run_config(pkg, torch, suite, po2, steps, warmup):
    F = contexts_in_flight(torch, po2)
    ctxs = [pkg.Context(0, po2, W, deterministic=True) for _ in range(F)]
    try:
        for c in ctxs:
            c.set_hash_suite(suite)
        gl = [c.witgen_synth(po2, TRACE_SEED + 7919 * i, 1) for i, c in enumerate(ctxs)]
        seals = [None] * F

        def run_all(n):
            errs = []

            def work(i):
                try:
                    ctxs[i].mark(0)
                    for k in range(n):
                        seals[i] = ctxs[i].prove_resident(1 + 17 * k + 101 * i)
                    ctxs[i].mark(1)
                except Exception as e:  # noqa: BLE001
                    errs.append(e)
            th = [threading.Thread(target=work, args=(i,)) for i in range(F)]
            [t.start() for t in th]
            [t.join() for t in th]
            if errs:
                raise errs[0]

        run_all(warmup)
        t0 = time.perf_counter()
        run_all(steps)
        host_s = time.perf_counter() - t0
        dev_s = max(a.mark_elapsed(0, b, 1) for a in ctxs for b in ctxs) * 1e-3
        stages = {"ms_hash_main": 0.0, "ms_fri": 0.0, "ms_device": 0.0, "ms_ntt_main": 0.0}
        for k in range(steps):
            ctxs[0].prove_resident(3 + 17 * k)
            st = ctxs[0].last_stats()
            for key in stages:
                stages[key] += st[key] / steps
        # the fixed-seed seal (context 0's segment, blind seed 1) and the control id of this suite
        fixed = ctxs[0].prove_resident(1)
        timed = [s.copy() for s in seals]
        code = ctxs[0].read_group(1)
        root = ctxs[0].control_root(po2, code)
        t0 = time.perf_counter()
        for s in timed:
            pkg.verify_segment(s, root, W, hashfn=suite)
        verify_ms = (time.perf_counter() - t0) * 1e3 / len(timed)
        pkg.verify_segment(fixed, root, W, hashfn=suite)
        res = {"suite": suite, "po2": po2, "contexts_in_flight": F, "steps": steps, "segments": F * steps,
               "segments_per_s": F * steps / dev_s, "device_s": dev_s, "host_wall_s": host_s,
               "stages_one_context_ms": {k: round(v, 3) for k, v in stages.items()},
               "host_verify_ms_per_seal": round(verify_ms, 2), "seals_verified": len(timed) + 1, "seal_words": int(len(fixed)),
               "control_id": root.tolist(), "fixed_seed_seal_sha256": hashlib.sha256(fixed.tobytes()).hexdigest()}
        return res
    finally:
        for c in ctxs:
            c.close()


def kernel_times(pkg, torch, iters, counts, clock_mhz):
    po2, cols = 20, W[1]
    rows = 4 << po2
    dev = torch.device("cuda:0")
    out = {}
    with pkg.Context(0, 12, (8, 16, 8)) as ctx:
        hal = pkg.Hal(ctx)
        stream = torch.cuda.ExternalStream(hal.stream)
        g = torch.Generator(device=dev).manual_seed(1)
        m = torch.randint(0, 2013265921, (cols, rows), dtype=torch.int64, device=dev, generator=g).to(torch.int32)
        nodes = torch.zeros((2 * rows, 8), dtype=torch.int32, device=dev)
        leaves = nodes[rows:]

        def timed(fn):
            fn()
            hal.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(iters):
                fn()
            e1.record(stream)
            e1.synchronize()
            return e0.elapsed_time(e1) / iters

        def folds():
            size = rows
            while size > 1:
                hal.sha_fold(nodes, size, size // 2)
                size //= 2

        ms_rows = timed(lambda: hal.sha_rows(leaves, m))
        ms_fold_top = timed(lambda: hal.sha_fold(nodes, rows, rows // 2))
        ms_folds = timed(folds)
        ms_p2_rows = timed(lambda: hal.hash_rows(leaves, m))
    blocks = (cols + 15) // 16
    cycles_per_s = SMS * SCHEDULERS_PER_SM * clock_mhz * 1e6   # warp-instructions per second, one per scheduler per cycle
    per_comp_rows = counts["ShaRowsKernel"]["instructions"] / 2   # the kernel holds two compressions: the 16-column loop and the tail
    per_comp_fold = counts["ShaFoldKernel"]["instructions"]
    bound_rows = rows * blocks * per_comp_rows / 32 / cycles_per_s * 1e3
    bound_fold = (rows // 2) * per_comp_fold / 32 / cycles_per_s * 1e3
    out["leaves"] = {"rows": rows, "cols": cols, "compressions": rows * blocks, "bytes_read": rows * cols * 4, "ms": round(ms_rows, 3),
                     "GB_per_s": round(rows * cols * 4 / ms_rows / 1e6, 1), "issue_bound_ms": round(bound_rows, 3),
                     "share_of_issue_bound": round(bound_rows / ms_rows, 3), "poseidon2_hash_rows_ms": round(ms_p2_rows, 3)}
    out["fold_level_2M"] = {"nodes": rows // 2, "ms": round(ms_fold_top, 3), "issue_bound_ms": round(bound_fold, 3),
                            "share_of_issue_bound": round(bound_fold / ms_fold_top, 3)}
    out["all_folds"] = {"nodes": rows - 1, "launches": rows.bit_length() - 1, "ms": round(ms_folds, 3)}
    out["timing"] = "CUDA events on the HAL stream around %d back-to-back calls after one warm-up call; inputs: a %.1f GB matrix (> 126 MB L2)" % (iters, rows * cols * 4 / 1e9)
    out["bound_model"] = ("SASS instructions per compression x compressions / 32 / (%d SMs x %d schedulers x %.0f MHz): one warp-instruction "
                          "per scheduler per cycle; rows kernel counted as half its static instructions (two compressions), fold kernel "
                          "as all of its static instructions (one compression plus loads and stores)" % (SMS, SCHEDULERS_PER_SM, clock_mhz))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--po2s", type=int, nargs="+", default=[16, 18, 20, 22])
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sha_suite_probe.json"))
    a = ap.parse_args()
    import torch
    pkg = hfb200_loader.load()
    info_before = gpu_info()
    counts = sass_counts(pkg.LIB_PATH)
    configs = []
    for po2 in a.po2s:
        for suite in SUITES:   # alternated per size: both suites see the same machine state
            r = run_config(pkg, torch, suite, po2, a.steps, a.warmup)
            print(json.dumps({k: r[k] for k in ("suite", "po2", "contexts_in_flight", "segments_per_s", "stages_one_context_ms", "host_verify_ms_per_seal")}), flush=True)
            configs.append(r)
    clock = float(re.sub(r"[^0-9.]", "", info_before["clocks.max.sm"]) or 0)
    kernels = kernel_times(pkg, torch, a.iters, counts, clock)
    info_after = gpu_info()
    by = {(c["suite"], c["po2"]): c for c in configs}
    ratios = {}
    for po2 in a.po2s:
        p2, sha = by[("poseidon2", po2)], by[("sha-256", po2)]
        ratios[str(po2)] = {"segments_per_s_sha_over_p2": round(sha["segments_per_s"] / p2["segments_per_s"], 3),
                            "ms_hash_main_sha_over_p2": round(sha["stages_one_context_ms"]["ms_hash_main"] / p2["stages_one_context_ms"]["ms_hash_main"], 3),
                            "ms_fri_sha_over_p2": round(sha["stages_one_context_ms"]["ms_fri"] / p2["stages_one_context_ms"]["ms_fri"], 3)}
    out = {"gpu": info_before, "gpu_after": info_after, "widths": list(W), "trace_seed": TRACE_SEED, "blinding": "deterministic",
           "configs": configs, "ratios": ratios, "sha_kernels": kernels, "sass": counts,
           "fixed_seed_seal_po2_20": next((c["fixed_seed_seal_sha256"] for c in configs if c["suite"] == "sha-256" and c["po2"] == 20), None)}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"ratios": ratios, "sha_kernels": kernels}, indent=1))


if __name__ == "__main__":
    main()
