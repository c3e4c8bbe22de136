"""Device time of every device-HAL operator (hfb200_hal_*) at po2 = 20, W = 256 (16 / 192 / 48) on one GPU, beside the fused
segment-prover stage of the same shape.

Inputs are device-resident torch tensors built from one synthetic segment (hfb200_witgen_synth, proved once so that the fused
stage times of hfb200_last_stats exist).  Every operator is warmed up, then timed with CUDA events recorded on the HAL stream
around `--iters` back-to-back calls (mean per call).  The fused comparisons:
    interpolate + zk_shift + expand x4 over the 192 data columns   vs  hfb200_bench_lde(20, 192): the fused LDE of the same columns
    hash_rows + every fold over 4N x 192                           vs  hfb200_bench_merkle(20, 192)
    batch_evaluate_any (the stand-in's taps) + mix_poly_coeffs + poly_divide   vs  ms_deep of the proved segment
    fri_fold at n = N                                              vs  ms_fri of the proved segment (all rounds and the queries)
The extra HBM traffic the HAL's interpolate-then-expand pays over the fused LDE is one coefficient round trip, 8 * w * N bytes;
its modelled time at the card's bandwidth is reported beside the measured difference.  Records the card name and power limit.

    python tools/hal_probe.py [--iters 10] [--out profiles/hal_probe.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hfb200_loader  # noqa: E402
import oracle  # noqa: E402  (the stand-in circuit's taps)

PO2, W = 20, (16, 192, 48)
HBM_GBS = 7700.0  # HGX B200 data sheet, one GPU: only for the modelled round-trip time


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True, timeout=60)
        return [line.strip() for line in out.strip().splitlines()][:1]
    except Exception as e:  # the numbers stand without it, but say so
        return ["nvidia-smi unavailable: %s" % e]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "hal_probe.json"))
    a = ap.parse_args()
    import torch
    pkg = hfb200_loader.load()
    n = 1 << PO2
    with pkg.Context(0, PO2, W, deterministic=True) as seg:
        seg.witgen_synth(PO2, 0x48595046, 1)
        seg.prove_resident(1)
        seg.prove_resident(1)
        fused = seg.last_stats()
        fused_lde = seg.bench_lde(PO2, W[1], a.iters)
        fused_merkle = seg.bench_merkle(PO2, W[1], a.iters)
        groups = [seg.read_group(g) for g in (0, 1, 2)]  # accum, code, data
    cols = np.concatenate(groups)  # 256 columns in the taps' global order: accum, code, data
    taps = oracle.Circuit(*W).taps()
    base = {0: 0, 1: W[2], 2: W[2] + W[0]}
    dev = torch.device("cuda:0")
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x, dtype=np.uint32).view(np.int32)).to(dev)

    with pkg.Context(0, 12, (8, 16, 8)) as ctx:
        hal = pkg.Hal(ctx)
        stream = torch.cuda.ExternalStream(hal.stream)
        rng = np.random.default_rng(1)
        data = t(groups[2])
        work = data.clone()  # transformed in place by every timed call (values stay canonical)
        ev = torch.empty((W[1], 4 * n), dtype=torch.int32, device=dev)
        nodes = torch.empty((8 * n, 8), dtype=torch.int32, device=dev)
        allc = t(cols)
        which = t(np.array([base[g] + o for g, o, _ in taps.tolist()], np.uint32))
        xs = t(rng.integers(0, 2013265921, (len(taps), 4), dtype=np.uint32))
        evals = torch.empty((len(taps), 4), dtype=torch.int32, device=dev)
        regs = {}
        for g, o, b in taps.tolist():
            regs.setdefault(base[g] + o, []).append(b)
        sets = sorted(set(tuple(v) for v in regs.values()))
        combo = t(np.array([sets.index(tuple(regs[c])) if c in regs else 0 for c in range(cols.shape[0])], np.uint32))
        combos = torch.zeros((len(sets), n, 4), dtype=torch.int32, device=dev)
        poly = t(rng.integers(0, 2013265921, (n, 4), dtype=np.uint32))
        rem = torch.empty(4, dtype=torch.int32, device=dev)
        fri_in = t(rng.integers(0, 2013265921, (4, n), dtype=np.uint32))
        fri_out = torch.empty((4, n // 16), dtype=torch.int32, device=dev)
        mix = t(rng.integers(0, 2013265921, 4, dtype=np.uint32))
        ms, mx = [5, 6, 7, 8], [9, 10, 11, 12]
        torch.cuda.synchronize()

        def folds():
            size = 4 * n
            while size > 1:
                hal.hash_fold(nodes, size, size // 2)
                size //= 2
        ops = {
            "batch_interpolate_ntt_192": lambda: hal.batch_interpolate_ntt(work),
            "zk_shift_192": lambda: hal.zk_shift(work),
            "batch_expand_x4_192": lambda: hal.batch_expand_into_evaluate_ntt(ev, work, 2),
            "batch_bit_reverse_192": lambda: hal.batch_bit_reverse(work),
            "hash_rows_4N_192": lambda: hal.hash_rows(nodes[4 * n:], ev),
            "hash_fold_all_levels_4N": folds,
            "batch_evaluate_any_taps_256cols": lambda: hal.batch_evaluate_any(allc, which, xs, evals),
            "mix_poly_coeffs_256cols": lambda: hal.mix_poly_coeffs(combos, ms, mx, allc, combo),
            "poly_divide_N": lambda: hal.poly_divide(poly, [1, 2, 3, 4], rem),
            "prefix_products_N": lambda: hal.prefix_products(poly),
            "fri_fold_N": lambda: hal.fri_fold(fri_out, fri_in, mix),
        }
        ms_of = {}
        for name, fn in ops.items():
            fn()  # warm-up
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(a.iters):
                fn()
            e1.record(stream)
            hal.sync()
            ms_of[name] = e0.elapsed_time(e1) / a.iters
        syncs = hal.host_syncs()

    hal_lde = ms_of["batch_interpolate_ntt_192"] + ms_of["zk_shift_192"] + ms_of["batch_expand_x4_192"]
    hal_tree = ms_of["hash_rows_4N_192"] + ms_of["hash_fold_all_levels_4N"]
    hal_deep = ms_of["batch_evaluate_any_taps_256cols"] + ms_of["mix_poly_coeffs_256cols"] + len(sets) * ms_of["poly_divide_N"]
    extra_bytes = 8 * W[1] * n
    res = {
        "gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "po2": PO2, "widths": W, "iters": a.iters,
        "hal_ms": {k: round(v, 4) for k, v in ms_of.items()},
        "taps": int(len(taps)), "combos": len(sets), "hal_host_syncs_end": int(syncs),
        "compare": {
            "lde_192": {"hal_interpolate_shift_expand_ms": round(hal_lde, 3), "fused_lde_ms": round(fused_lde, 3),
                        "ratio": round(hal_lde / fused_lde, 3) if fused_lde else None,
                        "coefficient_round_trip_bytes": extra_bytes, "modelled_round_trip_ms_at_7700_gbs": round(extra_bytes / HBM_GBS / 1e6, 3)},
            "merkle_4N_192": {"hal_hash_rows_folds_ms": round(hal_tree, 3), "fused_merkle_ms": round(fused_merkle, 3),
                              "ratio": round(hal_tree / fused_merkle, 3) if fused_merkle else None},
            "deep": {"hal_evaluate_mix_divide_ms": round(hal_deep, 3), "segment_ms_deep": round(fused["ms_deep"], 3),
                     "note": "poly_divide counted once per combo; segment ms_deep also computes the DEEP quotient on the LDE domain"},
            "fri": {"hal_fri_fold_N_ms": round(ms_of["fri_fold_N"], 4), "segment_ms_fri": round(fused["ms_fri"], 3),
                    "note": "segment ms_fri covers every FRI round, its Merkle trees and the query openings"},
        },
        "segment_stats": {k: (round(v, 3) if isinstance(v, float) else v) for k, v in fused.items()},
    }
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
