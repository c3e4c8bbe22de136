#!/usr/bin/env python3
"""bench.py -- po2=20 segments/second (and camt53 end-to-end proof seconds) of the B200 segment prover.

  python bench.py --gpus N --steps K --warmup W            (N=1 directly; N>1 under torchrun, one rank per GPU)
  python bench.py --impl reference --steps K --warmup W    (the CPU baseline arm, see below)

A "step" is one pass of the hot path over one batch = ONE synthetic rv32im-shaped segment of 2^po2 cycles
(BASELINE.json configs[1]: circuit "synth-rv32im-shape v1", W = 16+192+48 = 256 columns) per GPU.  Segments are
independent, so N GPUs prove N segments per step with no collective on the data path (weak scaling); NCCL is used
only for the timing barrier and the max-over-ranks reduction.

  value : segments/s with the trace already resident in HBM when the timed region starts (hfb200_prove_resident)
  e2e   : the same metric through the reference-facing C-ABI call hfb200_prove_segment with HOST (pinned) trace
          buffers: host->device copy of code+data columns and device->host seal inside the timed region
  roofline : the NTT/LDE pipeline (iNTT+zk_shift and x4 expand+NTT of all 256 columns; 9 launches per segment),
             algorithmic bytes 28*W*N over its CUDA-event time, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline : the CPU oracle (the only CPU implementation of this path that exists here: upstream's Rust crates
             are not vendored / buildable) on a bounded sample, scaled linearly in cycles to po2=20

--dump-outputs DIR writes the seals of the last timed step of `value` (one per context in flight, the arrays
prove_resident returns) as DIR/seal_rank<R>_ctx<I>.npy, u32 words stored exactly as float64.  Blinding is then
derived from the seeds, so the same arguments give the same seals on every run and build.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: the bench writes nothing into it

METRIC = "po2=20 segments/sec (synthetic rv32im-shaped segment, W=256); camt53 proof seconds measured on a 37-segment proof (camt53.proof_seconds)"
UNIT = "segments/s"
WIDTHS = (16, 192, 48)
CAMT53_SEGMENTS = 37  # /root/reference/docs/runtime.md:50 (segment_count of the test camt53 proof)
TRACE_SEED = 0x48595046
DUMP_LIMIT = 64 * 10**6  # bytes --dump-outputs may write over all ranks


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def oracle_sample_po2(steps, warmup):
    # ~7.5 s per po2=16 W=256 segment on 8 cores; keep the whole reference run within a few minutes
    total = max(1, steps + warmup)
    for po2, est in ((16, 8.0), (15, 4.0), (14, 2.0), (13, 1.0)):
        if total * est <= 150:
            return po2
    return 12


def run_oracle_sample(po2, repeats=1):
    """Times the CPU oracle (all host threads, OpenMP) proving one W=256 segment of 2^po2 cycles."""
    import oracle
    # all host cores, regardless of OMP_NUM_THREADS (torchrun exports OMP_NUM_THREADS=1 to its workers)
    try:
        ncpu = len(os.sched_getaffinity(0))
    except AttributeError:
        ncpu = os.cpu_count() or 1
    oracle.lib().orc_set_threads(ncpu)
    cir = oracle.Circuit(*WIDTHS)
    code = cir.gen_code(po2)
    g = cir.gen_globals(TRACE_SEED)
    data = cir.gen_data(po2, code, g, TRACE_SEED, 1)
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        cir.prove(po2, g, code, data, 1)
        times.append(time.perf_counter() - t0)
    cores = oracle.lib().orc_num_threads()
    return times, cores


def reference_arm(args):
    """`--impl reference`: the reference's CPU implementation of the path on the box's host cores.  The real one
    (risc0 3.0.5 Rust crates) cannot be built here, so this is the oracle port (kind = "port").  Every step proves a bounded
    sample segment (2^sample_po2 cycles, W = 256); after the K timed steps ONE real po2 = 20, W = 256 segment -- bench.py's own
    configuration -- is proved and timed, and `value` is that measurement (the scaled sample is reported beside it)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    po2 = args.sample_po2 if args.sample_po2 else oracle_sample_po2(args.steps, args.warmup)
    run_oracle_sample(po2, max(0, args.warmup)) if args.warmup else None
    t0 = time.perf_counter()
    times, cores = run_oracle_sample(po2, args.steps)
    per = sum(times) / len(times)
    scale = float(1 << (args.po2 - po2))
    sample_value = 1.0 / (per * scale)
    full = None
    if not args.no_full_size:
        full_times, _ = run_oracle_sample(args.po2, 1)
        full = full_times[0]
    wall = time.perf_counter() - t0
    value = 1.0 / full if full else sample_value
    sample = "oracle CPU restatement (kind=port), %d threads: K steps of one W=256 segment of 2^%d cycles (%.2f s each; x%d linear in cycles = %.4f segments/s)" % (
        cores, po2, per, int(scale), sample_value)
    if full:
        sample += "; then ONE real po2=%d W=256 segment: %.1f s = the value reported" % (args.po2, full)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (BabyBear mod p)", "data": "synthetic",
            "config": {"workload": "configs[1]: single synthetic rv32im-shaped segment, po2=%d, W=256 (16 code + 192 data + 48 accum)" % args.po2, "po2": args.po2,
                       "sample_po2": po2, "full_size_measured": bool(full), "full_size_seconds": full, "scaled_sample_segments_per_s": sample_value,
                       "camt53_proof_seconds": CAMT53_SEGMENTS / value, "camt53_segments": CAMT53_SEGMENTS},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": wall}
    print(json.dumps(line))
    return 0


def camt53_leg(pkg, ctx, device, po2, inflight, g, code_h, data_h, rank=0, world=1, dist=None, barrier=None, max_over_ranks=None):
    """One camt53-sized proof end to end: 37 po2-sized segments, host buffers in, verified receipt out.  With N ranks the
    segments of the ONE proof are sharded round-robin (scheduler.shard), every rank proves its share on its own GPU through
    the host mirror of the reference call site, and only the seals return to rank 0 over the host (gather_object), where
    the receipt is assembled, sent through its JSON wire form and verified seal by seal.  No data-path collective."""
    import numpy as np
    import importlib
    sched = importlib.import_module("hyperfridge_r0_b200.scheduler")
    with open(os.path.join(ROOT, "tests", "golden", "reference_journal.json")) as f:
        journal_bytes = bytes(json.load(f)["journal_bytes"])
    journal_text = pkg.decode_journal(journal_bytes)
    mine = sched.shard([{"segment": i, "po2": po2} for i in range(CAMT53_SEGMENTS)], rank, world)
    segs = [pkg.Segment(j["segment"], po2, g, code_h, data_h, sched.job_seed(1, 0, j["segment"])) for j in mine]
    opts = pkg.ProverOpts(max_segment_po2=po2, circuit=WIDTHS, devices=(device,), contexts_per_device=inflight)
    cap = ctx.seal_words(po2)
    gathered = None
    with pkg.default_prover(opts) as prover:
        warm = prover.prove(pkg.Session(segs[:inflight], journal_text), seal_cap=cap, n_total=CAMT53_SEGMENTS)  # warm-up: one segment per worker
        if dist is not None:
            tmp = [None] * world if rank == 0 else None
            dist.gather_object([np.asarray(s.seal)[:8] for s in warm.receipt.inner.segments], tmp, dst=0)  # warm the gather path
            barrier()
        t0 = time.perf_counter()
        info = prover.prove(pkg.Session(segs, journal_text), seal_cap=cap, n_total=CAMT53_SEGMENTS)
        if dist is not None:
            gathered = [None] * world if rank == 0 else None
            dist.gather_object([(s.index, np.asarray(s.seal, dtype=np.uint32)) for s in info.receipt.inner.segments], gathered, dst=0)
        prove_s = time.perf_counter() - t0
    if max_over_ranks is not None:
        prove_s = max_over_ranks(prove_s)
    if rank != 0:
        return None
    if gathered is not None:
        allsegs = sorted((x for part in gathered for x in part), key=lambda t: t[0])
        full = pkg.Receipt(pkg.CompositeReceipt([pkg.SegmentReceipt(seal=seal, index=i) for i, seal in allsegs]), pkg.Journal(journal_bytes))
    else:
        full = info.receipt
    t0 = time.perf_counter()
    wire = full.to_json()
    receipt = pkg.Receipt.from_json(wire)
    json_s = time.perf_counter() - t0
    control_id = ctx.control_root(po2, code_h)
    t0 = time.perf_counter()
    receipt.verify(pkg.default_image_id(), {po2: control_id}, circuit=WIDTHS)  # seals + claim chain (image id, state chain, journal digest)
    verify_s = time.perf_counter() - t0
    ok = receipt.journal.bytes_ == journal_bytes and [s.index for s in receipt.inner.segments] == list(range(CAMT53_SEGMENTS))
    if not ok:
        raise SystemExit("bench.py: camt53 receipt does not carry the reference journal / all segments")
    return {"segments": CAMT53_SEGMENTS, "po2": po2, "n_gpus": world, "proof_seconds": prove_s, "segments_per_s": CAMT53_SEGMENTS / prove_s,
            "receipt_json_bytes": len(wire), "receipt_json_roundtrip_seconds": json_s, "verify_seconds": verify_s, "verified": True,
            "journal": "reference fixture journal (tests/golden/reference_journal.json), %d bytes" % len(journal_bytes),
            "how": "default_prover().prove(session) through hfb200_pool_prove with host trace buffers, %d contexts in flight per GPU, segments of the "
                   "one proof sharded round-robin over %d GPU(s), seals gathered on rank 0 over the host; every seal checked by "
                   "hfb200_verify_segment against hfb200_control_root; wall clock, max over ranks" % (inflight, world)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--po2", type=int, default=20)
    ap.add_argument("--sample-po2", type=int, default=0, help="reference arm: size of the CPU sample segment (default: chosen from steps)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-size", action="store_true", help="CPU legs: skip the one real po2-sized oracle segment (sample only)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-control-cache", action="store_true", help="skip the informational e2e leg with the control group kept on the device")
    ap.add_argument("--no-camt53", action="store_true", help="skip the measured 37-segment proof")
    ap.add_argument("--ir-scale", action="store_true", help="run tools/ir_scale_probe.py live (51 k-step data-defined circuit; ~1 min) instead of quoting profiles/r2_ir_scale.json")
    ap.add_argument("--inflight", type=int, default=0, help="prover contexts (segments in flight) per GPU; 0 = auto: 8 (measured best on one B200: 20.0 / 19.7 "
                    "segments/s resident / e2e against 19.9 / 19.1 with 4), fewer when the ranks' pinned trace buffers would take more than a quarter of the host's free memory, never below 4")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the seals of the last timed step as DIR/seal_rank<R>_ctx<I>.npy (float64, at most 64 MB in all; "
                    "blinding derived from the seeds so that runs compare seal for seal)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return reference_arm(args)
    if args.warmup < 3:
        args.warmup = 3
    # stdout carries exactly one JSON line: anything a library prints there (NCCL's version banner, for one) goes to
    # stderr instead; the line itself is written to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import numpy as np
    import torch
    import hfb200_loader
    pkg = hfb200_loader.load()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the prover has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    po2 = args.po2
    N = 1 << po2
    W = sum(WIDTHS)
    if args.inflight > 0:
        F = args.inflight
    else:
        F = 8
        try:  # every context of every rank pins one trace (code + data columns) in host memory for the e2e leg
            avail = next(int(l.split()[1]) * 1024 for l in open("/proc/meminfo") if l.startswith("MemAvailable:"))
            per_ctx = (WIDTHS[0] + WIDTHS[1]) * N * 4 + (64 << 20)
            F = max(4, min(8, int(0.25 * avail / (world * per_ctx))))
        except Exception:
            F = 4
        # device side: one context's arena is ~7.3 GB at po2 = 20 (x4 per two more bits); keep all of them inside 80 % of the free HBM
        free_dev = torch.cuda.mem_get_info(local_rank)[0]
        F = max(1, min(F, int(0.8 * free_dev / (7.4e9 * 2.0 ** (po2 - 20)))))
    # F prover contexts per GPU, each driven by its own host thread (ctypes releases the GIL): while one segment sits
    # in its serial Fiat-Shamir tail or copies its trace, the other keeps the SMs busy.  A step = F segments per GPU.
    deterministic = bool(args.dump_outputs) or os.environ.get("HFB200_DETERMINISTIC_BLINDING", "0") == "1"
    ctxs = [pkg.Context(device=local_rank, max_po2=po2, circuit=WIDTHS, deterministic=deterministic) for _ in range(F)]
    if args.dump_outputs:
        dump_bytes = world * F * ctxs[0].seal_words(po2) * 8
        if dump_bytes > DUMP_LIMIT:
            raise SystemExit("bench.py: --dump-outputs would write %.1f MB (more than %d MB); use fewer --inflight contexts" % (dump_bytes / 1e6, DUMP_LIMIT // 10**6))
        os.makedirs(args.dump_outputs, exist_ok=True)
    # per-(rank, context) segment: seed = f(global seed, rank, slot) -> every context proves a different segment
    gl = [c.witgen_synth(po2, TRACE_SEED + 1000003 * rank + 7919 * i, 1 + rank) for i, c in enumerate(ctxs)]
    ctx, g = ctxs[0], gl[0]

    def run_all(fn, steps):
        """fn(slot, step) on every context, `steps` times each, one thread per context.  Every context records a
        device-timeline mark on its own stream before its first and after its last step (hfb200_mark)."""
        errs = []

        def work(slot):
            try:
                ctxs[slot].mark(0)
                for k in range(steps):
                    fn(slot, k)
                ctxs[slot].mark(1)
            except Exception as e:  # noqa: BLE001
                errs.append(e)
        th = [threading.Thread(target=work, args=(i,)) for i in range(F)]
        [t.start() for t in th]
        [t.join() for t in th]
        if errs:
            raise errs[0]

    def device_seconds():
        """Device time of the last run_all on this GPU: earliest start mark to latest end mark over the contexts
        (CUDA events on the library's own streams; torch.cuda.Event would only see torch's stream)."""
        return max(a.mark_elapsed(0, b, 1) for a in ctxs for b in ctxs) * 1e-3

    # ---------------- value: resident trace ----------------
    seals = [None] * F
    stage = {}
    dev_ms = [0.0]

    def step_resident(slot, k):
        seals[slot] = ctxs[slot].prove_resident(1 + rank + 17 * k + 101 * slot)  # new accum blinding each step: no cached outputs

    run_all(step_resident, args.warmup)
    # per-stage CUDA-event times (and the roofline numerator) are taken with ONE context in flight, so a kernel's
    # duration is its own: `steps` segments on context 0 alone, events on the library's stream
    barrier()
    for k in range(args.steps):
        ctxs[0].prove_resident(3 + rank + 17 * k)
        st = ctxs[0].last_stats()
        dev_ms[0] += st["ms_device"]
        for kk, v in st.items():
            stage[kk] = stage.get(kk, 0.0) + float(v)
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    l0 = sum(c.total_launches() for c in ctxs)
    t0 = time.perf_counter()
    run_all(step_resident, args.steps)
    barrier()
    host_wall = max_over_ranks(time.perf_counter() - t0)
    launches = sum(c.total_launches() for c in ctxs) - l0
    clocks = sampler.stop() if rank == 0 else None
    wall = max_over_ranks(device_seconds())  # device timeline, max over ranks
    dev_ms = max_over_ranks(dev_ms[0])
    launches_all = int(sum_over_ranks(float(launches)))
    ms_per_step = wall * 1e3 / args.steps
    value = world * F * args.steps / wall
    seal = seals[0]
    seal_words = int(len(seal))

    # ---------------- e2e: host buffers through the C ABI ----------------
    e2e = None
    camt53 = None
    if not args.no_e2e:
        hb = []
        for c in ctxs:
            code_h = c.host_alloc((WIDTHS[0], N))
            data_h = c.host_alloc((WIDTHS[1], N))
            code_h[...] = c.read_group(1)
            data_h[...] = c.read_group(2)
            hb.append((code_h, data_h))
        h2d_ms = [0.0]
        seal_h = [None]

        def step_host(slot, k):
            seal_h[0] = ctxs[slot].prove_segment(po2, gl[slot], hb[slot][0], hb[slot][1], 1 + rank + 17 * k + 101 * slot)
            if slot == 0:
                h2d_ms[0] += ctxs[0].last_stats()["ms_h2d"]

        run_all(step_host, 2)
        h2d_ms[0] = 0.0
        barrier()
        t0 = time.perf_counter()
        run_all(step_host, args.steps)
        barrier()
        host_wall_e = max_over_ranks(time.perf_counter() - t0)
        # e2e includes the host side of the call (pinned-buffer H2D enqueue, transcript, seal D2H): the larger of the
        # device-timeline span and the host wall clock around the same K steps, max over ranks
        wall_e = max(max_over_ranks(device_seconds()), host_wall_e)
        e2e_value = world * F * args.steps / wall_e
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(F * ((WIDTHS[0] + WIDTHS[1]) * N * 4 + 128 + 4 * WIDTHS[2])),
               "d2h_bytes_per_step": int(F * len(seal_h[0]) * 4), "ms_per_step": wall_e * 1e3 / args.steps, "host_wall_ms_per_step": host_wall_e * 1e3 / args.steps, "ms_code_h2d_span_per_segment": h2d_ms[0] / args.steps, "h2d_note": "span of the code-column copy on context 0's stream (it queues behind the other contexts' data copies on the copy engine; those contexts keep the SMs busy meanwhile)",
               "host_memory": "pinned (hfb200_host_alloc)"}
        # ---------------- the same e2e call with the control group kept on the device (opt-in, informational) ----------------
        # The control (code) columns depend on (circuit, po2) only; hfb200_control_root commits them once and segments then
        # pass code == NULL: identical seals, one LDE + Merkle tree of 16 columns and 64 MiB of H2D less per segment.  NOT the
        # headline: `value` and `e2e` above rebuild the control commitment for every segment, as upstream's prover does.
        if not args.no_control_cache:
            for c, (code_h, data_h) in zip(ctxs, hb):
                c.control_root(po2, code_h)

            def step_host_cc(slot, k):
                seal_h[0] = ctxs[slot].prove_segment(po2, gl[slot], None, hb[slot][1], 1 + rank + 17 * k + 101 * slot)

            run_all(step_host_cc, 2)
            barrier()
            t0 = time.perf_counter()
            run_all(step_host_cc, args.steps)
            barrier()
            host_wall_c = max_over_ranks(time.perf_counter() - t0)
            wall_c = max(max_over_ranks(device_seconds()), host_wall_c)
            e2e["control_cached"] = {"value": world * F * args.steps / wall_c, "unit": UNIT, "h2d_bytes_per_step": int(F * (WIDTHS[1] * N * 4 + 128)),
                                     "note": "opt-in: control group committed once per (circuit, po2) with hfb200_control_root, segments pass code = NULL; seals identical; not the headline"}

        # ---------------- camt53-sized proof, measured (BASELINE.json configs[2]) ----------------
        # 37 segments (the reference's segment count for data/test, docs/runtime.md:50) of po2=20 through the host mirror
        # of the reference call site: default_prover().prove(session) -> Receipt (host trace buffers, pool of F contexts),
        # then the receipt goes through its JSON wire form, every seal through the product verifier, and the journal
        # must be the reference fixture's.  Wall clock around prove(); verification timed separately.
        if not args.no_camt53:
            camt53 = camt53_leg(pkg, ctxs[0], local_rank, po2, F, gl[0], hb[0][0], hb[0][1], rank, world, dist, barrier, max_over_ranks)
        for c, (code_h, data_h) in zip(ctxs, hb):
            c.host_free(code_h)
            c.host_free(data_h)

    # ---------------- roofline of the NTT/LDE pipeline ----------------
    peak, peak_src = measured_hbm_peak()
    ntt_ms = stage["ms_ntt_main"] / args.steps
    ntt_bytes = 28.0 * W * N
    achieved = ntt_bytes / (ntt_ms * 1e-3) / 1e9 if ntt_ms > 0 else 0.0
    traffic = None
    try:  # measured DRAM bytes per trace element of the three NTT/LDE kernels (one ncu --set full capture, profiles/)
        with open(os.path.join(ROOT, "profiles", "r2_ntt_traffic.json")) as f:
            traffic = float(json.load(f)["bytes_per_trace_element"]) * W * N
    except Exception:
        pass
    roofline = {"kernel": "NTT/LDE pipeline of the 3 main groups: strided_tma_kernel<inverse> (TMA tensor-map tiles, 3-buffer pipeline) + mid_warp_kernel (fused iNTT.zk_shift.expand.NTT chunk stage: one warp per transform, four-warp teams, radix-32 register rounds, 16-byte stores) + strided_tma_kernel<forward>, 9 launches/segment",
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "algorithmic_bytes": ntt_bytes, "ms": ntt_ms, "peak_source": peak_src,
                "note": "traffic = dram__bytes_read+write of the 3 kernels from one ncu --set full capture of THIS round's kernels (profiles/r2_ntt_traffic.json, 59.2 B per trace element) scaled to W*N elements; by design 60*W*N (8+20+32 B per element over the three passes) vs 28*W*N algorithmic; the binding units are the integer-multiply and ALU pipes, not HBM (DESIGN.md section 5)"}
    # Poseidon2 (integer-ALU bound, no HBM roofline): permutations/s
    perms = 4 * N * sum((w + 15) // 16 for w in WIDTHS) + 3 * 4 * N
    hash_ms = stage["ms_hash_main"] / args.steps
    # measured integer-multiply peaks of this GPU (hfb200_bench_modmul: every SM busy with the bare product sequences);
    # one permutation = 852 Montgomery products (213 S-boxes x 4) + 504 Shoup constant products (21 x 24 diagonal)
    barrier()
    peak_sbox = ctx.bench_modmul(2)
    peak_shoup = ctx.bench_modmul(1)
    ideal_ms = perms * (852.0 / peak_sbox + 504.0 / peak_shoup) * 1e3 if peak_sbox > 0 and peak_shoup > 0 else 0.0
    hash_ncu = None
    try:  # pipe utilisation of HashRowsKernel from this round's ncu capture (profiles/r2_hash_ncu.json; not re-measured by this run)
        with open(os.path.join(ROOT, "profiles", "r2_hash_ncu.json")) as f:
            hash_ncu = json.load(f)
    except Exception:
        pass
    poseidon = {"kernel": "HashRowsKernel + HashFoldKernel (Poseidon2 t=24) over the 3 main trees", "bound": "integer multiply pipe (FMA-heavy)", "permutations": perms,
                "ms": hash_ms, "gperm_per_s": perms / (hash_ms * 1e-3) / 1e9 if hash_ms > 0 else 0.0,
                "modmul_per_permutation": {"montgomery_sbox": 852, "shoup_const": 504},
                "modmul_peak_measured_gmul_s": {"sbox_chain": peak_sbox / 1e9, "shoup": peak_shoup / 1e9},
                "ms_at_modmul_peak": ideal_ms, "frac_of_modmul_peak": ideal_ms / hash_ms if hash_ms > 0 else 0.0,
                "ncu": hash_ncu,
                "note": "multiplications only: the 2160 modular additions per permutation share the issue slots (ALU pipe); integer multiplies issue on the heavy half of the FMA pipe only (fmalite = 0), which is ~96 % busy"}

    # the NTT/LDE pipeline against the bound that binds it on sm_100a: 50 butterflies + 6 plain products per trace element,
    # every one a Shoup-form modular product on the heavy half of the FMA pipe (DESIGN.md section 5)
    ntt_products = 56.0 * W * N
    ntt_ideal_ms = ntt_products / peak_shoup * 1e3 if peak_shoup > 0 else 0.0
    roofline["multiply_bound"] = {"bound": "integer multiply pipe (FMA-heavy)", "modular_products": ntt_products, "peak_measured_gmul_s": peak_shoup / 1e9,
                                  "ms_at_peak": ntt_ideal_ms, "frac": ntt_ideal_ms / ntt_ms if ntt_ms > 0 else 0.0,
                                  "note": "multiplications only; at this bound the pipeline would reach %.2f of the HBM peak, which is why the north_star's 0.5 is out of reach for radix-2 BabyBear butterflies on the SIMT pipes" % (ntt_bytes / (ntt_ideal_ms * 1e-3) / 1e9 / peak if ntt_ideal_ms > 0 else 0.0)}

    # ---------------- CPU baseline (rank 0, N=1 only, bounded sample) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        spo2 = 16
        times, cores = run_oracle_sample(spo2, 1)
        scale = float(1 << (po2 - spo2))
        scaled_value = 1.0 / (times[0] * scale)
        full = None
        if not args.no_full_size and po2 <= 20:
            full = run_oracle_sample(po2, 1)[0][0]   # ONE real segment of bench.py's own size (tens of seconds on the box's cores)
        cpu_value = 1.0 / full if full else scaled_value
        cpu = {"value": cpu_value, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "oracle CPU restatement, %d threads: " % cores + (("ONE real W=256 segment of 2^%d cycles: %.1f s (the value); " % (po2, full)) if full else "") +
                         "one W=256 segment of 2^%d cycles: %.2f s, x%d linear in cycles = %.4f segments/s" % (spo2, times[0], int(scale), scaled_value),
               "full_size_seconds": full, "scaled_sample_segments_per_s": scaled_value}

    # the data-defined circuit path at rv32im-v2 scale (51 k PolyExtSteps, W = 400): a static capture of tools/ir_scale_probe.py on this
    # pool's B200 (profiles/r2_ir_scale.json) unless --ir-scale asks for a live run
    ir_obj = None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ir_scale.json")) as f:
            ir_obj = json.load(f)
            ir_obj["measured_by_this_run"] = False
    except Exception:
        pass
    if args.ir_scale and rank == 0:
        for c in ctxs[1:]:
            c.close()
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ir_scale_probe.py"), "run", str(min(po2, 20))], capture_output=True, text=True)
        try:
            ir_obj = json.loads(r.stdout.strip().splitlines()[-1])
            ir_obj["measured_by_this_run"] = True
        except Exception:
            ir_obj = {"error": (r.stderr or r.stdout)[-400:]}
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "host_wall_ms_per_step": host_wall * 1e3 / args.steps, "timing": "CUDA events on the prover streams (hfb200_mark), earliest start to latest end over the contexts, max over ranks",
                "ms_per_segment_device_events_single_context": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u32 (BabyBear mod p, Montgomery)", "data": "synthetic",
                "config": {"workload": "configs[1]: single synthetic rv32im-shaped segment per GPU per step, po2=%d, W=256 (16 code + 192 data + 48 accum), circuit synth-rv32im-shape v1" % po2,
                           "po2": po2, "segments_per_step": world * F, "inflight_per_gpu": F,
                           "parallelism": "segments sharded across %d GPU(s), %d prover contexts in flight per GPU, no collectives" % (world, F),
                           "cache": "inputs (1 GiB trace, 4 GiB LDE) are larger than L2; no flush needed", "seal_words": seal_words,
                           "camt53_segments": CAMT53_SEGMENTS,
                           "camt53_proof_seconds": (camt53 or {}).get("proof_seconds"), "camt53_proof_seconds_is": "MEASURED: wall clock of one 37-segment proof with host trace buffers (camt53 object); null when --no-camt53 / --no-e2e",
                           "blinding": "library default: a fresh 256-bit key from OS entropy per segment, ChaCha20-expanded on the device (the seeds passed are only mixed in)" if not deterministic else "deterministic test mode (HFB200_DETERMINISTIC_BLINDING=1 or --dump-outputs)",
                           "host_syncs_per_segment": stage.get("host_syncs", 0.0) / args.steps},
                "stages_ms_per_segment": {k: v / args.steps for k, v in stage.items() if k.startswith("ms_")},
                "stages_note": "CUDA events on the library stream, one context in flight (kernel durations undisturbed); value/e2e use %d contexts in flight" % F,
                "roofline": roofline, "poseidon2": poseidon, "cpu_baseline": cpu, "e2e": e2e, "camt53": camt53, "ir": ir_obj,
                "gpu_launches": launches_all, "clocks": clocks}
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if args.dump_outputs:
        for slot, s in enumerate(seals):
            np.save(os.path.join(args.dump_outputs, "seal_rank%d_ctx%d.npy" % (rank, slot)), s.astype(np.float64))
    for c in ctxs:
        c.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
