"""Segment sizes that change inside one context or one pool worker.

A context is created for its largest segment size (max_po2) and proves whatever size each call passes.  Real sessions mix
sizes: the last segment of a session is usually shorter, and a pool worker proves whatever jobs it draws.  State that depends
on the size has to follow every change: the arena layout with the resident trace and the cached control group, the pinned
landing buffer of the device transcript, the CUDA graphs of transcript mode 2 (one per shape) and the NVRTC eval_check
kernels of a data-defined circuit (one specialisation per size).

Every seal is compared word for word with the CPU oracle's seal for the same globals, traces and blind seed.  Every segment
of a sequence has its own trace seed and blind seed, so a stale seal, a stale check buffer or a stale control group cannot
pass.
"""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import numpy as np
import pytest
from conftest import TRACE_SEED, make_segment

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WIDTHS = (16, 64, 16)
MAX_PO2 = 14
# starts below max_po2, so the first larger segment (the 4th) comes after the small shape has been captured and replayed,
# and the 5th segment (12 after 14) is a replay of the po2 12 graph in transcript mode 2
SEQUENCE = [12, 12, 12, 14, 12, 13, 14, 14, 12]
IR_SEQUENCE = [14, 12, 13, 12, 14]
# three pool calls on one worker: a batch is proved longest first, so the size can only go up within a call
POOL_CALLS = [[12, 12, 12], [14], [12, 12]]

_inputs, _oracle = {}, {}


def segment_inputs(orc, po2, trace_seed, blind):
    """(globals, code, data) of the built-in circuit at WIDTHS; the data columns carry `blind` in their blinding rows."""
    key = (po2, trace_seed, blind)
    if key not in _inputs:
        _, g, code, data = make_segment(orc, WIDTHS, po2, trace_seed=trace_seed, blind_seed=blind)
        _inputs[key] = (g, code, data)
    return _inputs[key]


def oracle_proof(orc, po2, trace_seed, blind):
    """(seal, checkpoints) of the oracle for segment_inputs(po2, trace_seed, blind), proved once per distinct input."""
    key = (po2, trace_seed, blind)
    if key not in _oracle:
        g, code, data = segment_inputs(orc, po2, trace_seed, blind)
        seal, cps, _ = orc.Circuit(*WIDTHS).prove(po2, g, code, data, blind)
        _oracle[key] = (seal, cps)
    return _oracle[key]


def assert_seal(seal, oseal, what):
    assert len(seal) == len(oseal) and (seal == oseal).all(), what


def prove_sequence(orc, c, seq, seed0, blind0):
    for i, po2 in enumerate(seq):
        ts, blind = seed0 + i, blind0 + i
        g, code, data = segment_inputs(orc, po2, ts, blind)
        seal = c.prove_segment(po2, g, code, data, blind)
        assert_seal(seal, oracle_proof(orc, po2, ts, blind)[0], (i, po2))


def check_sequence_in_mode(pkg, lib, orc, mode):
    """SEQUENCE through one context in transcript mode `mode`, then a control group captured at po2 13 and reloaded with other
    columns at the same po2.  Returns (graph launches after the sequence, after the control-group segments)."""
    with pkg.Context(0, MAX_PO2, WIDTHS, lib=lib, deterministic=True) as c:
        c.set_transcript(mode)
        prove_sequence(orc, c, SEQUENCE, 1000, 40)
        after_sequence = c.graph_launches()
        # code == None: the cached control group (a shape of its own in mode 2): plain run, capture, replay
        _, code, _ = segment_inputs(orc, 13, 2000, 70)
        c.control_root(13, code)
        for i in range(3):
            g, _, data = segment_inputs(orc, 13, 2000 + i, 70 + i)
            assert_seal(c.prove_segment(13, g, None, data, 70 + i), oracle_proof(orc, 13, 2000 + i, 70 + i)[0], ("control", i))
        # other control columns at the same po2: the replayed graph must commit the reloaded group, not the captured one
        code2 = code.copy()
        code2[6, :100] = code[7, :100]
        c.control_root(13, code2)
        g, _, data = segment_inputs(orc, 13, 2003, 73)
        oseal2 = orc.Circuit(*WIDTHS).prove(13, g, code2, data, 73)[0]
        assert not (oseal2 == oracle_proof(orc, 13, 2003, 73)[0]).all()
        assert_seal(c.prove_segment(13, g, None, data, 73), oseal2, "reloaded control group")
        return after_sequence, c.graph_launches()


# ---- CPU tier: the host emulator of the same kernel sources -----------------------------------------------------------------

@pytest.mark.parametrize("mode", [0, 1, 2])
def test_mixed_sizes_in_one_context(pkg, emu_lib, orc, mode):
    """Host transcript (0), device transcript (1) and device transcript with graph replay (2; the emulator has no graphs)."""
    assert check_sequence_in_mode(pkg, emu_lib, orc, mode) == (0, 0)


def test_two_phase_entries_across_sizes(pkg, emu_lib, orc):
    cir = orc.Circuit(*WIDTHS)
    with pkg.Context(0, MAX_PO2, WIDTHS, lib=emu_lib, deterministic=True) as c:
        for i, po2 in enumerate((13, 12, 14)):
            ts, blind = 3000 + i, 80 + i
            g, code, data = segment_inputs(orc, po2, ts, blind)
            oseal, ocps = oracle_proof(orc, po2, ts, blind)
            mix = c.segment_begin(po2, g, code, data, blind)
            assert (mix == ocps["accum_mix"]).all(), po2
            assert_seal(c.segment_finish(cir.step_accum(po2, data, mix, blind)), oseal, po2)


def test_resident_trace_and_control_group_follow_the_size(pkg, emu_lib, orc):
    """The resident trace is the last one placed in the context, whatever its size; a control group does not survive a size
    change."""
    cir = orc.Circuit(*WIDTHS)
    with pkg.Context(0, MAX_PO2, WIDTHS, lib=emu_lib, deterministic=True) as c:
        c.witgen_synth(12, TRACE_SEED, 1)
        g, code, data = segment_inputs(orc, 13, 4000, 90)
        assert_seal(c.prove_segment(13, g, code, data, 90), oracle_proof(orc, 13, 4000, 90)[0], "host buffers")
        assert (c.read_group(2) == data).all()
        # another blind seed: a new proof of the resident po2 13 trace (the data keeps its blinding rows, the accum noise follows the call)
        assert_seal(c.prove_resident(91), cir.prove(13, g, code, data, 91)[0], "resident")
        c.control_root(13, code)
        assert_seal(c.prove_segment(13, g, None, data, 90), oracle_proof(orc, 13, 4000, 90)[0], "control group")
        g12, code12, data12 = segment_inputs(orc, 12, 4001, 92)
        assert_seal(c.prove_segment(12, g12, code12, data12, 92), oracle_proof(orc, 12, 4001, 92)[0], "po2 12")
        with pytest.raises(pkg.Hfb200Error, match="no control group"):
            c.prove_segment(13, g, None, data, 90)
        c.control_root(13, code)
        assert (c.read_group(1) == code).all()
        assert_seal(c.prove_segment(13, g, None, data, 90), oracle_proof(orc, 13, 4000, 90)[0], "reloaded control group")


def ir_circuit(orc):
    from oracle import synth_ir
    ir = synth_ir.build(WIDTHS, 1, nest=True)
    cir_ir = orc.Circuit(*WIDTHS, variant=1)
    cir_ir.set_ir(ir["taps"], ir["steps"], ir["ret"], ir.get("info"))
    return ir, orc.Circuit(*WIDTHS, variant=1), cir_ir


def prove_ir_sequence(c, cir, cir_ir, seq, seed0):
    seals = []
    for i, po2 in enumerate(seq):
        ts, blind = seed0 + i, 20 + i
        code = cir.gen_code(po2); g = cir.gen_globals(ts); data = cir.gen_data(po2, code, g, ts, blind)
        key = ("ir", po2, ts, blind)
        if key not in _oracle:
            _oracle[key] = cir_ir.prove(po2, g, code, data, blind)[0]
        mix = c.segment_begin(po2, g, code, data, blind)
        seal = c.segment_finish(cir.step_accum(po2, data, mix, blind))
        assert_seal(seal, _oracle[key], (i, po2))
        seals.append(seal)
    return seals


def test_data_defined_circuit_mixed_sizes(pkg, emu_lib, orc):
    ir, cir, cir_ir = ir_circuit(orc)
    with pkg.Context(0, MAX_PO2, WIDTHS, lib=emu_lib, ir=ir, deterministic=True) as c:
        prove_ir_sequence(c, cir, cir_ir, IR_SEQUENCE, 5000)


def test_seal_words_only_for_supported_sizes(pkg, emu_lib, orc):
    """hfb200_seal_words is 0 outside [12, 22] (the sizes a context can be created for), model-exact inside it -- also above the
    context's own max_po2 -- and grows with po2, so a buffer sized for max_po2 holds the seal of every smaller segment."""
    cir = orc.Circuit(*WIDTHS)
    with pkg.Context(0, MAX_PO2, WIDTHS, lib=emu_lib) as c:
        for po2 in (0, 11, 23, 32, 40, 64, 70):
            assert c.seal_words(po2) == 0, po2
        sizes = [c.seal_words(po2) for po2 in range(12, 23)]
        assert sizes == [cir.seal_words_model(po2) for po2 in range(12, 23)]
        assert all(a < b for a, b in zip(sizes, sizes[1:]))


def test_pool_rejects_each_job_outside_its_range(pkg, emu_lib, orc):
    """Jobs of unsupported sizes fail one by one with their own reason; the valid job of the batch is proved.  Called through
    ctypes: Pool.prove sizes the trace as 1 << po2 and rejects these jobs before the library sees them."""
    g, code, data = segment_inputs(orc, 12, 6000, 110)
    oseal = oracle_proof(orc, 12, 6000, 110)[0]
    po2s = [11, 23, 12, 64]
    cap = len(oseal) + 64
    seals = [np.zeros(cap, np.uint32) for _ in po2s]
    jobs = (pkg.SegmentJob * len(po2s))()
    for i, po2 in enumerate(po2s):
        jobs[i].po2, jobs[i].blind_seed = po2, 110
        jobs[i].globals, jobs[i].code, jobs[i].data = g.ctypes.data, code.ctypes.data, data.ctypes.data
        jobs[i].seal_out, jobs[i].seal_cap = seals[i].ctypes.data, cap
    with pkg.Pool(devices=(0,), contexts_per_device=1, max_po2=13, circuit=WIDTHS, lib=emu_lib, deterministic=True) as pool:
        e = emu_lib.hfb200_pool_prove(pool._h, jobs, len(po2s))
        assert e
        msg = C.cast(e, C.c_char_p).value.decode()
        emu_lib.hfb200_free_error(e)
        assert msg == "job 0: job po2 11 outside [12, 13]"
        for i, po2 in enumerate(po2s):
            if po2 == 12:
                assert not jobs[i].error and jobs[i].attempts == 1
                assert_seal(seals[i][:jobs[i].seal_words], oseal, "valid job")
                continue
            err = C.cast(jobs[i].error, C.c_char_p).value.decode()
            emu_lib.hfb200_free_error(jobs[i].error)
            assert err == "job po2 %d outside [12, 13]" % po2
            assert jobs[i].seal_words == 0 and jobs[i].attempts == 0


def pool_calls(pkg, lib, orc):
    """POOL_CALLS on a pool with one worker (max_po2 14).  Returns the seals of every call."""
    cap = orc.Circuit(*WIDTHS).seal_words_model(MAX_PO2)
    out = []
    with pkg.Pool(devices=(0,), contexts_per_device=1, max_po2=MAX_PO2, circuit=WIDTHS, lib=lib, deterministic=True) as pool:
        for k, call in enumerate(POOL_CALLS):
            jobs = []
            for i, po2 in enumerate(call):
                ts, blind = 7000 + 10 * k + i, 120 + 10 * k + i
                jobs.append((po2, *segment_inputs(orc, po2, ts, blind), blind))
            seals, _, _ = pool.prove(jobs, cap)
            out.append(seals)
    return out


def expected_pool_seals(orc):
    return [[oracle_proof(orc, po2, 7000 + 10 * k + i, 120 + 10 * k + i)[0] for i, po2 in enumerate(call)] for k, call in enumerate(POOL_CALLS)]


def test_pool_worker_changes_size_between_calls(pkg, emu_lib, orc):
    got = pool_calls(pkg, emu_lib, orc)
    for k, (seals, expect) in enumerate(zip(got, expected_pool_seals(orc))):
        for i, (a, b) in enumerate(zip(seals, expect)):
            assert_seal(a, b, (k, i))


# ---- GPU tier -------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_mixed_sizes_in_one_context_on_gpu(pkg, gpu_lib, orc, mode, monkeypatch):
    """In mode 2 the first segment of a shape runs plainly and every later one is a graph launch; the 5th segment (12 after 14)
    replays a graph captured before the context proved a larger segment.  Checkpoint read-back is off: it disables replay."""
    monkeypatch.delenv("HFB200_DEBUG_CHECKPOINTS", raising=False)
    after_sequence, after_control = check_sequence_in_mode(pkg, gpu_lib, orc, mode)
    if mode == 2:
        assert after_sequence == len(SEQUENCE) - len(set(SEQUENCE))
        assert after_control == after_sequence + 3   # control group: plain, capture, replay, replay after the reload
    else:
        assert after_sequence == after_control == 0


_POOL_CHILD = r"""
import hashlib, json, os, sys
root = sys.argv[1]
sys.path[:0] = [root, os.path.join(root, "tests")]
import hfb200_loader, oracle
import test_mixed_po2 as t
pkg = hfb200_loader.load()
lib = pkg.load_library()
seals = t.pool_calls(pkg, lib, oracle)
# the transcript mode of this process, seen by a context that never sets one: 3 segments of one shape -> 2 graph launches
with pkg.Context(0, 12, t.WIDTHS, lib=lib, deterministic=True) as c:
    for i in range(3):
        g, code, data = t.segment_inputs(oracle, 12, 7000 + i, 120 + i)
        c.prove_segment(12, g, code, data, 120 + i)
    launches = c.graph_launches()
print(json.dumps({"seals": [[hashlib.sha256(s.tobytes()).hexdigest() for s in call] for call in seals], "graph_launches": launches}))
"""


@pytest.mark.gpu
def test_pool_worker_changes_size_between_calls_graph_replay_on_gpu(orc):
    """The pool sequence in transcript mode 2.  The pool takes the mode from the environment, read once per process, so it runs
    in a child process started with HFB200_DEVICE_TRANSCRIPT=2."""
    env = dict(os.environ, HFB200_DEVICE_TRANSCRIPT="2", HFB200_DETERMINISTIC_BLINDING="1")
    env.pop("HFB200_DEBUG_CHECKPOINTS", None)
    r = subprocess.run([sys.executable, "-c", _POOL_CHILD, ROOT], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    assert got["graph_launches"] == 2
    expect = [[hashlib.sha256(np.ascontiguousarray(s, np.uint32).tobytes()).hexdigest() for s in call] for call in expected_pool_seals(orc)]
    assert got["seals"] == expect


@pytest.mark.gpu
def test_data_defined_circuit_mixed_sizes_on_gpu(pkg, gpu_lib, orc, monkeypatch):
    """The NVRTC kernels are specialised per size (max_po2 at creation, the others when first proved): every size must run its
    own.  The interpreter kernel (HFB200_IR_JIT=0) gives the same seals."""
    ir, cir, cir_ir = ir_circuit(orc)
    seals = {}
    for jit in ("1", "0"):
        monkeypatch.setenv("HFB200_IR_JIT", jit)
        with pkg.Context(0, MAX_PO2, WIDTHS, lib=gpu_lib, ir=ir, deterministic=True) as c:
            assert c.ir_jit_active()[0] == (jit == "1")
            seals[jit] = prove_ir_sequence(c, cir, cir_ir, IR_SEQUENCE, 5000)
    assert all((a == b).all() for a, b in zip(seals["1"], seals["0"]))


@pytest.mark.gpu
def test_data_defined_circuit_at_rv32im_scale_mixed_sizes_on_gpu(pkg, gpu_lib, orc):
    """~51 k PolyExtSteps, W = 400, in a max_po2 = 16 context proving po2 16, 12, 16 with the NVRTC kernels (two
    specialisations); random data columns, one oracle proof per segment."""
    from oracle import synth_ir
    ir = synth_ir.build_scaled(n_groups=560)
    W = ir["widths"]
    cir = orc.Circuit(*W)
    cir_ir = orc.Circuit(*W)
    cir_ir.set_ir(ir["taps"], ir["steps"], ir["ret"], ir.get("info"))
    with pkg.Context(0, 16, W, lib=gpu_lib, ir=ir, deterministic=True) as c:
        assert c.ir_jit_active()[0]
        for i, po2 in enumerate((16, 12, 16)):
            code = cir.gen_code(po2); g = cir.gen_globals(30 + i)
            data = np.random.default_rng(30 + i).integers(0, orc.P, size=(W[1], 1 << po2), dtype=np.uint32)
            oseal = cir_ir.prove(po2, g, code, data, 30 + i)[0]
            mix = c.segment_begin(po2, g, code, data, 30 + i)
            assert_seal(c.segment_finish(cir.step_accum(po2, data, mix, 30 + i)), oseal, (i, po2))


@pytest.mark.gpu
def test_four_contexts_with_different_size_sequences_on_gpu(pkg, gpu_lib, orc):
    """Four contexts on one GPU, one host thread each: trace uploads of contexts on a device are chained in FIFO order, and
    here neighbouring uploads differ in size."""
    seqs = [[12, 13, 14, 12, 14], [14, 12, 13, 14, 12], [13, 14, 12, 12, 13], [12, 14, 14, 13, 12]]
    for k, seq in enumerate(seqs):   # inputs and oracle seals first: the threads only prove
        for i, po2 in enumerate(seq):
            oracle_proof(orc, po2, 8000 + 100 * k + i, 40 + 100 * k + i)
    ctxs = [pkg.Context(0, MAX_PO2, WIDTHS, lib=gpu_lib, deterministic=True) for _ in seqs]
    barrier = threading.Barrier(len(seqs))
    errors = [None] * len(seqs)

    def work(k):
        try:
            barrier.wait()
            prove_sequence(orc, ctxs[k], seqs[k], 8000 + 100 * k, 40 + 100 * k)
        except BaseException as e:  # re-raised on the main thread
            errors[k] = e
    try:
        th = [threading.Thread(target=work, args=(k,)) for k in range(len(seqs))]
        [t.start() for t in th]
        [t.join() for t in th]
    finally:
        [c.close() for c in ctxs]
    for e in errors:
        if e is not None:
            raise e
