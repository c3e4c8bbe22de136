"""The device witness seam: hfb200_segment_witness_dev opens a segment's DATA columns in the context's device memory and derives its
blinding key; the caller's witness generator writes the active rows (from a compact input it copies into hfb200_segment_scratch),
hfb200_segment_data_blind writes the blinding rows from the segment key, and a begin with data == NULL commits the columns as they
stand.  Pools take each job's witness from a witgen callback (hfb200_pool_set_witgen), alone or together with an accum callback.

CPU tier: the host emulator, where device addresses are host addresses and the callbacks are numpy.  GPU tier: a callback
compiled with nvcc into its own shared object (tools/witness_seam_cb.cu), which expands one 64-bit seed per column on the device."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
from conftest import SMALL, ROOT, make_segment

P = 2013265921
ZK = 1994
DATA = 2


# ---- the blinding rows and the GPU callback's expansion, in numpy ---------------------------------------------------------------

def _rotl(v, r):
    return (v << np.uint32(r)) | (v >> np.uint32(32 - r))


def blind_rows(seed, group, w, n, zk=ZK):
    """[w, zk]: blind_value(key(seed), group, col, row) for rows [n - zk, n) -- the deterministic-mode key of csrc/blind.cuh,
    the ChaCha20 block function (RFC 8439) vectorised over (col, row), six words folded mod p, Montgomery form."""
    cols = np.repeat(np.arange(w, dtype=np.uint32), zk)
    rows = np.tile(np.arange(n - zk, n, dtype=np.uint32), w)
    m = cols.size
    key = [seed & 0xFFFFFFFF, seed >> 32, 0x32626668, 0x74656430, 0x696D7265, 0x7473696E, 0x73206369, 0x64656573]
    s = [np.full(m, v, np.uint32) for v in [0x61707865, 0x3320646E, 0x79622D32, 0x6B206574] + key]
    s += [rows, np.full(m, group, np.uint32), cols, np.full(m, 0x646E6C62, np.uint32)]
    x = [a.copy() for a in s]

    def qr(a, b, c, d):
        x[a] += x[b]; x[d] = _rotl(x[d] ^ x[a], 16)
        x[c] += x[d]; x[b] = _rotl(x[b] ^ x[c], 12)
        x[a] += x[b]; x[d] = _rotl(x[d] ^ x[a], 8)
        x[c] += x[d]; x[b] = _rotl(x[b] ^ x[c], 7)
    for _ in range(10):
        qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)
        qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)
    v = np.zeros(m, np.uint64)
    for i in range(6):
        v = ((v << np.uint64(32)) + (x[i] + s[i]).astype(np.uint64)) % np.uint64(P)
    return ((v << np.uint64(32)) % np.uint64(P)).astype(np.uint32).reshape(w, zk)


def _splitmix64(z):
    z = z + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def expand_columns(seeds, po2, blind_seed):
    """What tools/witness_seam_cb.cu writes: data[c][r] = splitmix64(seeds[c] + r) mod p on the active rows, and the blinding
    rows of the segment key."""
    n = 1 << po2
    out = np.empty((len(seeds), n), np.uint32)
    r = np.arange(n - ZK, dtype=np.uint64)
    for c, s in enumerate(seeds):
        out[c, :n - ZK] = (_splitmix64(r + np.uint64(s)) % np.uint64(P)).astype(np.uint32)
    out[:, n - ZK:] = blind_rows(blind_seed, DATA, len(seeds), n)
    return out


def column_seeds(job_seed, w_data):
    return np.random.default_rng(job_seed).integers(0, 1 << 63, size=w_data, dtype=np.uint64)


# ---- numpy callbacks (host emulator) -------------------------------------------------------------------------------------------

def chain_src(r, w_data):
    return (13 * r + 5) % w_data


def numpy_accum(handle, seg, job):
    """The stand-in step_accum through the accum seam (terms, scan, blinding rows), as in test_device_accum_seam."""
    acc, data, mix = seg.host_view("accum"), seg.host_view("data"), seg.mix_array()
    rows = seg.rows - seg.zk_rows
    for r in range(seg.w_accum // 4):
        acc[4 * r, :rows] = (data[chain_src(r, seg.w_data), :rows].astype(np.uint64) + int(mix[4 * r])) % P
        for k in range(1, 4):
            acc[4 * r + k, :rows] = mix[4 * r + k]
    handle.accum_scan(0, 0, seg.w_accum // 4, rows)
    handle.accum_blind()


def witgen_from(pkg, datas):
    """A witgen callback that stages job `job`'s active rows through the context's scratch into the data columns, then lets the
    library write the blinding rows."""
    def fn(h, w, job):
        src = datas[job]
        assert src.shape == (w.w_data, w.rows) and w.zk_rows == ZK and not w.stream
        nbytes = src.size * 4
        sv = pkg.scratch_view(h.scratch(nbytes), nbytes)
        sv[:] = np.ascontiguousarray(src).view(np.uint8).ravel()
        cols = w.host_view()
        cols[...] = sv.view(np.uint32).reshape(src.shape)
        cols[:, w.rows - ZK:] = 0
        h.data_blind()
    return fn


def builtin_jobs(orc, widths, po2s, seed0):
    jobs, datas, expect = [], [], []
    for i, po2 in enumerate(po2s):
        cir, g, code, data = make_segment(orc, widths, po2, trace_seed=seed0 + i, blind_seed=seed0 + i)
        jobs.append((po2, g, code, None, seed0 + i))
        datas.append(data)
        expect.append(cir.prove(po2, g, code, data, seed0 + i)[0])
    return jobs, datas, expect


def ir_oracle(orc, ir, widths):
    cir = orc.Circuit(*widths)
    cir.set_ir(ir["taps"], ir["steps"], ir["ret"], ir.get("info"))
    return cir


# ---- CPU tier: one context ------------------------------------------------------------------------------------------------------

def test_numpy_blinding_rows_match_the_oracle(orc):
    got = blind_rows(0x1234567890AB, DATA, 3, 1 << 12)
    for c, i in [(0, 0), (1, 7), (2, ZK - 1), (1, 1000)]:
        assert got[c, i] == orc.blind_value(0x1234567890AB, DATA, c, (1 << 12) - ZK + i)


@pytest.mark.parametrize("code_mode", ["host_code", "resident_control"])
def test_builtin_circuit_through_witness_dev(pkg, emu_lib, orc, code_mode):
    po2, seed = 12, 77
    cir, g, code, data = make_segment(orc, SMALL, po2, trace_seed=seed, blind_seed=seed)
    oseal = cir.prove(po2, g, code, data, seed)[0]
    n = 1 << po2
    with pkg.Context(0, po2, SMALL, lib=emu_lib, deterministic=True) as c:
        if code_mode == "resident_control":
            root = c.control_root(po2, code)
        w = c.segment_witness_dev(po2, seed)
        assert (w.po2, w.zk_rows, w.w_code, w.w_data, w.device) == (po2, ZK, SMALL[0], SMALL[1], 0) and not w.stream
        cols = w.host_view()
        cols[...] = data
        cols[:, n - ZK:] = 0
        c.segment_data_blind()
        blind = c.read_group(DATA)[:, n - ZK:]
        assert all(blind[col, i] == orc.blind_value(seed, DATA, col, n - ZK + i) for col in range(SMALL[1]) for i in range(ZK))
        assert (blind == blind_rows(seed, DATA, SMALL[1], n)).all()
        c.segment_begin(po2, g, code if code_mode == "host_code" else None, None, seed)
        seal = c.segment_finish(None)
        assert len(seal) == len(oseal) and (seal == oseal).all()
        if code_mode == "resident_control":
            assert (root == cir.control_id(po2)).all()
            # the control group stays resident: the next segment of that po2 lays out again and reuses it
            w = c.segment_witness_dev(po2, seed)
            w.host_view()[...] = data
            c.segment_begin(po2, g, None, None, seed)
            assert (c.segment_finish(None) == oseal).all()
        assert pkg.verify_segment(seal, cir.control_id(po2), SMALL, lib=emu_lib) == po2


def test_witness_dev_then_begin_dev_and_accum_seam(pkg, emu_lib, orc):
    """begin_dev with data == NULL after witness_dev, then the accum seam: the accum blinding rows use the key of witness_dev."""
    po2, seed = 12, 91
    cir, g, code, data = make_segment(orc, SMALL, po2, trace_seed=seed, blind_seed=seed)
    oseal = cir.prove(po2, g, code, data, seed)[0]
    with pkg.Context(0, po2, SMALL, lib=emu_lib, deterministic=True) as c:
        w = c.segment_witness_dev(po2, seed)
        witgen_from(pkg, [data])(pkg.WitnessHandle(emu_lib, c._h), w, 0)
        seg = c.segment_begin_dev(po2, g, code, None, seed)
        assert (seg.host_view("data") == data).all()
        numpy_accum(pkg.SegmentHandle(emu_lib, c._h), seg, 0)
        assert (c.segment_finish_dev() == oseal).all()


def test_satisfiable_ir_through_witness_and_accum_seams(pkg, emu_lib, orc, monkeypatch):
    """A satisfiable random data-defined circuit (tests/test_ir_differential.py) whose witness is written through witness_dev:
    its blinding rows, which the circuit's taps at back > 0 read from the first active rows, are the segment key's."""
    import test_ir_differential as tid
    seed, widths, n_out = tid.SAT_CASES[0]
    po2, blind = 12, 9
    real_rng = np.random.default_rng

    class KeyedBlindingRng:   # the witness generator's random columns, with the blinding rows data_blind will write
        def __init__(self, s):
            self._r = real_rng(s)

        def integers(self, *a, **k):
            out = self._r.integers(*a, **k)
            out[:, out.shape[1] - ZK:] = blind_rows(blind, DATA, out.shape[0], out.shape[1])
            return out
    with monkeypatch.context() as m:
        m.setattr(np.random, "default_rng", KeyedBlindingRng)
        ir, g, code, data = tid.satisfiable_ir(seed, widths, po2, n_out, n_cons=70)
    cir = ir_oracle(orc, ir, widths)
    oseal = cir.prove(po2, g, code, data, blind)[0]
    with pkg.Context(0, po2, widths, lib=emu_lib, ir=ir, deterministic=True) as c:
        w = c.segment_witness_dev(po2, blind)
        witgen_from(pkg, [data])(pkg.WitnessHandle(emu_lib, c._h), w, 0)
        seg = c.segment_begin_dev(po2, g, code, None, blind)
        numpy_accum(pkg.SegmentHandle(emu_lib, c._h), seg, 0)
        seal = c.segment_finish_dev()
    assert len(seal) == len(oseal) and (seal == oseal).all()
    root = cir.control_id(po2)
    assert cir.verify(seal, root) == po2
    assert pkg.verify_segment(seal, root, widths, ir=ir, lib=emu_lib) == po2


def test_refusals(pkg, emu_lib, orc):
    po2 = 12
    cir, g, code, data = make_segment(orc, SMALL, po2)
    oseal = cir.prove(po2, g, code, data, 1)[0]
    with pkg.Context(0, po2, SMALL, lib=emu_lib, deterministic=True) as c:
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_data_blind()
        assert str(e.value) == "hfb200_segment_data_blind: no witness open (call hfb200_segment_witness_dev)"
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_scratch(64)
        assert str(e.value) == "hfb200_segment_scratch: no witness open (call hfb200_segment_witness_dev)"
        for bad in (11, 13, 23):
            with pytest.raises(pkg.Hfb200Error) as e:
                c.segment_witness_dev(bad, 1)
            assert str(e.value) == "hfb200_segment_witness_dev: po2 %d outside [12, 12]" % bad
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_begin(po2, g, code, None, 1)   # no witness open, no resident trace: today's refusal
        assert str(e.value).startswith("no trace: pass code/data")

        w = c.segment_witness_dev(po2, 1)
        w.host_view()[...] = data
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_begin(po2, g, code, None, 2)
        assert str(e.value) == "blind_seed 2 differs from the one of hfb200_segment_witness_dev (1)"
        with pytest.raises(pkg.Hfb200Error):
            c.segment_data_blind()                   # the refusal abandoned the witness

        c.segment_witness_dev(po2, 1)
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_begin(po2, g, None, None, 1)
        assert str(e.value) == "code is NULL and no control group is resident for this po2 (hfb200_control_root)"

        w = c.segment_witness_dev(po2, 1)            # the columns are still the ones written above
        c.segment_begin(po2, g, code, None, 1)
        assert (c.segment_finish(None) == oseal).all()
        assert (c.prove_segment(po2, g, code, data, 1) == oseal).all()   # host inputs after the seam: unchanged
    e = emu_lib.hfb200_segment_witness_dev(None, 12, 1, C.byref(pkg.WitnessDev()))
    with pytest.raises(pkg.Hfb200Error, match="^hfb200_segment_witness_dev: NULL argument$"):
        pkg.binding._raise_err(emu_lib, e)


def test_scratch_grows_only(pkg, emu_lib):
    with pkg.Context(0, 12, SMALL, lib=emu_lib, deterministic=True) as c:
        c.segment_witness_dev(12, 1)
        a = c.segment_scratch(1 << 12)
        assert a and c.segment_scratch(100) == a and c.segment_scratch(1 << 12) == a
        b = c.segment_scratch(1 << 20)
        pkg.scratch_view(b, 1 << 20)[:] = 7     # the whole request is usable
        c.segment_witness_dev(12, 2)
        assert c.segment_scratch(1 << 16) == b   # kept across segments


def square_ir():
    """code[0] * (data[1] - data[0]^2) = 0, every tap at back 0: a witness written before its blinding rows are known satisfies
    it (the stand-in circuit reads a blinding row at row 0 through a back-1 tap, so its witness needs the key's rows first)."""
    GET, SUB, MUL, TRUE, EQZ = 1, 4, 5, 6, 7
    taps = [(1, 0, 0), (DATA, 0, 0), (DATA, 1, 0)]
    steps = [(GET, 0, 0, 0), (GET, 1, 0, 0), (GET, 2, 0, 0), (MUL, 1, 1, 0), (SUB, 2, 3, 0), (MUL, 0, 4, 0), (TRUE, 0, 0, 0), (EQZ, 0, 5, 0)]
    return {"taps": np.array(taps, np.uint32), "steps": np.array(steps, np.uint32), "ret": 1, "n_mix": SMALL[2], "widths": SMALL, "info": None}


def test_os_entropy_blinding_differs_per_segment(pkg, emu_lib, orc):
    """Without the deterministic mode the key comes from the OS at witness_dev: the same job proved twice gets other DATA
    blinding rows and another seal, and both seals verify."""
    po2, seed = 12, 5
    n = 1 << po2
    ir = square_ir()
    cir = ir_oracle(orc, ir, SMALL)
    code, g = cir.gen_code(po2), cir.gen_globals(seed)
    data = np.random.default_rng(seed).integers(0, P, size=(SMALL[1], n), dtype=np.uint32)
    data[1] = orc.encode(orc.decode(data[0]).astype(np.uint64) ** 2 % P)
    rows, seals = [], []
    with pkg.Context(0, po2, SMALL, lib=emu_lib, ir=ir, deterministic=False) as c:
        for _ in range(2):
            w = c.segment_witness_dev(po2, seed)
            w.host_view()[...] = data
            c.segment_data_blind()
            rows.append(c.read_group(DATA)[:, n - ZK:].copy())
            seg = c.segment_begin_dev(po2, g, code, None, seed)
            numpy_accum(pkg.SegmentHandle(emu_lib, c._h), seg, 0)
            seals.append(c.segment_finish_dev())
    assert (rows[0] != rows[1]).mean() > 0.99
    assert (rows[0] != blind_rows(seed, DATA, SMALL[1], n)).mean() > 0.99
    assert len(seals[0]) == len(seals[1]) and not (seals[0] == seals[1]).all()
    for s in seals:
        assert pkg.verify_segment(s, cir.control_id(po2), SMALL, ir=ir, lib=emu_lib) == po2
        assert cir.verify(s, cir.control_id(po2)) == po2


# ---- CPU tier: pools ------------------------------------------------------------------------------------------------------------

def test_builtin_pool_with_python_witgen(pkg, emu_lib, orc):
    jobs, datas, expect = builtin_jobs(orc, SMALL, [12, 13, 12, 13, 12], 900)
    cap = orc.Circuit(*SMALL).seal_words_model(13)
    calls = []
    with pkg.Pool(devices=(0, 0), contexts_per_device=1, max_po2=13, circuit=SMALL, lib=emu_lib, deterministic=True) as pool:
        _, _, _, errs = pool.prove(jobs[:1], cap, return_errors=True)
        assert errs[0] == "job has a NULL globals / data / seal_out pointer"   # no witgen callback: today's refusal

        gen = witgen_from(pkg, datas)

        def witgen(h, w, job):
            calls.append(job)
            assert w.po2 == jobs[job][0]
            gen(h, w, job)
        pool.set_witgen(witgen)
        # witgen jobs beside a job with host columns, in one call
        mixed = jobs + [(12, jobs[0][1], jobs[0][2], datas[0], jobs[0][4])]
        seals, devs, _ = pool.prove(mixed, cap)
        assert sorted(calls) == list(range(len(jobs)))
        for i, (a, b) in enumerate(zip(seals, expect + expect[:1])):
            assert len(a) == len(b) and (a == b).all(), i
        assert pool.last_attempts == [1] * len(mixed)
        # shared control group
        pool.load_control(12, jobs[0][2])
        shared = [(po2, g, None if po2 == 12 else code, d, s) for po2, g, code, d, s in jobs]
        seals, _, _ = pool.prove(shared, cap)
        assert all((a == b).all() for a, b in zip(seals, expect))
        pool.set_witgen(None)
        _, _, _, errs = pool.prove(jobs[:1], cap, return_errors=True)
        assert errs[0] == "job has a NULL globals / data / seal_out pointer"


def test_ir_pool_with_witgen_and_accum(pkg, emu_lib, orc):
    from oracle import synth_ir
    ir = synth_ir.build(SMALL, 0)
    cir_ir = ir_oracle(orc, ir, SMALL)
    jobs, datas, _ = builtin_jobs(orc, SMALL, [13, 12, 13, 12], 950)
    expect = [cir_ir.prove(po2, g, code, d, s)[0] for (po2, g, code, _, s), d in zip(jobs, datas)]
    cap = cir_ir.seal_words_model(13)
    with pkg.Pool(devices=(0, 0), contexts_per_device=1, max_po2=13, circuit=SMALL, lib=emu_lib, ir=ir, deterministic=True) as pool:
        pool.set_witgen(witgen_from(pkg, datas))
        _, _, _, errs = pool.prove(jobs[:1], cap, return_errors=True)
        assert "step_accum is the caller's" in errs[0]   # a data-defined circuit still needs the caller's step_accum
        pool.set_accum(numpy_accum)
        pool.load_control(13, jobs[0][2])
        shared = [(po2, g, None if po2 == 13 else code, d, s) for po2, g, code, d, s in jobs]
        seals, _, _ = pool.prove(shared, cap)
        for i, (a, b) in enumerate(zip(seals, expect)):
            assert len(a) == len(b) and (a == b).all(), i
            assert cir_ir.verify(a, cir_ir.control_id(jobs[i][0])) == jobs[i][0]


def test_failing_witgen_fails_its_job_only(pkg, emu_lib, orc):
    jobs, datas, expect = builtin_jobs(orc, SMALL, [12, 12, 12, 12], 1000)
    cap = orc.Circuit(*SMALL).seal_words_model(12)
    gen = witgen_from(pkg, datas)
    with pkg.Pool(devices=(0,), contexts_per_device=1, max_po2=12, circuit=SMALL, lib=emu_lib, deterministic=True) as pool:
        def witgen(h, w, job):
            if job == 2:
                h.data_blind()                    # work already queued when the callback gives up
                raise ValueError("no preflight trace for job 2")
            gen(h, w, job)
        pool.set_witgen(witgen)
        seals, _, _, errs = pool.prove(jobs, cap, return_errors=True)
        assert errs[2] == "witgen callback returned 1: ValueError: no preflight trace for job 2"
        assert [e for i, e in enumerate(errs) if i != 2] == [None] * 3
        for i in (0, 1, 3):
            assert (seals[i] == expect[i]).all()
        assert pool.last_attempts[2] == 1 and pool.stats()["retries"] == 0
        with pytest.raises(pkg.Hfb200Error, match="^job 2: witgen callback returned 1: ValueError: no preflight trace for job 2$"):
            pool.prove(jobs, cap)
        pool.set_witgen(gen)                      # the same (single) context proves correctly afterwards
        seals, _, _ = pool.prove(jobs, cap)
        assert all((a == b).all() for a, b in zip(seals, expect))


def test_device_fault_reruns_the_witgen_callback(pkg, emu_lib, orc):
    jobs, datas, expect = builtin_jobs(orc, SMALL, [12, 12, 12], 1100)
    gen = witgen_from(pkg, datas)
    calls = {}
    with pkg.Pool(devices=(0,), contexts_per_device=1, max_po2=12, circuit=SMALL, lib=emu_lib, deterministic=True) as pool:
        def witgen(h, w, job):
            calls[job] = calls.get(job, 0) + 1
            gen(h, w, job)
        pool.set_witgen(witgen)
        pool.inject_fault(0, 1, 0)                # the worker proves one job, then its context "faults" on the next
        seals, _, _ = pool.prove(jobs, cap := orc.Circuit(*SMALL).seal_words_model(12))
        assert sorted(pool.last_attempts) == [1, 1, 2]
        st = pool.stats()
        assert st["faults"] == 1 and st["retries"] == 1 and st["contexts_recreated"] == 1
        retried = pool.last_attempts.index(2)     # its callback ran on the re-created context
        assert calls[retried] == 1 and sum(calls.values()) == 3
        assert all((a == b).all() for a, b in zip(seals, expect))
        seals, _, _ = pool.prove(jobs, cap)
        assert all((a == b).all() for a, b in zip(seals, expect))


# ---- GPU tier -------------------------------------------------------------------------------------------------------------------

class SeamInput(C.Structure):
    """witness_seam_input of tools/witness_seam_cb.cu."""
    _fields_ = [("seeds", C.c_void_p), ("w_data", C.c_uint32), ("calls", C.c_int)]


@pytest.fixture(scope="module")
def seam_cbs(pkg, tmp_path_factory):
    """tools/witness_seam_cb.cu and tools/accum_seam_cb.cu, compiled for sm_100a into their own shared objects."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    d = tmp_path_factory.mktemp("witness_seam_cb")
    libdir = os.path.dirname(pkg.LIB_PATH)
    libs = {}
    for name in ("witness_seam_cb", "accum_seam_cb"):
        so = d / ("lib%s.so" % name)
        subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-Xcompiler", "-fPIC", "-shared",
                               "-I", os.path.join(ROOT, "include"), "-o", str(so), os.path.join(ROOT, "tools", name + ".cu"),
                               "-L", libdir, "-l:libhfb200.so", "-Xlinker", "-rpath," + libdir])
        libs[name] = C.CDLL(str(so))
    libs["witness_seam_cb"].seam_witgen.restype = C.c_int
    libs["witness_seam_cb"].seam_witgen.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(pkg.WitnessDev), C.c_size_t]
    libs["accum_seam_cb"].seam_accum.restype = C.c_int
    libs["accum_seam_cb"].seam_accum.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(pkg.SegmentDev), C.c_size_t]
    return libs["witness_seam_cb"], libs["accum_seam_cb"]


class PinnedSeeds:
    """One row of column seeds per job in pinned host memory (hfb200_host_alloc), described by a SeamInput."""

    def __init__(self, pkg, lib, rows):
        rows = np.asarray(rows, np.uint64)
        self.lib, self.p = lib, C.c_void_p()
        pkg.binding._raise_err(lib, lib.hfb200_host_alloc(rows.nbytes, C.byref(self.p)))
        arr = np.ctypeslib.as_array(C.cast(self.p, C.POINTER(C.c_uint64)), shape=(rows.size,)).reshape(rows.shape)
        arr[...] = rows
        self.input = SeamInput(self.p.value, rows.shape[1], 0)

    def close(self):
        self.lib.hfb200_host_free(self.p)


def _gpu_jobs(orc, widths, po2s, seed0, host=True):
    """(jobs with data None, host columns of the same witness, column seeds); code / globals of the oracle's stand-in."""
    cir = orc.Circuit(*widths)
    jobs, cols, seeds = [], [], []
    for i, po2 in enumerate(po2s):
        s = column_seeds(seed0 + i, widths[1])
        jobs.append((po2, cir.gen_globals(seed0 + i), cir.gen_code(po2), None, seed0 + i))
        cols.append(expand_columns(s, po2, seed0 + i) if host else None)
        seeds.append(s)
    return jobs, cols, seeds


GPU_WIDTHS = (16, 64, 16)
GPU_PO2S = [13, 14, 15, 16]


@pytest.fixture(scope="module")
def gpu_cases(orc):
    """Built-in and data-defined circuits at po2 13-16: jobs, host columns and the oracle's seals of those columns."""
    from oracle import synth_ir
    ir = synth_ir.build(GPU_WIDTHS, 0)
    jobs, cols, seeds = _gpu_jobs(orc, GPU_WIDTHS, GPU_PO2S, 1200)
    builtin, cir_ir = orc.Circuit(*GPU_WIDTHS), ir_oracle(orc, ir, GPU_WIDTHS)
    expect = {"builtin": [], "ir": []}
    for (po2, g, code, _, s), d in zip(jobs, cols):
        expect["builtin"].append(builtin.prove(po2, g, code, d, s)[0])
        expect["ir"].append(cir_ir.prove(po2, g, code, d, s)[0])
    return {"ir": ir, "jobs": jobs, "cols": cols, "seeds": seeds, "expect": expect}


@pytest.mark.gpu
def test_c_witgen_through_context_on_gpu(pkg, gpu_lib, seam_cbs, gpu_cases):
    wit, acc = seam_cbs
    jobs, cols, expect = gpu_cases["jobs"], gpu_cases["cols"], gpu_cases["expect"]
    seeds = PinnedSeeds(pkg, gpu_lib, gpu_cases["seeds"])
    try:
        with pkg.Context(0, max(GPU_PO2S), GPU_WIDTHS, lib=gpu_lib, deterministic=True) as c:
            for j, (po2, g, code, _, s) in enumerate(jobs):
                w = c.segment_witness_dev(po2, s)
                assert w.stream and w.device == 0 and w.po2 == po2
                assert wit.seam_witgen(C.byref(seeds.input), c._h, C.byref(w), j) == 0
                if j == 0:
                    assert (c.read_group(DATA) == cols[j]).all()   # the device expansion and the key's blinding rows
                c.segment_begin(po2, g, code, None, s)
                seal = c.segment_finish(None)
                assert len(seal) == len(expect["builtin"][j]) and (seal == expect["builtin"][j]).all(), po2
        with pkg.Context(0, max(GPU_PO2S), GPU_WIDTHS, lib=gpu_lib, ir=gpu_cases["ir"], deterministic=True) as c:
            for j, (po2, g, code, _, s) in enumerate(jobs):
                w = c.segment_witness_dev(po2, s)
                assert wit.seam_witgen(C.byref(seeds.input), c._h, C.byref(w), j) == 0
                seg = c.segment_begin_dev(po2, g, code, None, s)
                assert acc.seam_accum(None, c._h, C.byref(seg), j) == 0
                seal = c.segment_finish_dev()
                assert len(seal) == len(expect["ir"][j]) and (seal == expect["ir"][j]).all(), po2
        assert seeds.input.calls == 2 * len(jobs)
    finally:
        seeds.close()


@pytest.mark.gpu
def test_pools_with_c_witgen_on_every_device(pkg, gpu_lib, seam_cbs, gpu_cases):
    wit, acc = seam_cbs
    ndev = pkg.device_count(gpu_lib)
    assert ndev >= 1
    jobs, expect = gpu_cases["jobs"] * 2, {k: v * 2 for k, v in gpu_cases["expect"].items()}
    seeds = PinnedSeeds(pkg, gpu_lib, gpu_cases["seeds"] * 2)
    wfn, afn = C.cast(wit.seam_witgen, C.c_void_p).value, C.cast(acc.seam_accum, C.c_void_p).value
    try:
        for kind in ("builtin", "ir"):
            ir = gpu_cases["ir"] if kind == "ir" else None
            with pkg.Pool(devices=tuple(range(ndev)), contexts_per_device=2, max_po2=max(GPU_PO2S), circuit=GPU_WIDTHS, lib=gpu_lib,
                          ir=ir, deterministic=True) as pool:
                pool.set_witgen(wfn, C.addressof(seeds.input))
                if kind == "ir":
                    pool.set_accum(afn)
                pool.load_control(14, jobs[1][2])
                shared = [(po2, g, None if po2 == 14 else code, d, s) for po2, g, code, d, s in jobs]
                before = seeds.input.calls
                seals, devs, _ = pool.prove(shared, 1 << 20)
                assert seeds.input.calls - before == len(jobs) and set(devs) <= set(range(ndev))
                for i, (a, b) in enumerate(zip(seals, expect[kind])):
                    assert len(a) == len(b) and (a == b).all(), (kind, i)
    finally:
        seeds.close()


@pytest.mark.gpu
def test_witgen_pool_equals_host_buffer_pool_at_po2_20(pkg, gpu_lib, orc, seam_cbs):
    """W = 256 (the declared shape), po2 20: jobs through the witgen callback give the seals of jobs carrying the same columns
    from host memory, in one pool call over every device."""
    wit, _ = seam_cbs
    ndev = pkg.device_count(gpu_lib)
    widths = (16, 192, 48)
    jobs, cols, seeds_rows = _gpu_jobs(orc, widths, [20, 20], 1300)
    seeds = PinnedSeeds(pkg, gpu_lib, seeds_rows)
    try:
        with pkg.Pool(devices=tuple(range(ndev)), contexts_per_device=2, max_po2=20, circuit=widths, lib=gpu_lib, deterministic=True) as pool:
            pool.set_witgen(C.cast(wit.seam_witgen, C.c_void_p).value, C.addressof(seeds.input))
            host = [(po2, g, code, d, s) for (po2, g, code, _, s), d in zip(jobs, cols)]
            seals, _, _ = pool.prove(jobs + host, 1 << 22)
        assert seeds.input.calls == len(jobs)
        for i in range(len(jobs)):
            assert len(seals[i]) == len(seals[len(jobs) + i]) and (seals[i] == seals[len(jobs) + i]).all(), i
    finally:
        seeds.close()


@pytest.mark.gpu
def test_both_callbacks_at_rv32im_scale_on_gpu(pkg, gpu_lib, orc, seam_cbs):
    """build_scaled(560): W = 400 (24 / 320 / 56), po2 20, on every device with a shared control group.  The witgen + accum
    callback job gives the seal of the host-buffer, accum-callback job for the same columns."""
    from oracle import synth_ir
    wit, acc = seam_cbs
    ndev = pkg.device_count(gpu_lib)
    ir = synth_ir.build_scaled(n_groups=560)
    W = ir["widths"]
    jobs, cols, seeds_rows = _gpu_jobs(orc, W, [20], 1400)
    seeds = PinnedSeeds(pkg, gpu_lib, seeds_rows)
    try:
        with pkg.Pool(devices=tuple(range(ndev)), contexts_per_device=1, max_po2=20, circuit=W, lib=gpu_lib, ir=ir, deterministic=True) as pool:
            pool.set_witgen(C.cast(wit.seam_witgen, C.c_void_p).value, C.addressof(seeds.input))
            pool.set_accum(C.cast(acc.seam_accum, C.c_void_p).value)
            po2, g, code, _, s = jobs[0]
            pool.load_control(po2, code)
            seals, _, _ = pool.prove([(po2, g, None, None, s), (po2, g, None, cols[0], s)], 1 << 22)
        assert seeds.input.calls == 1
        assert len(seals[0]) == len(seals[1]) and (seals[0] == seals[1]).all()
    finally:
        seeds.close()
