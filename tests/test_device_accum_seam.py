"""The device seam of the two-phase prover: hfb200_segment_begin_dev hands the caller the committed columns, the mix and the
writable accum columns in device memory; the caller's step_accum (its own term kernel, then hfb200_segment_accum_scan and
hfb200_segment_accum_blind) fills them in place; hfb200_segment_finish_dev commits them.  Pools carry data-defined circuits
through an accum callback (hfb200_pool_set_accum).

CPU tier: the host emulator, where device addresses are host addresses and the callbacks are numpy.  GPU tier: a callback
compiled with nvcc into its own shared object, running its term kernel on the context's stream."""
import ctypes as C
import os
import shutil
import subprocess
import numpy as np
import pytest
from conftest import SMALL, ROOT, make_segment

P = 2013265921
ZK = 1994


def chain_src(r, w_data):
    """Column the stand-in circuit's chain r accumulates (oracle/circuit.h chain_src)."""
    return (13 * r + 5) % w_data


def write_terms(seg):
    """The stand-in step_accum's terms data[chain_src(r)] + mix_r on the active rows, in the emulator's accum columns."""
    acc, data, mix = seg.host_view("accum"), seg.host_view("data"), seg.mix_array()
    rows = seg.rows - seg.zk_rows
    for r in range(seg.w_accum // 4):
        acc[4 * r, :rows] = (data[chain_src(r, seg.w_data), :rows].astype(np.uint64) + int(mix[4 * r])) % P
        for k in range(1, 4):
            acc[4 * r + k, :rows] = mix[4 * r + k]
    return rows


def numpy_accum(handle, seg, job):
    rows = write_terms(seg)
    handle.accum_scan(0, 0, seg.w_accum // 4, rows)   # HFB200_SCAN_PRODUCT
    handle.accum_blind()


def ir_segment(orc, widths, po2, seed):
    cir, g, code, data = make_segment(orc, widths, po2, trace_seed=seed, blind_seed=seed)
    return g, code, data


def ir_oracle(orc, ir, widths):
    cir_ir = orc.Circuit(*widths)
    cir_ir.set_ir(ir["taps"], ir["steps"], ir["ret"], ir.get("info"))
    return cir_ir


# ---- CPU tier -------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("device_inputs", [False, True])
def test_builtin_circuit_through_the_device_seam(pkg, emu_lib, orc, device_inputs):
    po2 = 12
    cir, g, code, data = make_segment(orc, SMALL, po2)
    oseal = cir.prove(po2, g, code, data, 1)[0]
    with pkg.Context(0, po2, SMALL, lib=emu_lib, deterministic=True) as c:
        if device_inputs:   # the emulator's "device" addresses are host addresses: this runs the device-to-device copy path
            seg = c.segment_begin_dev(po2, g, code.ctypes.data, data.ctypes.data, 1, device_inputs=True)
        else:
            seg = c.segment_begin_dev(po2, g, code, data, 1)
        assert (seg.po2, seg.zk_rows, seg.w_code, seg.w_data, seg.w_accum, seg.n_mix) == (po2, ZK, *SMALL, SMALL[2])
        assert seg.blind_seed == 1 and seg.device == 0 and not seg.stream
        assert (seg.globals_array() == g).all() and (seg.host_view("data") == data).all() and (seg.host_view("code") == code).all()
        mix = seg.mix_array()
        rows = write_terms(seg)
        c.segment_accum_scan(pkg.SCAN_PRODUCT, 0, SMALL[2] // 4, rows)
        c.segment_accum_blind()
        accum = seg.host_view("accum").copy()
        seal = c.segment_finish_dev()
        assert len(seal) == len(oseal) and (seal == oseal).all()
        assert (accum == cir.step_accum(po2, data, mix, 1)).all()
        # either finish follows either begin: begin_dev + the built-in step_accum, begin (host) + finish_dev
        c.segment_begin_dev(po2, g, code, data, 1)
        assert (c.segment_finish(None) == oseal).all()
        c.segment_begin(po2, g, code, data, 1)
        seg2 = c.segment_begin_dev(po2, g, code, data, 1)   # a second begin restarts the segment
        numpy_accum(pkg.SegmentHandle(emu_lib, c._h), seg2, 0)
        assert (c.segment_finish_dev() == oseal).all()


def test_accum_scan_sum_is_a_running_sum(pkg, emu_lib, orc):
    """SCAN_SUM over random Fp4 columns equals numpy's running sum mod p; other chains and rows past `rows` stay untouched.
    rows spans several scan blocks (2048 rows each) and ends inside one."""
    po2, widths = 13, (8, 16, 16)
    cir, g, code, data = make_segment(orc, widths, po2)
    rng = np.random.default_rng(5)
    with pkg.Context(0, po2, widths, lib=emu_lib, deterministic=True) as c:
        seg = c.segment_begin_dev(po2, g, code, data, 1)
        acc = seg.host_view("accum")
        acc[...] = rng.integers(0, P, size=acc.shape, dtype=np.uint32)
        before = acc.copy()
        rows = 5000
        c.segment_accum_scan(pkg.SCAN_SUM, 1, 2, rows)
        expect = before.copy()
        expect[4:12, :rows] = (np.cumsum(before[4:12, :rows].astype(np.uint64), axis=1) % P).astype(np.uint32)
        assert (acc == expect).all()
        c.segment_accum_scan(pkg.SCAN_SUM, 0, 1, 0)       # empty range: nothing happens
        assert (acc == expect).all()
        c.segment_finish_dev()


def test_refusals(pkg, emu_lib, orc):
    po2 = 12
    cir, g, code, data = make_segment(orc, SMALL, po2)
    with pkg.Context(0, po2, SMALL, lib=emu_lib, deterministic=True) as c:
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_finish_dev()
        assert str(e.value) == "hfb200_segment_finish_dev: no segment in flight"
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_accum_scan(0, 0, 1, 10)
        assert str(e.value) == "hfb200_segment_accum_scan: no segment in flight"
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_accum_blind()
        assert str(e.value) == "hfb200_segment_accum_blind: no segment in flight"
        seg = c.segment_begin_dev(po2, g, code, data, 1)
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_accum_scan(0, 1, 2, 10)
        assert str(e.value) == "hfb200_segment_accum_scan: chains [1, 3) beyond w_accum / 4 = 2"
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_accum_scan(0, 0, 1, (1 << po2) + 1)
        assert str(e.value) == "hfb200_segment_accum_scan: rows 4097 > N = 4096"
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_accum_scan(2, 0, 1, 10)
        assert str(e.value) == "hfb200_segment_accum_scan: kind must be HFB200_SCAN_PRODUCT (0) or HFB200_SCAN_SUM (1)"
        numpy_accum(pkg.SegmentHandle(emu_lib, c._h), seg, 0)   # refused calls left the segment in flight
        assert (c.segment_finish_dev() == cir.prove(po2, g, code, data, 1)[0]).all()
        e = emu_lib.hfb200_segment_begin_dev(c._h, po2, g.ctypes.data, code.ctypes.data, data.ctypes.data, 1, 2, C.byref(pkg.SegmentDev()))
        with pytest.raises(pkg.Hfb200Error, match="^hfb200_segment_begin_dev: unknown flags$"):
            c._check(e)


def _ir_jobs(orc, cir_ir, widths, po2s, seed0):
    jobs, expect = [], []
    for i, po2 in enumerate(po2s):
        g, code, data = ir_segment(orc, widths, po2, seed0 + i)
        jobs.append((po2, g, code, data, seed0 + i))
        expect.append(cir_ir.prove(po2, g, code, data, seed0 + i)[0])
    return jobs, expect


def test_ir_pool_with_python_accum(pkg, emu_lib, orc):
    """A pool over a data-defined circuit proves once it has an accum callback; without one it refuses as before."""
    from oracle import synth_ir
    ir = synth_ir.build(SMALL, 0)
    cir_ir = ir_oracle(orc, ir, SMALL)
    jobs, expect = _ir_jobs(orc, cir_ir, SMALL, [12, 13, 12, 13, 12, 12], 300)
    cap = cir_ir.seal_words_model(13)
    calls = []
    with pkg.Pool(devices=(0, 0), contexts_per_device=1, max_po2=13, circuit=SMALL, lib=emu_lib, ir=ir, deterministic=True) as pool:
        _, _, _, errs = pool.prove(jobs[:1], cap, return_errors=True)
        assert "step_accum is the caller's" in errs[0]

        def accum(h, seg, job):
            calls.append(job)
            assert seg.po2 == jobs[job][0] and (seg.mix_array() != 0).any()
            numpy_accum(h, seg, job)
        pool.set_accum(accum)
        seals, devs, _ = pool.prove(jobs, cap)
        assert sorted(calls) == list(range(len(jobs)))
        for i, (a, b) in enumerate(zip(seals, expect)):
            assert len(a) == len(b) and (a == b).all(), i
            assert cir_ir.verify(a, cir_ir.control_id(jobs[i][0])) == jobs[i][0]
        assert pool.last_attempts == [1] * len(jobs)
        pool.set_accum(None)
        _, _, _, errs = pool.prove(jobs[:1], cap, return_errors=True)
        assert "step_accum is the caller's" in errs[0]


def test_failing_callback_fails_its_job_only(pkg, emu_lib, orc):
    from oracle import synth_ir
    ir = synth_ir.build(SMALL, 0)
    cir_ir = ir_oracle(orc, ir, SMALL)
    jobs, expect = _ir_jobs(orc, cir_ir, SMALL, [12, 12, 12, 12], 400)
    cap = cir_ir.seal_words_model(12)
    with pkg.Pool(devices=(0,), contexts_per_device=1, max_po2=12, circuit=SMALL, lib=emu_lib, ir=ir, deterministic=True) as pool:
        def accum(h, seg, job):
            if job == 2:
                h.accum_scan(0, 0, 1, seg.rows)               # work already queued when the callback gives up
                raise ValueError("no witness for job 2")
            numpy_accum(h, seg, job)
        pool.set_accum(accum)
        seals, _, _, errs = pool.prove(jobs, cap, return_errors=True)
        assert errs[2] == "accum callback returned 1: ValueError: no witness for job 2"
        assert [e for i, e in enumerate(errs) if i != 2] == [None] * 3
        for i in (0, 1, 3):
            assert (seals[i] == expect[i]).all()
        assert pool.last_attempts[2] == 1 and pool.stats()["retries"] == 0
        with pytest.raises(pkg.Hfb200Error, match="^job 2: accum callback returned 1: ValueError: no witness for job 2$"):
            pool.prove(jobs, cap)
        pool.set_accum(numpy_accum)                              # the same (single) context proves correctly afterwards
        seals, _, _ = pool.prove(jobs, cap)
        assert all((a == b).all() for a, b in zip(seals, expect))
        # a callback that calls the scan with bad arguments: the library's refusal is the job's error
        pool.set_accum(lambda h, seg, job: h.accum_scan(0, 0, 99, seg.rows))
        _, _, _, errs = pool.prove(jobs[:1], cap, return_errors=True)
        assert errs[0] == "accum callback returned 1: Hfb200Error: hfb200_segment_accum_scan: chains [0, 99) beyond w_accum / 4 = 2"


def test_device_fault_reruns_the_callback(pkg, emu_lib, orc):
    from oracle import synth_ir
    ir = synth_ir.build(SMALL, 0)
    cir_ir = ir_oracle(orc, ir, SMALL)
    jobs, expect = _ir_jobs(orc, cir_ir, SMALL, [12, 12, 12], 500)
    calls = {}
    with pkg.Pool(devices=(0,), contexts_per_device=1, max_po2=12, circuit=SMALL, lib=emu_lib, ir=ir, deterministic=True) as pool:
        def accum(h, seg, job):
            calls[job] = calls.get(job, 0) + 1
            numpy_accum(h, seg, job)
        pool.set_accum(accum)
        pool.inject_fault(0, 1, 0)           # the worker proves one job, then its context "faults" on the next
        seals, _, _ = pool.prove(jobs, cap := cir_ir.seal_words_model(12))
        assert sorted(pool.last_attempts) == [1, 1, 2]
        st = pool.stats()
        assert st["faults"] == 1 and st["retries"] == 1 and st["contexts_recreated"] == 1
        # the injected fault hits before begin_dev: the re-queued job runs the callback on the re-created context
        retried = pool.last_attempts.index(2)
        assert calls[retried] == 1 and sum(calls.values()) == 3
        for a, b in zip(seals, expect):
            assert (a == b).all()
        seals, _, _ = pool.prove(jobs, cap)
        assert all((a == b).all() for a, b in zip(seals, expect))


def test_shared_control_group_with_accum(pkg, emu_lib, orc):
    from oracle import synth_ir
    ir = synth_ir.build(SMALL, 0)
    cir_ir = ir_oracle(orc, ir, SMALL)
    jobs, expect = _ir_jobs(orc, cir_ir, SMALL, [12, 12, 13, 12], 600)
    with pkg.Pool(devices=(0, 0), contexts_per_device=1, max_po2=13, circuit=SMALL, lib=emu_lib, ir=ir, deterministic=True) as pool:
        pool.set_accum(numpy_accum)
        pool.load_control(12, jobs[0][2])
        shared = [(po2, g, None if po2 == 12 else code, data, s) for po2, g, code, data, s in jobs]
        seals, _, _ = pool.prove(shared, cir_ir.seal_words_model(13))
        for a, b in zip(seals, expect):
            assert (a == b).all()


def test_builtin_pool_with_accum_replaces_the_builtin_step_accum(pkg, emu_lib, orc):
    jobs, expect = [], []
    for i in range(3):
        cir, g, code, data = make_segment(orc, SMALL, 12, trace_seed=700 + i, blind_seed=700 + i)
        jobs.append((12, g, code, data, 700 + i))
        expect.append(cir.prove(12, g, code, data, 700 + i)[0])
    calls = []
    with pkg.Pool(devices=(0,), contexts_per_device=1, max_po2=12, circuit=SMALL, lib=emu_lib, deterministic=True) as pool:
        pool.set_accum(lambda h, seg, job: (calls.append(job), numpy_accum(h, seg, job)))
        seals, _, _ = pool.prove(jobs, 40000)
        assert sorted(calls) == [0, 1, 2] and all((a == b).all() for a, b in zip(seals, expect))


def test_device_count(pkg, emu_lib):
    """A count is a query: without a device the sm_100a library reports 0 instead of failing (the GPU tier asserts >= 1)."""
    assert pkg.device_count(emu_lib) == 1
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert pkg.device_count() == 0


# ---- GPU tier -------------------------------------------------------------------------------------------------------------

CALLBACK_CU = os.path.join(ROOT, "tools", "accum_seam_cb.cu")  # the term kernel + exported callback, outside libhfb200


@pytest.fixture(scope="module")
def seam_cb(pkg, tmp_path_factory):
    """The callback above, compiled for sm_100a into its own shared object linked against the built libhfb200.so."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    d = tmp_path_factory.mktemp("seam_cb")
    so = d / "libseam_cb.so"
    libdir = os.path.dirname(pkg.LIB_PATH)
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-Xcompiler", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"),
                           "-o", str(so), CALLBACK_CU, "-L", libdir, "-l:libhfb200.so", "-Xlinker", "-rpath," + libdir])
    lib = C.CDLL(str(so))
    lib.seam_accum.restype = C.c_int
    lib.seam_accum.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(pkg.SegmentDev), C.c_size_t]
    return lib


def _run_cb(cb, ctx, seg):
    counter = C.c_int(0)
    assert cb.seam_accum(C.byref(counter), ctx._h, C.byref(seg), 0) == 0 and counter.value == 1


@pytest.mark.gpu
def test_c_callback_through_context_on_gpu(pkg, gpu_lib, orc, seam_cb):
    import torch
    from oracle import synth_ir
    po2 = 12
    cir, g, code, data = make_segment(orc, SMALL, po2)
    oseal = cir.prove(po2, g, code, data, 1)[0]
    with pkg.Context(0, po2, SMALL, lib=gpu_lib, deterministic=True) as c:
        seg = c.segment_begin_dev(po2, g, code, data, 1)
        assert seg.stream and seg.device == 0
        _run_cb(seam_cb, c, seg)
        assert (c.segment_finish_dev() == oseal).all()
        assert (c.read_group(0) == cir.step_accum(po2, data, seg.mix_array(), 1)).all()
        assert c.last_stats()["ms_accum"] > 0
        # device inputs: columns uploaded by torch, copied device to device
        code_t, data_t = torch.from_numpy(code.astype(np.int32)).cuda(), torch.from_numpy(data.astype(np.int32)).cuda()
        torch.cuda.synchronize()
        seg = c.segment_begin_dev(po2, g, code_t.data_ptr(), data_t.data_ptr(), 1, device_inputs=True)
        _run_cb(seam_cb, c, seg)
        assert (c.segment_finish_dev() == oseal).all()
        with pytest.raises(pkg.Hfb200Error) as e:
            c.segment_begin_dev(po2, g, code.ctypes.data, data_t.data_ptr(), 1, device_inputs=True)
        assert str(e.value) == "HFB200_DEV_INPUTS: code is not device memory of device 0"
        assert (c.prove_segment(po2, g, code, data, 1) == oseal).all()   # refused before anything was queued: the context goes on
    widths, po2 = (16, 64, 16), 13
    ir = synth_ir.build(widths, 1, nest=True)
    cir = orc.Circuit(*widths, variant=1)
    code = cir.gen_code(po2); g = cir.gen_globals(5); data = cir.gen_data(po2, code, g, 5, 1)
    oseal = ir_oracle(orc, ir, widths).prove(po2, g, code, data, 1)[0]
    with pkg.Context(0, po2, widths, lib=gpu_lib, ir=ir, deterministic=True) as c:
        seg = c.segment_begin_dev(po2, g, code, data, 1)
        _run_cb(seam_cb, c, seg)
        assert (c.segment_finish_dev() == oseal).all()
        code_t, data_t = torch.from_numpy(code.astype(np.int32)).cuda(), torch.from_numpy(data.astype(np.int32)).cuda()
        torch.cuda.synchronize()
        seg = c.segment_begin_dev(po2, g, code_t.data_ptr(), data_t.data_ptr(), 1, device_inputs=True)
        _run_cb(seam_cb, c, seg)
        assert (c.segment_finish_dev() == oseal).all()


@pytest.mark.gpu
def test_ir_pool_with_c_callback_on_every_device(pkg, gpu_lib, orc, seam_cb):
    from oracle import synth_ir
    ndev = pkg.device_count(gpu_lib)
    assert ndev >= 1
    widths = (16, 64, 16)
    ir = synth_ir.build(widths, 0)
    cir_ir = ir_oracle(orc, ir, widths)
    jobs, expect = _ir_jobs(orc, cir_ir, widths, [13, 12, 14, 12, 13, 14, 12, 13], 800)
    cap = cir_ir.seal_words_model(14)
    fn = C.cast(seam_cb.seam_accum, C.c_void_p).value
    got = {}
    for devices in (tuple(range(ndev)), (0,)):
        with pkg.Pool(devices=devices, contexts_per_device=2, max_po2=14, circuit=widths, lib=gpu_lib, ir=ir, deterministic=True) as pool:
            counter = C.c_int(0)
            pool.set_accum(fn, C.addressof(counter))
            seals, devs, _ = pool.prove(jobs, cap)
            assert counter.value == len(jobs) and set(devs) <= set(devices)
            got[devices] = seals
    roots = {po2: cir_ir.control_id(po2) for po2 in (12, 13, 14)}
    for i, (a, b) in enumerate(zip(got[tuple(range(ndev))], expect)):
        assert len(a) == len(b) and (a == b).all(), i
        assert pkg.verify_segment(a, roots[jobs[i][0]], circuit=widths, ir=ir, lib=gpu_lib) == jobs[i][0]
        assert (got[(0,)][i] == a).all()


@pytest.mark.gpu
def test_device_seam_at_rv32im_scale_on_gpu(pkg, gpu_lib, orc, seam_cb):
    """build_scaled(560): ~51 k PolyExtSteps, W = 400 (14 accum chains), po2 20.  The device seam gives the seal of the host
    two-phase path for the same seeds."""
    from oracle import synth_ir
    ir = synth_ir.build_scaled(n_groups=560)
    W, po2 = ir["widths"], 20
    cir = orc.Circuit(*W)
    code = cir.gen_code(po2); g = cir.gen_globals(11)
    data = np.random.default_rng(11).integers(0, P, size=(W[1], 1 << po2), dtype=np.uint32)
    with pkg.Context(0, po2, W, lib=gpu_lib, ir=ir, deterministic=True) as c:
        mix = c.segment_begin(po2, g, code, data, 11)
        host = c.segment_finish(cir.step_accum(po2, data, mix, 11))
        seg = c.segment_begin_dev(po2, g, code, data, 11)
        assert (seg.mix_array() == mix).all()
        _run_cb(seam_cb, c, seg)
        dev = c.segment_finish_dev()
    assert len(dev) == len(host) and (dev == host).all()
