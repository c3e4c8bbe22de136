"""The process-wide cache of the specialised eval_check kernels of data-defined circuits, and kernel bundles.

Every (circuit, po2) is compiled with NVRTC once per process: contexts, pool workers and contexts re-created after a fault
take the cubins from the cache, and concurrent contexts wait for one compile.  hfb200_ir_compile fills the cache ahead of time
and serialises it as a bundle; hfb200_ir_load_kernels adds a bundle to the cache of another process, which then needs no NVRTC.

The cache belongs to the process, so every case runs in a fresh child process and reports the change of
hfb200_ir_nvrtc_programs() it saw.  CPU tier: the sm_100a library compiles and loads bundles without a device.  GPU tier:
seals with deterministic blinding, against the oracle and against the interpreter kernel (HFB200_IR_JIT=0).
"""
import ctypes as C
import hashlib
import json
import os
import shutil
import subprocess
import sys
import threading
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W = (16, 64, 16)
CALLBACK_CU = os.path.join(ROOT, "tools", "accum_seam_cb.cu")  # step_accum of the stand-in circuit, outside libhfb200
_ENV_KNOBS = ("HFB200_IR_CHUNK", "HFB200_IR_JIT", "HFB200_NVRTC_LIB", "HFB200_IR_JIT_MINB", "HFB200_IR_JIT_FENCE")

_CHILD = r"""
import json, os, sys
root = sys.argv[1]
sys.path[:0] = [root, os.path.join(root, "tests")]
import test_ir_kernel_cache as t
print(json.dumps(t.CASES[sys.argv[2]](*json.loads(sys.argv[3]))))
"""


def run_case(case, *args, env=None, timeout=1800):
    """CASES[case](*args) in a fresh process (its own kernel cache); returns what the case returned."""
    e = {k: v for k, v in os.environ.items() if k not in _ENV_KNOBS}
    e["HFB200_DETERMINISTIC_BLINDING"] = "1"
    e.update(env or {})
    r = subprocess.run([sys.executable, "-c", _CHILD, ROOT, case, json.dumps(args)], cwd=ROOT, env=e, capture_output=True, text=True,
                       timeout=timeout)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


# ---- what the child processes run ------------------------------------------------------------------------------------------

def _pkg():
    import hfb200_loader
    pkg = hfb200_loader.load()
    return pkg, pkg.load_library()


def _small_ir(variant=1):
    from oracle import synth_ir
    return synth_ir.build(W, variant, nest=variant == 1)


def _chunks(pkg, lib, ir, widths=W):
    return pkg.ir_source(ir, widths, lib=lib).count("__global__")


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, np.uint32).tobytes()).hexdigest()


def _ir_desc(pkg, ir, widths=W):
    taps, steps = np.ascontiguousarray(ir["taps"], np.uint32), np.ascontiguousarray(ir["steps"], np.uint32)
    d = pkg.binding._mk_ir(ir, widths[0], widths[1], widths[2], int(ir["n_mix"]), taps.ctypes.data, taps.size // 3, steps.ctypes.data,
                           steps.size // 4, int(ir["ret"]))
    return d, (taps, steps)


def _error(lib, e):
    assert e, "expected an error"
    msg = C.cast(e, C.c_char_p).value.decode()
    lib.hfb200_free_error(e)
    return msg


def case_compile_twice(path):
    pkg, lib = _pkg()
    ir = _small_ir()
    n0 = pkg.ir_nvrtc_programs(lib)
    b1 = pkg.ir_compile(ir, W, [12, 13], lib=lib)
    n1 = pkg.ir_nvrtc_programs(lib)
    b2 = pkg.ir_compile(ir, W, [13, 12, 13], lib=lib)
    n2 = pkg.ir_nvrtc_programs(lib)
    with open(path, "wb") as f:
        f.write(b1)
    return {"chunks": _chunks(pkg, lib, ir), "first": n1 - n0, "second": n2 - n1, "same": b1 == b2}


def case_need_cap():
    pkg, lib = _pkg()
    ir = _small_ir()
    desc, keep = _ir_desc(pkg, ir)
    po2s = (C.c_uint32 * 1)(12)
    out = {"chunks": _chunks(pkg, lib, ir)}
    n0 = pkg.ir_nvrtc_programs(lib)
    assert not lib.hfb200_ir_compile(C.byref(desc), po2s, 1, 0, None, 0, None)   # warm only
    out["warm"] = pkg.ir_nvrtc_programs(lib) - n0
    need = C.c_size_t(0)
    assert not lib.hfb200_ir_compile(C.byref(desc), po2s, 1, 0, None, 0, C.byref(need))
    out["need"] = need.value
    buf = C.create_string_buffer(need.value)
    got = C.c_size_t(0)
    out["small"] = _error(lib, lib.hfb200_ir_compile(C.byref(desc), po2s, 1, 0, buf, need.value - 1, C.byref(got)))
    out["need_again"] = got.value
    assert not lib.hfb200_ir_compile(C.byref(desc), po2s, 1, 2, buf, need.value, C.byref(got))
    out["same"] = buf.raw[:got.value] == pkg.ir_compile(ir, W, [12], lib=lib)
    out["after"] = pkg.ir_nvrtc_programs(lib) - n0
    return out


def case_chunk_setting():
    pkg, lib = _pkg()
    ir = _small_ir()
    out = {}
    for chunk in ("64", "128", "64"):
        os.environ["HFB200_IR_CHUNK"] = chunk
        n0 = pkg.ir_nvrtc_programs(lib)
        pkg.ir_compile(ir, W, [12], lib=lib, bundle=False)
        out.setdefault(chunk, []).append([_chunks(pkg, lib, ir), pkg.ir_nvrtc_programs(lib) - n0])
    return out


def case_load_then_compile(path):
    pkg, lib = _pkg()
    bundle = open(path, "rb").read()
    specs = pkg.ir_load_kernels(bundle, lib=lib)
    n0 = pkg.ir_nvrtc_programs(lib)
    b = pkg.ir_compile(_small_ir(), W, [12, 13], lib=lib)
    return {"specs": specs, "compiled": pkg.ir_nvrtc_programs(lib) - n0, "same": b == bundle}


def case_bad_bundles(path):
    pkg, lib = _pkg()
    good = open(path, "rb").read()
    arch_at = good.index(b"sm_100a")
    first_cubin = arch_at + 7 + 4 + 8 + 32 + 8   # n_specs, (po2, chunks), key, length
    flipped = bytearray(good)
    flipped[first_cubin + 100] ^= 0x10
    bad = {"truncated": good[:-1], "truncated_header": good[:20], "flipped": bytes(flipped), "magic": b"XFB200KB" + good[8:],
           "arch": good[:arch_at] + b"sm_101a" + good[arch_at + 7:], "trailing": good + b"\0"}
    out = {}
    for name, b in bad.items():
        try:
            pkg.ir_load_kernels(b, lib=lib)
            out[name] = None
        except pkg.Hfb200Error as e:
            out[name] = str(e)
    n0 = pkg.ir_nvrtc_programs(lib)
    pkg.ir_compile(_small_ir(), W, [12, 13], lib=lib, bundle=False)
    out["compiled_after"] = pkg.ir_nvrtc_programs(lib) - n0
    out["chunks"] = _chunks(pkg, lib, _small_ir())
    return out


def case_compile_bundle(path, po2s, scaled):
    """A bundle for po2s written to `path` (scaled: the rv32im-scale IR; otherwise the small one, variant 0 or 1)."""
    pkg, lib = _pkg()
    ir, widths = _case_ir(scaled)
    n0 = pkg.ir_nvrtc_programs(lib)
    b = pkg.ir_compile(ir, widths, po2s, lib=lib)
    with open(path, "wb") as f:
        f.write(b)
    return {"compiled": pkg.ir_nvrtc_programs(lib) - n0, "chunks": _chunks(pkg, lib, ir, widths)}


def _case_ir(scaled):
    from oracle import synth_ir
    if scaled == "rv32im":
        ir = synth_ir.build_scaled(n_groups=560)
        return ir, tuple(ir["widths"])
    return _small_ir(int(scaled)), W


def _prove_ir(pkg, c, orc, ir, widths, variant, seq, seed0, oracle_at=()):
    """Seals (sha256) of seq proved on context c through the two-phase entries, and for the sizes in oracle_at whether the
    oracle's seal is the same."""
    cir = orc.Circuit(*widths, variant=variant)
    cir_ir = orc.Circuit(*widths, variant=variant)
    cir_ir.set_ir(ir["taps"], ir["steps"], ir["ret"], ir.get("info"))
    seals, match = [], []
    for i, po2 in enumerate(seq):
        code = cir.gen_code(po2); g = cir.gen_globals(seed0 + i)
        if widths == W:
            data = cir.gen_data(po2, code, g, seed0 + i, seed0 + i)
        else:
            data = np.random.default_rng(seed0 + i).integers(0, orc.P, size=(widths[1], 1 << po2), dtype=np.uint32)
        mix = c.segment_begin(po2, g, code, data, seed0 + i)
        seal = c.segment_finish(cir.step_accum(po2, data, mix, seed0 + i))
        seals.append(_sha(seal))
        if po2 in oracle_at:
            oseal = cir_ir.prove(po2, g, code, data, seed0 + i)[0]
            match.append(bool(len(seal) == len(oseal) and (seal == oseal).all()))
    return seals, match


def case_rv32im_from_bundle(path, interpreter):
    """rv32im-scale IR, max_po2 = 16, proving 16, 12, 16: after loading the bundle (interpreter=False), or on the interpreter
    kernel (HFB200_IR_JIT=0)."""
    import oracle
    oracle.build()
    pkg, lib = _pkg()
    ir, widths = _case_ir("rv32im")
    if interpreter:
        os.environ["HFB200_IR_JIT"] = "0"
    else:
        assert pkg.ir_load_kernels(open(path, "rb").read(), lib=lib) == 2
    n0 = pkg.ir_nvrtc_programs(lib)
    with pkg.Context(0, 16, widths, lib=lib, ir=ir, deterministic=True) as c:
        active = c.ir_jit_active()[0]
        seals, match = _prove_ir(pkg, c, oracle, ir, widths, 0, [16, 12, 16], 30, oracle_at=(12,) if interpreter else ())
    return {"active": bool(active), "compiled": pkg.ir_nvrtc_programs(lib) - n0, "seals": seals, "oracle": match}


def case_pool(cb_path):
    """Pool of 2 contexts on every visible GPU over a data-defined circuit, no bundle: creation, a mixed-size batch, then a
    batch in which one worker meets an injected device fault."""
    import oracle
    oracle.build()
    pkg, lib = _pkg()
    ir = _small_ir(0)
    cb = C.CDLL(cb_path)
    cir_ir = oracle.Circuit(*W)
    cir_ir.set_ir(ir["taps"], ir["steps"], ir["ret"], ir.get("info"))
    cir = oracle.Circuit(*W)
    jobs, expect = [], []
    for i, po2 in enumerate([13, 12, 14, 12, 13, 14, 12, 13]):
        code = cir.gen_code(po2); g = cir.gen_globals(900 + i); data = cir.gen_data(po2, code, g, 900 + i, 900 + i)
        jobs.append((po2, g, code, data, 900 + i))
        expect.append(cir_ir.prove(po2, g, code, data, 900 + i)[0])
    cap = cir_ir.seal_words_model(14)
    ndev = pkg.device_count(lib)
    out = {"chunks": _chunks(pkg, lib, ir), "devices": ndev}
    n0 = pkg.ir_nvrtc_programs(lib)
    with pkg.Pool(devices=tuple(range(ndev)), contexts_per_device=2, max_po2=14, circuit=W, lib=lib, ir=ir, deterministic=True) as pool:
        out["create"] = pkg.ir_nvrtc_programs(lib) - n0
        pool.set_accum(C.cast(cb.seam_accum, C.c_void_p).value, None)
        n1 = pkg.ir_nvrtc_programs(lib)
        seals, _, _ = pool.prove(jobs, cap)
        out["batch"] = pkg.ir_nvrtc_programs(lib) - n1
        out["batch_ok"] = all(len(a) == len(b) and bool((a == b).all()) for a, b in zip(seals, expect))
        pool.inject_fault(0, 0, 0)
        n2 = pkg.ir_nvrtc_programs(lib)
        seals, _, _ = pool.prove(jobs, cap)
        out["fault"] = pkg.ir_nvrtc_programs(lib) - n2
        out["fault_ok"] = all(len(a) == len(b) and bool((a == b).all()) for a, b in zip(seals, expect))
        out["recreated"] = pool.stats()["contexts_recreated"]
    return out


def case_concurrent_init():
    """Four threads create contexts of one data-defined circuit at once, then each proves the same segment."""
    import oracle
    oracle.build()
    pkg, lib = _pkg()
    ir = _small_ir()
    n0 = pkg.ir_nvrtc_programs(lib)
    ctxs, errors = [None] * 4, []
    barrier = threading.Barrier(4)

    def make(k):
        try:
            barrier.wait()
            ctxs[k] = pkg.Context(0, 13, W, lib=lib, ir=ir, deterministic=True)
        except BaseException as e:  # reported below
            errors.append(repr(e))
    th = [threading.Thread(target=make, args=(k,)) for k in range(4)]
    [t.start() for t in th]
    [t.join() for t in th]
    out = {"errors": errors, "compiled": pkg.ir_nvrtc_programs(lib) - n0, "chunks": _chunks(pkg, lib, ir), "seals": [], "oracle": []}
    for c in ctxs:
        if c is None:
            continue
        with c:
            out["active"] = bool(c.ir_jit_active()[0])
            seals, match = _prove_ir(pkg, c, oracle, ir, W, 1, [13], 77, oracle_at=(13,) if not out["oracle"] else ())
            out["seals"] += seals
            out["oracle"] += match
    return out


def case_without_nvrtc(path):
    """HFB200_NVRTC_LIB names no library: without the bundle the interpreter runs; with the bundle (po2 13) the specialised
    kernels run for 13 and the interpreter for 12, which the bundle lacks."""
    import oracle
    oracle.build()
    pkg, lib = _pkg()
    ir = _small_ir()
    out = {}
    with pkg.Context(0, 13, W, lib=lib, ir=ir, deterministic=True) as c:
        out["active_before"] = bool(c.ir_jit_active()[0])
        out["seals_before"], out["oracle_before"] = _prove_ir(pkg, c, oracle, ir, W, 1, [13], 50, oracle_at=(13,))
    out["specs"] = pkg.ir_load_kernels(open(path, "rb").read(), lib=lib)
    with pkg.Context(0, 13, W, lib=lib, ir=ir, deterministic=True) as c:
        out["active_after"] = bool(c.ir_jit_active()[0])
        out["seals_after"], out["oracle_after"] = _prove_ir(pkg, c, oracle, ir, W, 1, [13, 12], 50, oracle_at=(13, 12))
    out["compiled"] = pkg.ir_nvrtc_programs(lib)
    return out


CASES = {f.__name__[len("case_"):]: f for f in (case_compile_twice, case_need_cap, case_chunk_setting, case_load_then_compile, case_bad_bundles,
                                                case_compile_bundle, case_rv32im_from_bundle, case_pool, case_concurrent_init, case_without_nvrtc)}


# ---- CPU tier --------------------------------------------------------------------------------------------------------------

def test_compiles_once_and_serialises_identically(tmp_path):
    r = run_case("compile_twice", str(tmp_path / "b"), env={"HFB200_IR_CHUNK": "64"})
    assert r["chunks"] >= 4
    assert r["first"] == 2 * r["chunks"]
    assert r["second"] == 0 and r["same"]


def test_need_and_cap():
    r = run_case("need_cap", env={"HFB200_IR_CHUNK": "64"})
    assert r["warm"] == r["chunks"] and r["after"] == r["chunks"]
    assert r["need"] > 0 and r["need_again"] == r["need"]
    assert r["small"] == "hfb200_ir_compile: bundle buffer too small: need %d bytes" % r["need"]
    assert r["same"]


def test_chunk_setting_is_part_of_the_key():
    r = run_case("chunk_setting")
    (k64, first), (_, again) = r["64"]
    (k128, other), = r["128"]
    assert first == k64 and k128 < k64 and other == k128 and again == 0


def test_bundle_loaded_in_a_fresh_process_compiles_nothing(tmp_path):
    path = str(tmp_path / "b")
    run_case("compile_twice", path, env={"HFB200_IR_CHUNK": "64"})
    r = run_case("load_then_compile", path, env={"HFB200_IR_CHUNK": "64"})
    assert r == {"specs": 2, "compiled": 0, "same": True}
    # other code-generation settings: the bundle loads but never matches
    r = run_case("load_then_compile", path, env={"HFB200_IR_CHUNK": "96"})
    assert r["specs"] == 2 and r["compiled"] > 0 and not r["same"]


def test_malformed_bundles_are_refused_whole(tmp_path):
    path = str(tmp_path / "b")
    run_case("compile_twice", path, env={"HFB200_IR_CHUNK": "64"})
    r = run_case("bad_bundles", path, env={"HFB200_IR_CHUNK": "64"})
    pre = "hfb200_ir_load_kernels: "
    assert r["truncated"] == pre + "bundle truncated" and r["truncated_header"] == pre + "bundle truncated"
    assert r["flipped"] == pre + "bundle digest does not match its contents (corrupted)"
    assert r["magic"] == pre + "not an eval_check kernel bundle (bad magic)"
    assert r["arch"] == pre + "bundle holds kernels for sm_101a, this library runs sm_100a"
    assert r["trailing"] == pre + "bundle has trailing bytes"
    assert r["compiled_after"] == 2 * r["chunks"]   # nothing was added


def test_refusals_match_init_ir(pkg, gpu_lib, emu_lib):
    ir = _small_ir()
    for po2 in (11, 23):
        with pytest.raises(pkg.Hfb200Error) as e:
            pkg.ir_compile(ir, W, [12, po2], lib=gpu_lib)
        with pytest.raises(pkg.Hfb200Error) as init:
            pkg.Context(0, po2, W, lib=emu_lib, ir=ir)
        assert str(e.value) == "po2 must be in [12, 22]" and str(init.value).endswith(str(e.value))
    # five distinct back values: over the declared limit of four
    over = dict(ir)
    over["taps"] = np.array([[2, k, k] for k in range(5)], np.uint32).ravel()
    for bad in (over, dict(ir, ret=10 ** 6)):
        with pytest.raises(pkg.Hfb200Error) as e:
            pkg.ir_compile(bad, W, [12], lib=gpu_lib)
        with pytest.raises(pkg.Hfb200Error) as init:
            pkg.Context(0, 12, W, lib=emu_lib, ir=bad)
        assert str(e.value) == str(init.value) and str(e.value).startswith("circuit: ")
        assert bad is not over or str(e.value) == "circuit: more than 4 distinct back values"


def test_host_emulator_has_no_kernels_to_compile(pkg, emu_lib):
    with pytest.raises(pkg.Hfb200Error, match="host emulator"):
        pkg.ir_compile(_small_ir(), W, [12], lib=emu_lib)
    with pytest.raises(pkg.Hfb200Error, match="host emulator"):
        pkg.ir_load_kernels(b"HFB200KB", lib=emu_lib)
    assert pkg.ir_nvrtc_programs(emu_lib) == 0


# ---- GPU tier --------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_rv32im_scale_from_a_bundle_on_gpu(tmp_path):
    path = str(tmp_path / "rv32im")
    made = run_case("compile_bundle", path, [12, 16], "rv32im")
    assert made["compiled"] == 2 * made["chunks"]
    jit = run_case("rv32im_from_bundle", path, False)
    assert jit["active"] and jit["compiled"] == 0
    interp = run_case("rv32im_from_bundle", path, True)
    assert not interp["active"] and interp["oracle"] == [True]
    assert jit["seals"] == interp["seals"]


@pytest.fixture(scope="module")
def seam_cb(pkg, tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    so = tmp_path_factory.mktemp("seam_cb") / "libseam_cb.so"
    libdir = os.path.dirname(pkg.LIB_PATH)
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-Xcompiler", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"),
                           "-o", str(so), CALLBACK_CU, "-L", libdir, "-l:libhfb200.so", "-Xlinker", "-rpath," + libdir])
    return str(so)


@pytest.mark.gpu
def test_pool_compiles_each_size_once_on_gpu(seam_cb):
    r = run_case("pool", seam_cb, env={"HFB200_IR_CHUNK": "64"})
    assert r["devices"] >= 1 and r["chunks"] >= 4
    assert r["create"] == r["chunks"]          # one set for max_po2, not one per context
    assert r["batch"] == 2 * r["chunks"]       # po2 12 and 13, once each
    assert r["batch_ok"]
    assert r["recreated"] >= 1 and r["fault"] == 0 and r["fault_ok"]


@pytest.mark.gpu
def test_concurrent_init_compiles_once_on_gpu():
    r = run_case("concurrent_init", env={"HFB200_IR_CHUNK": "64"})
    assert r["errors"] == [] and r["active"]
    assert r["compiled"] == r["chunks"]
    assert len(r["seals"]) == 4 and len(set(r["seals"])) == 1 and r["oracle"] == [True]


@pytest.mark.gpu
def test_without_nvrtc_on_gpu(tmp_path):
    path = str(tmp_path / "b13")
    run_case("compile_bundle", path, [13], "1")
    r = run_case("without_nvrtc", path, env={"HFB200_NVRTC_LIB": "/nonexistent/libnvrtc.so"})
    assert not r["active_before"] and r["oracle_before"] == [True]
    assert r["specs"] == 1 and r["active_after"] and r["oracle_after"] == [True, True]
    assert r["seals_after"][0] == r["seals_before"][0]
    assert r["compiled"] == 0
