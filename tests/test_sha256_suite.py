"""The SHA-256 hash suite (upstream's segment_prover("sha-256")): the compression and the suite's hashes, ShaRng, the Merkle
kernels, whole seals, the verifier, suite switching on one context and pools.

CPU tier: the host emulator of the kernel sources and the CPU oracle, both against a short pure-Python FIPS 180-4 restatement
written here (and hashlib for the padded hash).  GPU tier: the sm_100a kernels against the oracle (live and pinned)."""
import hashlib
import struct
import threading

import numpy as np
import pytest
from conftest import SMALL, DEFAULT, make_segment, rand_elems
from oracle import sha_suite as osha   # the oracle's prover and verifier in the SHA-256 suite

P = 2013265921
MASK = 0xFFFFFFFF
SHA = "sha-256"


# ---- FIPS 180-4, restated: constants from the primes, one compression, the suite's byte conventions ------------------------

def _primes(n):
    out, k = [], 2
    while len(out) < n:
        if all(k % p for p in out):
            out.append(k)
        k += 1
    return out


def _iroot(x, k):
    r = int(round(x ** (1.0 / k)))
    while r ** k > x:
        r -= 1
    while (r + 1) ** k <= x:
        r += 1
    return r


K = [_iroot(p << 96, 3) & MASK for p in _primes(64)]   # first 32 bits of the fractional parts of the cube roots
IV = [_iroot(p << 64, 2) & MASK for p in _primes(8)]   # ... of the square roots


def _rotr(x, n):
    return ((x >> n) | (x << (32 - n))) & MASK


def py_compress(state, block):
    w = list(struct.unpack(">16I", block))
    for t in range(16, 64):
        s0 = _rotr(w[t - 15], 7) ^ _rotr(w[t - 15], 18) ^ (w[t - 15] >> 3)
        s1 = _rotr(w[t - 2], 17) ^ _rotr(w[t - 2], 19) ^ (w[t - 2] >> 10)
        w.append((w[t - 16] + s0 + w[t - 7] + s1) & MASK)
    a, b, c, d, e, f, g, h = state
    for t in range(64):
        t1 = (h + (_rotr(e, 6) ^ _rotr(e, 11) ^ _rotr(e, 25)) + ((e & f) ^ (~e & g)) + K[t] + w[t]) & MASK
        t2 = ((_rotr(a, 2) ^ _rotr(a, 13) ^ _rotr(a, 22)) + ((a & b) ^ (a & c) ^ (b & c))) & MASK
        a, b, c, d, e, f, g, h = (t1 + t2) & MASK, a, b, c, (d + t1) & MASK, e, f, g
    return [(x + y) & MASK for x, y in zip(state, (a, b, c, d, e, f, g, h))]


def py_digest_words(state):
    """the 32 output bytes as 8 little-endian words"""
    return np.frombuffer(struct.pack(">8I", *state), dtype="<u4").astype(np.uint32)


def py_sha256(msg):
    m = msg + b"\x80" + b"\x00" * ((55 - len(msg)) % 64) + struct.pack(">Q", 8 * len(msg))
    st = IV
    for i in range(0, len(m), 64):
        st = py_compress(st, m[i:i + 64])
    return py_digest_words(st)


def py_hash_words(words):
    """hash_raw_data_slice: little-endian bytes of the words, 64 per block, the last block zero-filled, no length."""
    data = np.asarray(words, dtype="<u4").tobytes()
    st = IV
    for i in range(0, len(data), 64):
        st = py_compress(st, data[i:i + 64].ljust(64, b"\x00"))
    return py_digest_words(st)


def py_hash_pair(a, b):
    return py_digest_words(py_compress(IV, np.asarray(a, "<u4").tobytes() + np.asarray(b, "<u4").tobytes()))


class PyShaRng:
    def __init__(self):
        self.pool0, self.pool1, self.used = py_sha256(b"Hello"), py_sha256(b"World"), 0

    def step(self):
        self.pool0 = py_hash_pair(self.pool0, self.pool1)
        self.pool1 = py_hash_pair(self.pool0, self.pool1)
        self.used = 0

    def mix(self, d):
        self.pool0 = self.pool0 ^ np.asarray(d, np.uint32)
        self.step()

    def next_u32(self):
        if self.used == 8:
            self.step()
        self.used += 1
        return int(self.pool0[self.used - 1])

    def random_elem(self):
        v = 0
        for _ in range(6):
            v = ((v << 32) + self.next_u32()) % P
        return (v << 32) % P   # Montgomery form

    def random_bits(self, b):
        return self.next_u32() & ((1 << b) - 1)


def py_rng_script(ops, digests):
    r, out, d = PyShaRng(), [], iter(np.asarray(digests, np.uint32).reshape(-1, 8))
    for op in ops:
        if op[0] == "mix":
            r.mix(next(d))
        elif op[0] == "elem":
            out.append(r.random_elem())
        else:
            out.append(r.random_bits(op[1]))
    return np.array(out, np.uint32)


# ---- fixtures ------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def emu(pkg, emu_lib):
    with pkg.Context(0, 12, SMALL, lib=emu_lib, deterministic=True) as c:
        c.set_hash_suite(SHA)
        yield c


@pytest.fixture(scope="module")
def small_segments(orc):
    """SMALL circuit at po2 12 and 13: (cir, globals, code, data, oracle SHA seal, oracle SHA checkpoints, oracle Poseidon2 seal)."""
    out = {}
    for po2 in (12, 13):
        cir, g, code, data = make_segment(orc, SMALL, po2)
        seal, cps = osha.Circuit(*SMALL).prove(po2, g, code, data, 1)
        out[po2] = (cir, g, code, data, seal, cps, cir.prove(po2, g, code, data, 1)[0])
    return out


def _same(a, b):
    return len(a) == len(b) and (np.asarray(a) == np.asarray(b)).all()


# ---- primitives ------------------------------------------------------------------------------------------------------------

MESSAGES = [b"abc", b"Hello", b"World", b"", b"a" * 55, bytes(range(56)), bytes(range(64)), bytes(i * 7 & 255 for i in range(1000))]


@pytest.mark.parametrize("msg", MESSAGES, ids=lambda m: "len%d" % len(m))
def test_padded_sha256_matches_hashlib(pkg, emu_lib, orc, msg):
    want = np.frombuffer(hashlib.sha256(msg).digest(), dtype="<u4")
    assert (py_sha256(msg) == want).all()       # the restatement above is FIPS 180-4
    assert (osha.sha256(msg) == want).all()
    assert (pkg.sha256(msg, lib=emu_lib) == want).all()


@pytest.mark.parametrize("width", [1, 15, 16, 17, 192, 256])
def test_row_hash_and_pair_match_restatement(pkg, emu_lib, orc, width):
    rng = np.random.default_rng(width)
    row = rand_elems(rng, width)
    want = py_hash_words(row)
    assert (osha.hash_elems(row) == want).all()
    assert (pkg.hash_elems(row, SHA, lib=emu_lib) == want).all()
    a, b = rng.integers(0, 1 << 32, 8, dtype=np.uint32), rng.integers(0, 1 << 32, 8, dtype=np.uint32)
    want = py_hash_pair(a, b)
    assert (osha.hash_pair(a, b) == want).all()
    assert (pkg.hash_pair(a, b, SHA, lib=emu_lib) == want).all()
    # a pair is the raw hash of its 16 words: one compression, no padding
    assert (want == py_hash_words(np.concatenate([a, b]))).all()
    # the Poseidon2 suite is untouched by the new entries
    assert (pkg.hash_elems(row, "poseidon2", lib=emu_lib) == orc.hash_elems(row)).all()


def test_sha_rng_draws(pkg, emu_lib, orc):
    rng = np.random.default_rng(7)
    digests = rng.integers(0, 1 << 32, (4, 8), dtype=np.uint32)
    ops = [("elem",)] * 3 + [("mix",)] + [("elem",)] * 9 + [("bits", 22), ("bits", 1), ("bits", 31)] + [("mix",), ("mix",)] + \
          [("bits", 16)] * 10 + [("elem",)] * 4 + [("mix",), ("elem",)]
    want = py_rng_script(ops, digests)
    assert len(want) == 30
    assert (osha.rng_draw(ops, digests) == want).all()
    assert (pkg.rng_script(ops, digests, SHA, lib=emu_lib) == want).all()
    assert not (pkg.rng_script(ops, digests, "poseidon2", lib=emu_lib) == want).all()


# ---- Merkle trees ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("rows,cols", [(2, 1), (8, 15), (64, 17), (32, 300), (256, 192), (1024, 33)])
def test_op_merkle_equals_oracle(emu, orc, rows, cols):
    m = rand_elems(np.random.default_rng(rows * 1000 + cols), (cols, rows))
    root, nodes = osha.merkle(m, want_nodes=True)
    got = emu.op_merkle(m)
    assert (got[1:] == nodes[1:]).all() and (got[1] == root).all()
    assert (nodes[rows + 1] == py_hash_words(m[:, 1])).all() and (nodes[1] == py_hash_pair(nodes[2], nodes[3])).all()
    assert not (orc.merkle(m) == root).all()


@pytest.mark.parametrize("rows,cols", [(1, 1), (100, 16), (333, 17), (129, 300)])
def test_hal_sha_rows_ragged(pkg, emu, orc, rows, cols):
    hal = pkg.Hal(emu)
    m = rand_elems(np.random.default_rng(rows + cols), (cols, rows))
    dig = np.zeros((rows, 8), np.uint32)
    hal.sha_rows(dig, m)
    hal.sync()
    for r in range(rows):
        assert (dig[r] == osha.hash_elems(m[:, r])).all(), r


@pytest.mark.parametrize("rows,cols", [(64, 5), (512, 64)])
def test_hal_sha_rows_and_folds_equal_oracle_tree(pkg, emu, orc, rows, cols):
    hal = pkg.Hal(emu)
    m = rand_elems(np.random.default_rng(cols), (cols, rows))
    nodes = np.zeros((2 * rows, 8), np.uint32)
    hal.sha_rows(nodes[rows:], m)
    size = rows
    while size > 1:
        hal.sha_fold(nodes, size, size // 2)
        size //= 2
    hal.sync()
    assert (nodes[1:] == osha.merkle(m, want_nodes=True)[1][1:]).all()
    # hash_rows stays Poseidon2 whatever the context's suite
    p2 = np.zeros((rows, 8), np.uint32)
    hal.hash_rows(p2, m)
    assert (p2 == orc.merkle(m, want_nodes=True)[1][rows:]).all()


def test_hal_sha_refusals(pkg, emu):
    hal = pkg.Hal(emu)
    nodes = np.zeros((16, 8), np.uint32)
    with pytest.raises(pkg.Hfb200Error, match="input_size must be 2 \\* output_size"):
        hal.sha_fold(nodes, 8, 3)
    with pytest.raises(pkg.Hfb200Error, match="digests must be"):
        hal.sha_rows(np.zeros((3, 8), np.uint32), np.zeros((2, 4), np.uint32))
    with pytest.raises(pkg.Hfb200Error, match="rows = 0"):
        hal.sha_rows(np.zeros((0, 8), np.uint32), np.zeros((2, 0), np.uint32))


# ---- whole seals -----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("po2", [12, 13])
def test_one_shot_seal_equals_oracle(pkg, emu_lib, small_segments, po2):
    cir, g, code, data, oseal, ocps, p2seal = small_segments[po2]
    with pkg.Context(0, 13, SMALL, lib=emu_lib, deterministic=True) as c:
        c.set_hash_suite(SHA)
        seal = c.prove_segment(po2, g, code, data, 1)
        assert _same(seal, oseal) and len(seal) == c.seal_words(po2)
        cps = c.checkpoints()
        for k, v in ocps.items():
            if k in cps:
                assert (cps[k] == v).all(), k
        assert len(seal) == len(p2seal) and not (seal == p2seal).all()      # same layout, other hashes
        assert (seal[:33] == p2seal[:33]).all() and not (seal[33:41] == p2seal[33:41]).all()   # globals ++ po2, then the roots


@pytest.mark.parametrize("po2", [12, 13])
def test_two_phase_host_accum_equals_oracle(pkg, emu_lib, small_segments, po2):
    cir, g, code, data, oseal, ocps, _ = small_segments[po2]
    with pkg.Context(0, 13, SMALL, lib=emu_lib, deterministic=True) as c:
        c.set_hash_suite(SHA)
        mix = c.segment_begin(po2, g, code, data, 1)
        assert (mix == ocps["accum_mix"]).all()
        assert _same(c.segment_finish(cir.step_accum(po2, data, mix, 1)), oseal)


def test_data_defined_circuit_equals_oracle(pkg, emu_lib, orc):
    from oracle import synth_ir
    widths, po2 = (12, 24, 8), 12
    cir, g, code, data = make_segment(orc, widths, po2)
    ir = synth_ir.build(widths, 0, nest=True)
    cir_ir = osha.Circuit(*widths, ir=ir)
    oseal, ocps = cir_ir.prove(po2, g, code, data, 1)
    with pkg.Context(0, po2, widths, lib=emu_lib, ir=ir, deterministic=True) as c:
        c.set_hash_suite(SHA)
        mix = c.segment_begin(po2, g, code, data, 1)
        seal = c.segment_finish(cir.step_accum(po2, data, mix, 1))
        assert _same(seal, oseal)
        cid = cir_ir.control_id(po2)
        assert cir_ir.verify(seal, cid) == po2
        assert pkg.verify_segment(seal, cid, widths, ir=ir, lib=emu_lib, hashfn=SHA) == po2


@pytest.mark.parametrize("po2", [12, 13])
def test_control_reuse_equals_oracle(pkg, emu_lib, small_segments, po2):
    cir, g, code, data, oseal, ocps, _ = small_segments[po2]
    with pkg.Context(0, 13, SMALL, lib=emu_lib, deterministic=True) as c:
        c.set_hash_suite(SHA)
        root = c.control_root(po2, code)
        assert (root == osha.Circuit(*cir.w).control_id(po2)).all() and (root == ocps["code_root"]).all()
        assert _same(c.prove_segment(po2, g, None, data, 1), oseal)
        assert _same(c.prove_segment(po2, g, None, data, 1), oseal)


# ---- verifier --------------------------------------------------------------------------------------------------------------

def test_verifier_accepts_and_rejects(pkg, emu_lib, small_segments):
    cir, g, code, data, oseal, ocps, p2seal = small_segments[12]
    cid, p2cid = osha.Circuit(*cir.w).control_id(12), cir.control_id(12)
    assert not (cid == p2cid).all()
    assert pkg.verify_segment(oseal, cid, SMALL, lib=emu_lib, hashfn=SHA) == 12
    assert osha.Circuit(*cir.w).verify(oseal, cid) == 12
    with pytest.raises(pkg.Hfb200Error, match="control id"):
        pkg.verify_segment(oseal, p2cid, SMALL, lib=emu_lib, hashfn=SHA)          # the other suite's control id
    with pytest.raises(RuntimeError, match="control id"):
        osha.Circuit(*cir.w).verify(oseal, p2cid)
    for root in (cid, p2cid):                                                    # verified as a Poseidon2 seal
        with pytest.raises(pkg.Hfb200Error):
            pkg.verify_segment(oseal, root, SMALL, lib=emu_lib)
        with pytest.raises(RuntimeError):
            cir.verify(oseal, root)
    with pytest.raises(pkg.Hfb200Error):                                         # a Poseidon2 seal verified as SHA-256
        pkg.verify_segment(p2seal, p2cid, SMALL, lib=emu_lib, hashfn=SHA)
    with pytest.raises(RuntimeError):
        osha.Circuit(*cir.w).verify(p2seal, p2cid)
    for pos in (40, len(oseal) // 2, len(oseal) - 3):                            # one flipped word anywhere
        bad = oseal.copy()
        bad[pos] ^= 1
        with pytest.raises(pkg.Hfb200Error):
            pkg.verify_segment(bad, cid, SMALL, lib=emu_lib, hashfn=SHA)
        with pytest.raises(RuntimeError):
            osha.Circuit(*cir.w).verify(bad, cid)
    with pytest.raises(pkg.Hfb200Error, match="not supported"):
        pkg.verify_segment(oseal, cid, SMALL, lib=emu_lib, hashfn="blake2b")


def test_verify_segments_reports_first_bad(pkg, emu_lib, small_segments):
    seals, roots = [], []
    for po2 in (12, 13, 12):
        cir, _, _, _, oseal, _, _ = small_segments[po2]
        seals.append(oseal.copy())
        roots.append(osha.Circuit(*cir.w).control_id(po2))
    assert pkg.verify_segments(seals, roots, SMALL, lib=emu_lib, hashfn=SHA) == [12, 13, 12]
    seals[2][100] ^= 4
    seals[1][200] ^= 4
    with pytest.raises(pkg.Hfb200Error, match="^segment 1: "):
        pkg.verify_segments(seals, roots, SMALL, lib=emu_lib, hashfn=SHA)
    with pytest.raises(pkg.Hfb200Error, match="^segment 0: "):
        pkg.verify_segments(seals, roots, SMALL, lib=emu_lib)


# ---- one context, both suites ----------------------------------------------------------------------------------------------

def test_suite_switching_and_control_cache(pkg, emu_lib, small_segments):
    cir, g, code, data, oseal, ocps, p2seal = small_segments[12]
    with pkg.Context(0, 12, SMALL, lib=emu_lib, deterministic=True) as c:
        assert _same(c.prove_segment(12, g, code, data, 1), p2seal)
        c.set_hash_suite(SHA)
        assert _same(c.prove_segment(12, g, code, data, 1), oseal)
        c.set_hash_suite("poseidon2")
        assert _same(c.prove_segment(12, g, code, data, 1), p2seal)
        # a resident control group belongs to the suite that committed it
        c.control_root(12, code)
        assert _same(c.prove_segment(12, g, None, data, 1), p2seal)
        c.set_hash_suite(SHA)
        with pytest.raises(pkg.Hfb200Error, match="no control group is resident"):
            c.prove_segment(12, g, None, data, 1)
        assert (c.control_root(12, code) == osha.Circuit(*cir.w).control_id(12)).all()
        assert _same(c.prove_segment(12, g, None, data, 1), oseal)
        c.set_hash_suite("poseidon2")
        with pytest.raises(pkg.Hfb200Error, match="no control group is resident"):
            c.segment_begin(12, g, None, data, 1)
        c.set_hash_suite(SHA)                      # the same suite again keeps nothing: the switch above dropped it
        with pytest.raises(pkg.Hfb200Error, match="no control group is resident"):
            c.prove_segment(12, g, None, data, 1)


def test_refused_combinations(pkg, emu_lib, small_segments):
    cir, g, code, data, oseal, _, _ = small_segments[12]
    with pkg.Context(0, 12, SMALL, lib=emu_lib, deterministic=True) as c:
        c.set_hash_suite(SHA)
        for mode in (1, 2):
            with pytest.raises(pkg.Hfb200Error, match="host transcript only"):
                c.set_transcript(mode)
        c.set_transcript(0)
        with pytest.raises(pkg.Hfb200Error, match="not supported"):
            c.set_hash_suite("blake2b")
        assert pkg.hash_suite("sha-256") == pkg.HASH_SHA256 and pkg.hash_suite("poseidon2") == pkg.HASH_POSEIDON2
        c.set_hash_suite("poseidon2")
        c.set_transcript(1)
        with pytest.raises(pkg.Hfb200Error, match="device transcript mode 1"):
            c.set_hash_suite(SHA)
        c.set_transcript(0)
        c.set_hash_suite(SHA)
        c.segment_begin(12, g, code, data, 1)
        with pytest.raises(pkg.Hfb200Error, match="in flight"):
            c.set_hash_suite("poseidon2")
        assert _same(c.segment_finish(None), oseal)       # the refused switch left the segment intact
    import ctypes as C
    lib = emu_lib
    e = lib.hfb200_set_hash_suite(None, 1)               # NULL ctx: an error message, not a crash
    assert e
    lib.hfb200_free_error(e)
    with pkg.Context(0, 12, SMALL, lib=emu_lib) as c:
        e = lib.hfb200_set_hash_suite(c._h, 2)
        assert e and "HFB200_HASH_SHA256" in C.cast(e, C.c_char_p).value.decode()
        lib.hfb200_free_error(e)


def test_device_transcript_env_does_not_apply(pkg, emu_lib, small_segments, monkeypatch):
    """HFB200_DEVICE_TRANSCRIPT selects the device transcript only for Poseidon2 contexts; a SHA-256 context proves on the host."""
    cir, g, code, data, oseal, _, _ = small_segments[12]
    monkeypatch.setenv("HFB200_DEVICE_TRANSCRIPT", "1")
    with pkg.Context(0, 12, SMALL, lib=emu_lib, deterministic=True) as c:
        c.set_hash_suite(SHA)
        assert _same(c.prove_segment(12, g, code, data, 1), oseal)


# ---- pools -----------------------------------------------------------------------------------------------------------------

def test_pool_survives_device_fault_with_suite(pkg, emu_lib, orc):
    jobs, expect = [], []
    for i in range(4):
        cir, g, code, data = make_segment(orc, SMALL, 12, trace_seed=700 + i)
        jobs.append((12, g, code, data, 30 + i))
        expect.append(osha.Circuit(*cir.w).prove(12, g, code, data, 30 + i)[0])
    with pkg.Pool(devices=(0, 0), contexts_per_device=1, max_po2=12, circuit=SMALL, lib=emu_lib, deterministic=True) as pool:
        pool.set_hash_suite(SHA)
        pool.inject_fault(worker=0, after_jobs=0, kind=0)
        seals, _, _ = pool.prove(jobs, 40000)
        assert all(_same(a, b) for a, b in zip(seals, expect))
        st = pool.stats()
        assert st["faults"] == 1 and st["contexts_recreated"] == 1
        pool.inject_fault(worker=1, after_jobs=0, kind=0)    # both workers now run on re-created contexts
        seals, _, _ = pool.prove(jobs, 40000)
        assert all(_same(a, b) for a, b in zip(seals, expect))
        pool.set_hash_suite("poseidon2")
        seals, _, _ = pool.prove(jobs[:1], 40000)
        assert _same(seals[0], orc.Circuit(*SMALL).prove(*jobs[0])[0])


def test_pool_control_group_follows_suite(pkg, emu_lib, orc):
    cir, g, code, data = make_segment(orc, SMALL, 12, trace_seed=77)
    with pkg.Pool(devices=(0,), contexts_per_device=1, max_po2=12, circuit=SMALL, lib=emu_lib, deterministic=True) as pool:
        pool.load_control(12, code)
        p2, _, _ = pool.prove([(12, g, None, data, 5)], 40000)
        pool.set_hash_suite(SHA)
        sha, _, _ = pool.prove([(12, g, None, data, 5)], 40000)    # re-committed in the new suite
        assert _same(p2[0], cir.prove(12, g, code, data, 5)[0])
        assert _same(sha[0], osha.Circuit(*cir.w).prove(12, g, code, data, 5)[0])


# ---- GPU tier --------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("widths", [SMALL, DEFAULT], ids=["small", "w256"])
def test_gpu_seals_equal_oracle(pkg, gpu_lib, orc, widths):
    with pkg.Context(0, 16, widths, lib=gpu_lib, deterministic=True) as c:
        c.set_hash_suite(SHA)
        for po2 in range(12, 17):
            cir, g, code, data = make_segment(orc, widths, po2)
            oseal, ocps = osha.Circuit(*widths).prove(po2, g, code, data, 1)
            seal = c.prove_segment(po2, g, code, data, 1)
            assert _same(seal, oseal), po2
            cps = c.checkpoints()
            for k in ("code_root", "data_root", "accum_root", "check_root", "hash_u", "fri_final_hash", "query_positions"):
                assert (cps[k] == ocps[k]).all(), (po2, k)


@pytest.mark.gpu
def test_gpu_po2_20_w256_pinned(pkg, gpu_lib, orc, monkeypatch):
    """The headline shape in the SHA-256 suite against pins generated from the oracle (tests/golden/make_golden_sha256.py):
    resident path and host-buffer path, every checkpoint, the seal's hash, length, head and tail."""
    import json
    import os
    from conftest import ROOT
    monkeypatch.setenv("HFB200_DEBUG_CHECKPOINTS", "1")
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "golden_sha256_po2_20_w256.json")))
    po2, W = gold["po2"], tuple(gold["widths"])

    def check(seal, cps):
        for k, v in gold["checkpoints"].items():
            assert cps[k].tolist() == v, k
        assert len(seal) == gold["seal_words"]
        assert seal[:64].tolist() == gold["seal_head"] and seal[-64:].tolist() == gold["seal_tail"]
        assert int(seal.astype(np.uint64).sum()) == gold["seal_sum_u64"]
        assert orc.hash_elems(seal % orc.P).tolist() == gold["seal_hash"]

    with pkg.Context(0, po2, W, lib=gpu_lib, deterministic=True) as c:
        c.set_hash_suite(SHA)
        g = c.witgen_synth(po2, gold["trace_seed"], gold["blind_seed"])
        seal = c.prove_resident(gold["blind_seed"])
        check(seal, c.checkpoints())
        code, data = c.read_group(1), c.read_group(2)
        check(c.prove_segment(po2, g, code, data, gold["blind_seed"]), c.checkpoints())
        assert pkg.verify_segment(seal, gold["control_id"], W, lib=gpu_lib, hashfn=SHA) == po2


@pytest.mark.gpu
def test_gpu_po2_22_w256_verifies(pkg, gpu_lib, orc):
    po2 = 22
    with pkg.Context(0, po2, DEFAULT, lib=gpu_lib, deterministic=True) as c:
        c.set_hash_suite(SHA)
        c.witgen_synth(po2, 0x48595046, 1)
        seal = c.prove_resident(1)
        cid = c.checkpoint("code_root")
        assert (c.control_root(po2, c.read_group(1)) == cid).all()
    assert len(seal) == orc.Circuit(*DEFAULT).seal_words_model(po2)
    assert pkg.verify_segment(seal, cid, DEFAULT, lib=gpu_lib, hashfn=SHA) == po2
    assert osha.Circuit(*DEFAULT).verify(seal, cid) == po2
    bad = seal.copy()
    bad[len(bad) // 3] ^= 1
    with pytest.raises(pkg.Hfb200Error):
        pkg.verify_segment(bad, cid, DEFAULT, lib=gpu_lib, hashfn=SHA)


@pytest.mark.gpu
def test_gpu_hal_sha_rows_and_fold(pkg, gpu_lib, orc):
    import torch
    with pkg.Context(0, 12, SMALL, lib=gpu_lib) as c:
        hal = pkg.Hal(c)
        rng = np.random.default_rng(5)
        for rows, cols in ((1000, 17), (4099, 192)):                 # rows not a multiple of the block size
            m = rand_elems(rng, (cols, rows))
            dig = torch.zeros((rows, 8), dtype=torch.int32, device="cuda:0")
            hal.sha_rows(dig, torch.from_numpy(m.view(np.int32)).cuda())
            hal.sync()
            got = dig.cpu().numpy().view(np.uint32)
            for r in list(range(0, rows, 97)) + [rows - 1]:
                assert (got[r] == osha.hash_elems(m[:, r])).all(), (rows, r)
        rows, cols = 1 << 14, 64
        m = rand_elems(rng, (cols, rows))
        nodes = torch.zeros((2 * rows, 8), dtype=torch.int32, device="cuda:0")
        hal.sha_rows(nodes[rows:], torch.from_numpy(m.view(np.int32)).cuda())
        size = rows
        while size > 1:
            hal.sha_fold(nodes, size, size // 2)
            size //= 2
        hal.sync()
        assert (nodes.cpu().numpy().view(np.uint32)[1:] == osha.merkle(m, want_nodes=True)[1][1:]).all()


@pytest.mark.gpu
def test_gpu_pool_across_devices(pkg, gpu_lib, orc):
    n_dev = pkg.device_count(gpu_lib)
    jobs, expect = [], []
    for i, po2 in enumerate([14, 12, 13, 12, 14, 13, 12, 12]):
        cir, g, code, data = make_segment(orc, SMALL, po2, trace_seed=500 + i)
        jobs.append((po2, g, code, data, 11 + i))
        expect.append(osha.Circuit(*cir.w).prove(po2, g, code, data, 11 + i)[0])
    cap = max(len(e) for e in expect)
    with pkg.Pool(devices=tuple(range(n_dev)), contexts_per_device=2, max_po2=14, circuit=SMALL, lib=gpu_lib, deterministic=True) as pool:
        pool.set_hash_suite(SHA)
        seals, devs, _ = pool.prove(jobs, cap)
    assert all(_same(a, b) for a, b in zip(seals, expect))
    with pkg.Context(0, 14, SMALL, lib=gpu_lib, deterministic=True) as c:
        c.set_hash_suite(SHA)
        for (po2, g, code, data, seed), s in zip(jobs, seals):
            assert _same(c.prove_segment(po2, g, code, data, seed), s)


@pytest.mark.gpu
def test_gpu_device_seam_accum_callback(pkg, gpu_lib, orc):
    """A built-in pool whose accum stage is the caller's: the callback writes the oracle's accum columns into the context's device
    accum buffer (wrapped as a torch tensor) and the SHA-256 seal equals the oracle's."""
    import torch
    po2 = 12
    cir, g, code, data = make_segment(orc, SMALL, po2, trace_seed=321)
    oseal = osha.Circuit(*cir.w).prove(po2, g, code, data, 9)[0]

    class Cols:
        def __init__(self, ptr, shape):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": "<i4", "data": (ptr, False), "version": 3}

    def accum(h, seg, job):
        acc = cir.step_accum(seg.po2, data, seg.mix_array(), seg.blind_seed)
        dst = torch.as_tensor(Cols(seg.accum, (seg.w_accum, seg.rows)), device="cuda:%d" % seg.device)
        dst.copy_(torch.from_numpy(acc.view(np.int32)).to(dst.device))
        torch.cuda.synchronize(dst.device)

    with pkg.Pool(devices=(0,), contexts_per_device=1, max_po2=po2, circuit=SMALL, lib=gpu_lib, deterministic=True) as pool:
        pool.set_hash_suite(SHA)
        pool.set_accum(accum)
        seals, _, _ = pool.prove([(po2, g, code, data, 9)], len(oseal))
    assert _same(seals[0], oseal)


@pytest.mark.gpu
def test_gpu_mixed_suites_concurrently(pkg, gpu_lib, orc):
    po2 = 14
    cir, g, code, data = make_segment(orc, DEFAULT, po2)
    want = {"poseidon2": cir.prove(po2, g, code, data, 1)[0], SHA: osha.Circuit(*DEFAULT).prove(po2, g, code, data, 1)[0]}
    out = {}

    def work(suite):
        with pkg.Context(0, po2, DEFAULT, lib=gpu_lib, deterministic=True) as c:
            c.set_hash_suite(suite)
            out[suite] = [c.prove_segment(po2, g, code, data, 1) for _ in range(3)]

    th = [threading.Thread(target=work, args=(s,)) for s in want]
    [t.start() for t in th]
    [t.join() for t in th]
    for s, seals in out.items():
        assert all(_same(x, want[s]) for x in seals), s
