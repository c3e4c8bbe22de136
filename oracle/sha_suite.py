"""ctypes binding of the oracle with upstream's SHA-256 hash suite (TEST INFRASTRUCTURE ONLY): oracle/sha_prover.cpp, the oracle's
own prover, verifier and control ids compiled with the Merkle hash and transcript RNG of `segment_prover("sha-256")`
(oracle/sha256.h: FIPS 180-4 over byte strings, the suite convention recalled from risc0-zkp 3.0.4 `core/hash/sha`).

Circuits here prove and verify; their traces come from `oracle.Circuit` (witness generation does not depend on the suite)."""
import ctypes as C
import os
import subprocess

import numpy as np


_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "liboracle_sha.so")
_SRCS = ["sha_prover.cpp", "sha256.h", "prover.cpp", "prover.h", "fp.h", "poseidon2.h", "poseidon2_consts.inc", "ntt.h", "merkle_iop.h",
         "blind.h", "circuit.h"]


def build(force=False):
    """Compile oracle/_build/liboracle_sha.so if missing or stale (the flags of oracle/Makefile)."""
    stale = force or not os.path.exists(_SO)
    if not stale:
        t = os.path.getmtime(_SO)
        stale = any(os.path.getmtime(os.path.join(_HERE, s)) > t for s in _SRCS)
    if stale:
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        tmp = _SO + ".%d.tmp" % os.getpid()
        subprocess.check_call([cxx, "-O3", "-std=c++17", "-fPIC", "-fopenmp", "-Wall", "-Wno-unknown-pragmas", "-shared", "-o", tmp,
                               os.path.join(_HERE, "sha_prover.cpp")])
        os.replace(tmp, _SO)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        vp, sz = C.c_void_p, C.c_size_t
        L.orc_sha_last_error.restype = C.c_char_p
        L.orc_sha_sha256.argtypes = [C.c_char_p, sz, vp]
        L.orc_sha_hash_elems.argtypes = [vp, sz, vp]
        L.orc_sha_hash_pair.argtypes = [vp, vp, vp]
        L.orc_sha_rng_script.restype = sz
        L.orc_sha_rng_script.argtypes = [vp, sz, vp, vp]
        L.orc_sha_merkle.argtypes = [vp, sz, sz, vp, vp]
        L.orc_sha_circuit_new.restype = vp
        L.orc_sha_circuit_new.argtypes = [C.c_uint32] * 4
        L.orc_sha_circuit_free.argtypes = [vp]
        L.orc_sha_circuit_set_ir.argtypes = [vp, vp, sz, vp, sz, C.c_uint32, C.c_char_p]
        L.orc_sha_control_id.argtypes = [vp, C.c_uint, vp]
        L.orc_sha_prove_segment.argtypes = [vp, C.c_uint, vp, vp, vp, C.c_uint64, C.POINTER(vp)]
        L.orc_sha_verify_segment.argtypes = [vp, vp, sz, vp, vp]
        L.orc_sha_proof_seal_words.restype = sz
        L.orc_sha_proof_seal_words.argtypes = [vp]
        L.orc_sha_proof_seal.argtypes = [vp, vp]
        L.orc_sha_proof_n_checkpoints.restype = sz
        L.orc_sha_proof_n_checkpoints.argtypes = [vp]
        L.orc_sha_proof_checkpoint.restype = sz
        L.orc_sha_proof_checkpoint.argtypes = [vp, sz, C.c_char_p, sz, vp, sz]
        L.orc_sha_proof_free.argtypes = [vp]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def _check(rc):
    if rc != 0:
        raise RuntimeError(lib().orc_sha_last_error().decode())


def sha256(data):
    """Standard (padded) SHA-256 of a byte string as 8 digest words (little-endian bytes = the standard output)."""
    data, out = bytes(data), np.zeros(8, np.uint32)
    lib().orc_sha_sha256(data, len(data), _p(out))
    return out


def hash_elems(elems):
    """The suite's hash of a word slice: little-endian bytes, 64 per compression, last block zero-filled, no length block."""
    e, out = _u32(elems).reshape(-1), np.zeros(8, np.uint32)
    lib().orc_sha_hash_elems(_p(e), e.size, _p(out))
    return out


def hash_pair(a, b):
    a, b, out = _u32(a), _u32(b), np.zeros(8, np.uint32)
    lib().orc_sha_hash_pair(_p(a), _p(b), _p(out))
    return out


def rng_draw(ops, digests):
    """ShaRng through `ops` (("mix",), ("elem",), ("bits", b)); mixes take the 8-word digests in order.  Returns the draws."""
    code = {"mix": 0, "elem": 1, "bits": 2}
    o = np.array([[code[op[0]], op[1] if len(op) > 1 else 0] for op in ops], dtype=np.uint32).reshape(-1)
    d = _u32(digests).reshape(-1)
    out = np.zeros(max(1, len(ops)), np.uint32)
    n = lib().orc_sha_rng_script(_p(o), len(ops), _p(d), _p(out))
    return out[:n]


def merkle(matrix, want_nodes=False):
    """matrix: [cols, rows] u32 (column-major rows).  Returns root (and heap-layout nodes [2*rows, 8])."""
    m = _u32(matrix)
    cols, rows = m.shape
    root = np.zeros(8, np.uint32)
    nodes = np.zeros((2 * rows, 8), np.uint32) if want_nodes else None
    _check(lib().orc_sha_merkle(_p(m), rows, cols, _p(root), _p(nodes) if want_nodes else None))
    return (root, nodes) if want_nodes else root


class Circuit:
    """oracle.Circuit's prover side in the SHA-256 suite: the built-in stand-in circuit (variant 0 / 1), or a data-defined one
    given as `ir` = {"taps", "steps", "ret", "info"} (oracle/synth_ir.py's form)."""

    def __init__(self, w_code=16, w_data=192, w_accum=48, variant=0, ir=None):
        self.w = (w_code, w_data, w_accum)
        self._h = lib().orc_sha_circuit_new(w_code, w_data, w_accum, variant)
        if not self._h:
            raise RuntimeError(lib().orc_sha_last_error().decode())
        if ir is not None:
            taps, steps, info = _u32(ir["taps"]), _u32(ir["steps"]), ir.get("info")
            if info is not None and len(info) != 16:
                raise ValueError("circuit info must be 16 bytes")
            _check(lib().orc_sha_circuit_set_ir(self._h, _p(taps), taps.size // 3, _p(steps), steps.size // 4, ir["ret"], info))

    def __del__(self):
        try:
            if self._h:
                lib().orc_sha_circuit_free(self._h)
                self._h = None
        except Exception:
            pass

    def control_id(self, po2):
        out = np.zeros(8, np.uint32)
        _check(lib().orc_sha_control_id(self._h, po2, _p(out)))
        return out

    def prove(self, po2, globals_, code, data, blind_seed):
        """Returns (seal u32 array, checkpoints dict name -> u32 array (ordered))."""
        h = C.c_void_p()
        globals_, code, data = _u32(globals_), _u32(code), _u32(data)
        _check(lib().orc_sha_prove_segment(self._h, po2, _p(globals_), _p(code), _p(data), blind_seed, C.byref(h)))
        try:
            seal = np.zeros(lib().orc_sha_proof_seal_words(h), np.uint32)
            lib().orc_sha_proof_seal(h, _p(seal))
            cps, name, buf = {}, C.create_string_buffer(64), np.zeros(4096, np.uint32)
            for i in range(lib().orc_sha_proof_n_checkpoints(h)):
                k = lib().orc_sha_proof_checkpoint(h, i, name, 64, _p(buf), buf.size)
                cps[name.value.decode()] = buf[:k].copy()
        finally:
            lib().orc_sha_proof_free(h)
        return seal, cps

    def verify(self, seal, code_root):
        seal, code_root = _u32(seal), _u32(code_root)
        po2 = C.c_uint()
        _check(lib().orc_sha_verify_segment(self._h, _p(seal), seal.size, _p(code_root), C.byref(po2)))
        return po2.value
