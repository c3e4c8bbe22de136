"""ctypes binding of libhfb200.so (include/hfb200.h).

This is host-side glue only: every call goes straight through the C ABI that a Rust `extern "C"` crate
would bind (INTEGRATION.md).  There is no CPU fallback: if the CUDA library is missing or no B200 is
visible, loading / `hfb200_init` raises.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhfb200.so")

N_GLOBAL = 32
P = 2013265921

# Every symbol include/hfb200.h declares (tests check that the built library exports all of them).
EXPORTS = [
    "hfb200_init", "hfb200_init_ir", "hfb200_ir_source", "hfb200_ir_jit_active", "hfb200_verify_segment", "hfb200_verify_segments", "hfb200_control_root", "hfb200_destroy", "hfb200_free_error", "hfb200_version", "hfb200_host_alloc", "hfb200_host_free",
    "hfb200_prove_segment", "hfb200_segment_begin", "hfb200_segment_finish", "hfb200_witgen_synth",
    "hfb200_prove_resident", "hfb200_read_group", "hfb200_seal_words", "hfb200_checkpoint", "hfb200_last_stats",
    "hfb200_total_launches", "hfb200_op_interpolate_ntt", "hfb200_op_expand_ntt", "hfb200_op_lde", "hfb200_op_merkle",
    "hfb200_op_poseidon2", "hfb200_op_fri_fold", "hfb200_bench_lde", "hfb200_bench_merkle", "hfb200_bench_modmul",
    "hfb200_mark", "hfb200_mark_elapsed",
    "hfb200_pool_create", "hfb200_pool_create_ir", "hfb200_pool_load_control", "hfb200_pool_prove", "hfb200_pool_destroy",
    "hfb200_set_blinding", "hfb200_pool_set_blinding", "hfb200_pool_stats", "hfb200_pool_inject_fault",
    "hfb200_set_transcript", "hfb200_graph_launches", "hfb200_digest_bytes", "hfb200_digest_pair", "hfb200_claim_encode", "hfb200_claim_decode", "hfb200_claim_next_state", "hfb200_verify_claims",
    "hfb200_segment_begin_dev", "hfb200_segment_finish_dev", "hfb200_segment_accum_scan", "hfb200_segment_accum_blind", "hfb200_device_count",
    "hfb200_pool_set_accum",
    "hfb200_segment_witness_dev", "hfb200_segment_data_blind", "hfb200_segment_scratch", "hfb200_pool_set_witgen",
    "hfb200_hal_stream", "hfb200_hal_sync", "hfb200_hal_host_syncs", "hfb200_hal_batch_interpolate_ntt", "hfb200_hal_zk_shift",
    "hfb200_hal_batch_expand_into_evaluate_ntt", "hfb200_hal_batch_bit_reverse", "hfb200_hal_hash_rows", "hfb200_hal_hash_fold",
    "hfb200_hal_batch_evaluate_any", "hfb200_hal_mix_poly_coeffs", "hfb200_hal_poly_divide", "hfb200_hal_eltwise_add_elem",
    "hfb200_hal_eltwise_sum_extelem", "hfb200_hal_eltwise_copy_elem", "hfb200_hal_eltwise_zeroize_elem", "hfb200_hal_gather_sample",
    "hfb200_hal_scatter", "hfb200_hal_prefix_products", "hfb200_hal_fri_fold",
]

BLIND_OS_ENTROPY, BLIND_DETERMINISTIC = 0, 1


def _default_blinding(deterministic):
    """The C ABI's default is OS entropy (zero-knowledge).  The parity tests and the bench need reproducible seals: they ask for
    the deterministic mode explicitly, or through HFB200_DETERMINISTIC_BLINDING=1 (set by tests/conftest.py and bench.py)."""
    if deterministic is None:
        deterministic = os.environ.get("HFB200_DETERMINISTIC_BLINDING", "0") == "1"
    return BLIND_DETERMINISTIC if deterministic else BLIND_OS_ENTROPY


class Hfb200Error(RuntimeError):
    pass


class CircuitDesc(C.Structure):
    _fields_ = [("w_code", C.c_uint32), ("w_data", C.c_uint32), ("w_accum", C.c_uint32), ("flags", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("ms_total", C.c_float), ("ms_device", C.c_float), ("ms_h2d", C.c_float), ("ms_ntt_main", C.c_float), ("ms_hash_main", C.c_float),
                ("ms_accum", C.c_float), ("ms_check", C.c_float), ("ms_deep", C.c_float), ("ms_fri", C.c_float),
                ("launches", C.c_uint64), ("ntt_main_bytes", C.c_uint64), ("host_syncs", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class CircuitIR(C.Structure):
    _fields_ = [("w_code", C.c_uint32), ("w_data", C.c_uint32), ("w_accum", C.c_uint32), ("n_mix", C.c_uint32),
                ("taps", C.c_void_p), ("n_taps", C.c_size_t), ("steps", C.c_void_p), ("n_steps", C.c_size_t), ("ret", C.c_uint32),
                ("info", C.c_uint8 * 16)]  # CIRCUIT_INFO; zeros = upstream's "RV32IM:v2_______"


def _mk_ir(ir, *fields):
    """hfb200_circuit_ir from positional fields + the circuit's 16-byte CIRCUIT_INFO (ir["info"]; absent / None = zeros = the
    library default for data-defined circuits, upstream's b"RV32IM:v2_______")."""
    d = CircuitIR(*fields)
    info = ir.get("info") if hasattr(ir, "get") else None
    if info is not None:
        if len(info) != 16:
            raise Hfb200Error("circuit info must be 16 bytes")
        C.memmove(d.info, bytes(info), 16)
    return d


class SegmentJob(C.Structure):
    _fields_ = [("po2", C.c_uint32), ("globals", C.c_void_p), ("code", C.c_void_p), ("data", C.c_void_p), ("blind_seed", C.c_uint64),
                ("seal_out", C.c_void_p), ("seal_cap", C.c_size_t), ("seal_words", C.c_size_t), ("error", C.c_void_p),
                ("device", C.c_int), ("ms", C.c_float), ("attempts", C.c_int)]


class Claim(C.Structure):
    """hfb200_claim: what upstream's ReceiptClaim boils down to on this path (pre / post state, exit code, output digest)."""
    _fields_ = [("pre", C.c_uint32 * 8), ("post", C.c_uint32 * 8), ("output", C.c_uint32 * 8), ("exit_code", C.c_uint32)]

    def to_obj(self):
        return {"pre": list(self.pre), "post": list(self.post), "exit_code": "SystemSplit" if self.exit_code else "Halted", "output": list(self.output)}


EXIT_HALTED, EXIT_SYSTEM_SPLIT = 0, 1
DEV_INPUTS = 1
SCAN_PRODUCT, SCAN_SUM = 0, 1


class SegmentDev(C.Structure):
    """hfb200_segment_dev: the segment in flight between segment_begin_dev and segment_finish_dev.  `code`, `data`, `globals`,
    `mix` and `accum` are device addresses (host addresses in the emulator); `stream` is the context's cudaStream_t."""
    _fields_ = [("po2", C.c_uint32), ("zk_rows", C.c_uint32), ("w_code", C.c_uint32), ("w_data", C.c_uint32), ("w_accum", C.c_uint32),
                ("n_mix", C.c_uint32), ("device", C.c_int), ("stream", C.c_void_p), ("code", C.c_void_p), ("data", C.c_void_p),
                ("globals", C.c_void_p), ("mix", C.c_void_p), ("accum", C.c_void_p), ("mix_host", C.POINTER(C.c_uint32)),
                ("globals_host", C.POINTER(C.c_uint32)), ("blind_seed", C.c_uint64)]

    @property
    def rows(self):
        return 1 << self.po2

    def mix_array(self):
        return np.ctypeslib.as_array(self.mix_host, shape=(self.n_mix,)).copy()

    def globals_array(self):
        return np.ctypeslib.as_array(self.globals_host, shape=(N_GLOBAL,)).copy()

    def host_view(self, name):
        """numpy view of a column group -- only where device addresses ARE host addresses (the host emulator)."""
        w = {"code": self.w_code, "data": self.w_data, "accum": self.w_accum}[name]
        return np.ctypeslib.as_array(C.cast(getattr(self, name), C.POINTER(C.c_uint32)), shape=(w * self.rows,)).reshape(w, self.rows)


# int (*hfb200_accum_fn)(void* user, hfb200_ctx* ctx, const hfb200_segment_dev* seg, size_t job)
ACCUM_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.POINTER(SegmentDev), C.c_size_t)


class WitnessDev(C.Structure):
    """hfb200_witness_dev: the writable DATA columns between segment_witness_dev and the begin that commits them.  `data` is a
    device address (a host address in the emulator); `stream` is the context's cudaStream_t."""
    _fields_ = [("po2", C.c_uint32), ("zk_rows", C.c_uint32), ("w_code", C.c_uint32), ("w_data", C.c_uint32), ("device", C.c_int),
                ("stream", C.c_void_p), ("data", C.c_void_p)]

    @property
    def rows(self):
        return 1 << self.po2

    def host_view(self):
        """numpy view [w_data, rows] of the data columns -- only where device addresses ARE host addresses (the host emulator)."""
        return np.ctypeslib.as_array(C.cast(self.data, C.POINTER(C.c_uint32)), shape=(self.w_data * self.rows,)).reshape(self.w_data, self.rows)


def scratch_view(addr, nbytes):
    """numpy uint8 view of a segment scratch buffer -- only in the host emulator, where it is host memory."""
    return np.ctypeslib.as_array(C.cast(addr, C.POINTER(C.c_uint8)), shape=(nbytes,))


# int (*hfb200_witgen_fn)(void* user, hfb200_ctx* ctx, const hfb200_witness_dev* w, size_t job)
WITGEN_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.POINTER(WitnessDev), C.c_size_t)


class PoolStats(C.Structure):
    _fields_ = [("contexts", C.c_size_t), ("contexts_retired", C.c_size_t), ("faults", C.c_uint64), ("retries", C.c_uint64),
                ("contexts_recreated", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


def load_library(path=None):
    """dlopen the product library.  Raises Hfb200Error when it has not been built (no fallback)."""
    path = path or os.environ.get("HFB200_LIB") or LIB_PATH  # HFB200_LIB: another build of the same library (kernel experiments)
    if not os.path.exists(path):
        raise Hfb200Error("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(the prover has no CPU fallback)" % path)
    lib = C.CDLL(path)
    vp, u32, u64, sz = C.c_void_p, C.c_uint32, C.c_uint64, C.c_size_t
    err = C.c_void_p  # const char* that we must free ourselves
    sig = {
        "hfb200_init": (err, [C.c_int, u32, C.POINTER(CircuitDesc), C.POINTER(vp)]),
        "hfb200_init_ir": (err, [C.c_int, u32, C.POINTER(CircuitIR), C.POINTER(vp)]),
        "hfb200_ir_source": (err, [C.POINTER(CircuitIR), C.c_char_p, sz, C.POINTER(sz)]),
        "hfb200_ir_jit_active": (C.c_int, [vp, C.POINTER(C.c_float)]),
        "hfb200_verify_segment": (err, [C.POINTER(CircuitDesc), C.POINTER(CircuitIR), vp, sz, vp, C.POINTER(u32)]),
        "hfb200_control_root": (err, [vp, u32, vp, vp]),
        "hfb200_destroy": (None, [vp]),
        "hfb200_free_error": (None, [vp]),
        "hfb200_version": (C.c_char_p, []),
        "hfb200_host_alloc": (err, [sz, C.POINTER(vp)]),
        "hfb200_host_free": (None, [vp]),
        "hfb200_prove_segment": (err, [vp, u32, vp, vp, vp, u64, vp, sz, C.POINTER(sz)]),
        "hfb200_segment_begin": (err, [vp, u32, vp, vp, vp, u64, vp, sz, C.POINTER(sz)]),
        "hfb200_segment_finish": (err, [vp, vp, vp, sz, C.POINTER(sz)]),
        "hfb200_witgen_synth": (err, [vp, u32, u64, u64, vp]),
        "hfb200_prove_resident": (err, [vp, u64, vp, sz, C.POINTER(sz)]),
        "hfb200_read_group": (err, [vp, u32, vp, sz]),
        "hfb200_seal_words": (sz, [vp, u32]),
        "hfb200_checkpoint": (err, [vp, C.c_char_p, vp, sz, C.POINTER(sz)]),
        "hfb200_last_stats": (err, [vp, C.POINTER(Stats)]),
        "hfb200_total_launches": (u64, [vp]),
        "hfb200_op_interpolate_ntt": (err, [vp, vp, sz, sz, C.c_int]),
        "hfb200_op_expand_ntt": (err, [vp, vp, vp, sz, sz, u32]),
        "hfb200_op_lde": (err, [vp, vp, vp, sz, sz]),
        "hfb200_op_merkle": (err, [vp, vp, sz, sz, vp]),
        "hfb200_op_poseidon2": (err, [vp, vp, sz]),
        "hfb200_op_fri_fold": (err, [vp, vp, vp, sz, vp]),
        "hfb200_bench_lde": (err, [vp, u32, u32, u32, C.POINTER(C.c_float)]),
        "hfb200_bench_merkle": (err, [vp, u32, u32, u32, C.POINTER(C.c_float)]),
        "hfb200_bench_modmul": (err, [vp, C.c_int, u32, C.POINTER(C.c_double)]),
        "hfb200_mark": (err, [vp, C.c_int]),
        "hfb200_mark_elapsed": (err, [vp, C.c_int, vp, C.c_int, C.POINTER(C.c_float)]),
        "hfb200_pool_create": (err, [C.POINTER(C.c_int), C.c_int, C.c_int, u32, C.POINTER(CircuitDesc), C.POINTER(vp)]),
        "hfb200_pool_prove": (err, [vp, C.POINTER(SegmentJob), sz]),
        "hfb200_pool_load_control": (err, [vp, u32, vp]),
        "hfb200_pool_destroy": (None, [vp]),
        "hfb200_pool_create_ir": (err, [C.POINTER(C.c_int), C.c_int, C.c_int, u32, C.POINTER(CircuitIR), C.POINTER(vp)]),
        "hfb200_set_blinding": (err, [vp, C.c_int]),
        "hfb200_pool_set_blinding": (err, [vp, C.c_int]),
        "hfb200_pool_stats": (err, [vp, C.POINTER(PoolStats)]),
        "hfb200_pool_inject_fault": (err, [vp, sz, u64, C.c_int]),
        "hfb200_set_transcript": (err, [vp, C.c_int]),
        "hfb200_graph_launches": (u64, [vp]),
        "hfb200_digest_bytes": (err, [C.c_char_p, sz, vp]),
        "hfb200_digest_pair": (err, [vp, vp, vp]),
        "hfb200_claim_encode": (err, [C.POINTER(Claim), vp]),
        "hfb200_claim_decode": (err, [vp, sz, C.POINTER(Claim)]),
        "hfb200_claim_next_state": (err, [vp, u32, u32, vp]),
        "hfb200_verify_segments": (err, [C.POINTER(CircuitDesc), C.POINTER(CircuitIR), C.POINTER(vp), C.POINTER(sz), sz, vp, vp, C.c_uint, C.POINTER(sz)]),
        "hfb200_verify_claims": (err, [C.POINTER(vp), C.POINTER(sz), sz, vp, C.c_char_p, sz]),
        "hfb200_segment_begin_dev": (err, [vp, u32, vp, vp, vp, u64, u32, C.POINTER(SegmentDev)]),
        "hfb200_segment_finish_dev": (err, [vp, vp, sz, C.POINTER(sz)]),
        "hfb200_segment_accum_scan": (err, [vp, C.c_int, u32, u32, sz]),
        "hfb200_segment_accum_blind": (err, [vp]),
        "hfb200_device_count": (err, [C.POINTER(C.c_int)]),
        "hfb200_pool_set_accum": (err, [vp, vp, vp]),
        "hfb200_segment_witness_dev": (err, [vp, u32, u64, C.POINTER(WitnessDev)]),
        "hfb200_segment_data_blind": (err, [vp]),
        "hfb200_segment_scratch": (err, [vp, sz, C.POINTER(vp)]),
        "hfb200_pool_set_witgen": (err, [vp, vp, vp]),
        "hfb200_hal_stream": (err, [vp, C.POINTER(vp), C.POINTER(C.c_int)]),
        "hfb200_hal_sync": (err, [vp]),
        "hfb200_hal_host_syncs": (u64, [vp]),
        "hfb200_hal_batch_interpolate_ntt": (err, [vp, vp, sz, sz]),
        "hfb200_hal_zk_shift": (err, [vp, vp, sz, sz]),
        "hfb200_hal_batch_expand_into_evaluate_ntt": (err, [vp, vp, vp, sz, sz, u32]),
        "hfb200_hal_batch_bit_reverse": (err, [vp, vp, sz, sz]),
        "hfb200_hal_hash_rows": (err, [vp, vp, vp, sz, sz]),
        "hfb200_hal_hash_fold": (err, [vp, vp, sz, sz]),
        "hfb200_hal_batch_evaluate_any": (err, [vp, vp, sz, sz, vp, vp, vp, sz]),
        "hfb200_hal_mix_poly_coeffs": (err, [vp, vp, vp, vp, vp, vp, sz, sz, sz]),
        "hfb200_hal_poly_divide": (err, [vp, vp, sz, vp, vp]),
        "hfb200_hal_eltwise_add_elem": (err, [vp, vp, vp, vp, sz]),
        "hfb200_hal_eltwise_sum_extelem": (err, [vp, vp, vp, sz, sz]),
        "hfb200_hal_eltwise_copy_elem": (err, [vp, vp, vp, sz]),
        "hfb200_hal_eltwise_zeroize_elem": (err, [vp, vp, sz]),
        "hfb200_hal_gather_sample": (err, [vp, vp, vp, sz, sz, sz]),
        "hfb200_hal_scatter": (err, [vp, vp, vp, vp, vp, sz]),
        "hfb200_hal_prefix_products": (err, [vp, vp, sz]),
        "hfb200_hal_fri_fold": (err, [vp, vp, vp, sz, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _u32(a):
    a = np.ascontiguousarray(a, dtype=np.uint32)
    return a


CHECKPOINT_NAMES = ["globals_hash", "code_root", "data_root", "accum_mix", "accum_root", "poly_mix", "check_root", "z",
                    "hash_u", "deep_mix", "final_poly_hash", "fri_root_0", "fri_mix_0", "fri_root_1", "fri_mix_1",
                    "fri_root_2", "fri_mix_2", "fri_root_3", "fri_mix_3", "fri_final_hash", "query_positions"]


class Context:
    """One hfb200_ctx: one host thread <-> one GPU.  Mirrors upstream's `segment_prover(hashfn)` object."""

    def __init__(self, device=0, max_po2=20, circuit=(16, 192, 48), lib=None, ir=None, deterministic=None):
        """`ir`: optional data-defined circuit {"taps": u32[n,3], "steps": u32[m,4], "ret": int, "n_mix": int} (hfb200_init_ir).
        `deterministic`: blinding derived from the blind_seed arguments alone (tests / bench); default = OS entropy unless
        HFB200_DETERMINISTIC_BLINDING=1."""
        self.lib = lib or load_library()
        self.circuit = tuple(int(x) for x in circuit)
        self.max_po2 = max_po2
        h = C.c_void_p()
        self._h = None
        self._po2 = max_po2
        if ir is not None:
            taps, steps = _u32(ir["taps"]), _u32(ir["steps"])
            desc = _mk_ir(ir, self.circuit[0], self.circuit[1], self.circuit[2], int(ir["n_mix"]), taps.ctypes.data, taps.size // 3,
                             steps.ctypes.data, steps.size // 4, int(ir["ret"]))
            self._check(self.lib.hfb200_init_ir(device, max_po2, C.byref(desc), C.byref(h)))
        else:
            desc = CircuitDesc(self.circuit[0], self.circuit[1], self.circuit[2], 0)
            self._check(self.lib.hfb200_init(device, max_po2, C.byref(desc), C.byref(h)))
        self._h = h
        self.set_blinding(_default_blinding(deterministic))

    def set_blinding(self, mode):
        self._check(self.lib.hfb200_set_blinding(self._h, int(mode)))

    def set_transcript(self, mode):
        """Fiat-Shamir transcript of the one-shot entries: 0 / False = host (default), 1 / True = device (one sync per segment),
        2 = device + CUDA-graph replay (one cudaGraphLaunch per segment from the third segment of a shape on)."""
        self._check(self.lib.hfb200_set_transcript(self._h, int(mode)))

    def graph_launches(self):
        return self.lib.hfb200_graph_launches(self._h)

    def _check(self, e):
        if e:
            msg = C.cast(e, C.c_char_p).value.decode(errors="replace")
            self.lib.hfb200_free_error(e)
            raise Hfb200Error(msg)

    def close(self):
        if self._h:
            self.lib.hfb200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def version(self):
        return self.lib.hfb200_version().decode()

    # ---- segment prover ----
    def seal_words(self, po2):
        return self.lib.hfb200_seal_words(self._h, po2)

    def prove_segment(self, po2, globals_, code, data, blind_seed):
        """code=None reuses the control group loaded by control_root(po2, code)."""
        globals_, data = _u32(globals_), _u32(data)
        code = _u32(code) if code is not None else None
        n = 1 << po2
        if globals_.size != N_GLOBAL or (code is not None and code.size != self.circuit[0] * n) or data.size != self.circuit[1] * n:
            raise Hfb200Error("prove_segment: trace shape does not match (circuit, po2)")
        cap = self.seal_words(po2)
        seal = np.empty(cap, np.uint32)
        got = C.c_size_t()
        self._check(self.lib.hfb200_prove_segment(self._h, po2, _ptr(globals_), _ptr(code), _ptr(data), blind_seed, _ptr(seal), cap, C.byref(got)))
        self._po2 = po2  # the proved trace is now the resident one (prove_resident, read_group)
        return seal[:got.value]

    def segment_begin(self, po2, globals_, code, data, blind_seed):
        globals_ = _u32(globals_)
        code = _u32(code) if code is not None else None
        data = _u32(data) if data is not None else None
        mix = np.empty(self.circuit[2], np.uint32)
        got = C.c_size_t()
        self._check(self.lib.hfb200_segment_begin(self._h, po2, _ptr(globals_), _ptr(code), _ptr(data), blind_seed, _ptr(mix), mix.size, C.byref(got)))
        self._po2 = po2
        return mix[:got.value]

    def segment_finish(self, accum=None):
        accum = _u32(accum) if accum is not None else None
        cap = self.seal_words(self._po2)
        seal = np.empty(cap, np.uint32)
        got = C.c_size_t()
        self._check(self.lib.hfb200_segment_finish(self._h, _ptr(accum), _ptr(seal), cap, C.byref(got)))
        return seal[:got.value]

    def segment_begin_dev(self, po2, globals_, code, data, blind_seed, device_inputs=False):
        """hfb200_segment_begin_dev.  Host numpy arrays by default; device_inputs=True takes device addresses (ints, e.g.
        torch_tensor.data_ptr()) of columns on this context's device, copied device to device.  Returns the SegmentDev."""
        globals_ = _u32(globals_)
        if device_inputs:
            code_p, data_p = code, data
        else:
            code = _u32(code) if code is not None else None
            data = _u32(data) if data is not None else None
            code_p, data_p = _ptr(code), _ptr(data)
        seg = SegmentDev()
        self._check(self.lib.hfb200_segment_begin_dev(self._h, po2, _ptr(globals_), code_p, data_p, blind_seed,
                                                      DEV_INPUTS if device_inputs else 0, C.byref(seg)))
        self._po2 = po2
        return seg

    def segment_accum_scan(self, kind, first_chain, n_chains, rows):
        """In-place inclusive scan (SCAN_PRODUCT / SCAN_SUM) of the Fp4 chains in accum columns 4c..4c+3 over rows [0, rows)."""
        self._check(self.lib.hfb200_segment_accum_scan(self._h, int(kind), first_chain, n_chains, rows))

    def segment_accum_blind(self):
        self._check(self.lib.hfb200_segment_accum_blind(self._h))

    def segment_witness_dev(self, po2, blind_seed):
        """hfb200_segment_witness_dev: lays the context out for po2, derives the segment's blinding key and returns the WitnessDev
        whose data columns the caller writes; segment_begin / segment_begin_dev with data=None then commit them as they stand."""
        w = WitnessDev()
        self._check(self.lib.hfb200_segment_witness_dev(self._h, po2, blind_seed, C.byref(w)))
        self._po2 = po2
        return w

    def segment_data_blind(self):
        """Writes the blinding rows of every data column from the segment's key (between segment_witness_dev and the begin)."""
        self._check(self.lib.hfb200_segment_data_blind(self._h))

    def segment_scratch(self, nbytes):
        """Address of >= nbytes of device memory owned by the context (host memory in the emulator: see scratch_view)."""
        p = C.c_void_p()
        self._check(self.lib.hfb200_segment_scratch(self._h, nbytes, C.byref(p)))
        return p.value

    def segment_finish_dev(self):
        """Completes the segment from the accum columns as they stand in device memory."""
        cap = self.seal_words(self._po2)
        seal = np.empty(cap, np.uint32)
        got = C.c_size_t()
        self._check(self.lib.hfb200_segment_finish_dev(self._h, _ptr(seal), cap, C.byref(got)))
        return seal[:got.value]

    def witgen_synth(self, po2, trace_seed, blind_seed):
        g = np.empty(N_GLOBAL, np.uint32)
        self._check(self.lib.hfb200_witgen_synth(self._h, po2, trace_seed, blind_seed, _ptr(g)))
        self._po2 = po2
        return g

    def prove_resident(self, blind_seed):
        cap = self.seal_words(self._po2)
        seal = np.empty(cap, np.uint32)
        got = C.c_size_t()
        self._check(self.lib.hfb200_prove_resident(self._h, blind_seed, _ptr(seal), cap, C.byref(got)))
        return seal[:got.value]

    def read_group(self, group):
        w = {0: self.circuit[2], 1: self.circuit[0], 2: self.circuit[1]}[group]
        out = np.empty((w, 1 << self._po2), np.uint32)
        self._check(self.lib.hfb200_read_group(self._h, group, _ptr(out), out.size))
        return out

    def checkpoint(self, name):
        buf = np.empty(4096, np.uint32)
        got = C.c_size_t()
        self._check(self.lib.hfb200_checkpoint(self._h, name.encode(), _ptr(buf), buf.size, C.byref(got)))
        return buf[:got.value].copy()

    def checkpoints(self):
        out = {}
        for name in CHECKPOINT_NAMES:
            try:
                out[name] = self.checkpoint(name)
            except Hfb200Error:
                pass
        return out

    def host_alloc(self, shape):
        """Pinned host memory (cudaHostAlloc) viewed as a uint32 numpy array; freed with host_free(arr)."""
        n = int(np.prod(shape))
        p = C.c_void_p()
        self._check(self.lib.hfb200_host_alloc(n * 4, C.byref(p)))
        arr = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint32)), shape=(n,)).reshape(shape)
        self._pinned = getattr(self, "_pinned", {})
        self._pinned[arr.ctypes.data] = p
        return arr

    def host_free(self, arr):
        p = self._pinned.pop(arr.ctypes.data)
        self.lib.hfb200_host_free(p)

    def last_stats(self):
        s = Stats()
        self._check(self.lib.hfb200_last_stats(self._h, C.byref(s)))
        return s.as_dict()

    def total_launches(self):
        return self.lib.hfb200_total_launches(self._h)

    # ---- HAL-level operators ----
    def op_interpolate_ntt(self, cols, zk_shift=False):
        a = _u32(cols).copy()
        a2 = a.reshape(-1, a.shape[-1])
        self._check(self.lib.hfb200_op_interpolate_ntt(self._h, _ptr(a), a2.shape[0], a2.shape[1], int(zk_shift)))
        return a

    def op_expand_ntt(self, cols, expand_bits=2):
        a = _u32(cols)
        a2 = a.reshape(-1, a.shape[-1])
        out = np.empty((a2.shape[0], a2.shape[1] << expand_bits), np.uint32)
        self._check(self.lib.hfb200_op_expand_ntt(self._h, _ptr(out), _ptr(a), a2.shape[0], a2.shape[1], expand_bits))
        return out

    def op_lde(self, cols):
        a = _u32(cols)
        a2 = a.reshape(-1, a.shape[-1])
        out = np.empty((a2.shape[0], a2.shape[1] * 4), np.uint32)
        self._check(self.lib.hfb200_op_lde(self._h, _ptr(out), _ptr(a), a2.shape[0], a2.shape[1]))
        return out

    def op_merkle(self, matrix):
        m = _u32(matrix)
        cols, rows = m.shape
        nodes = np.empty((2 * rows, 8), np.uint32)
        self._check(self.lib.hfb200_op_merkle(self._h, _ptr(m), rows, cols, _ptr(nodes)))
        return nodes

    def op_poseidon2(self, states):
        s = _u32(states).copy()
        self._check(self.lib.hfb200_op_poseidon2(self._h, _ptr(s), s.size // 24))
        return s

    def op_fri_fold(self, coeffs, mix4):
        a = _u32(coeffs)
        n = a.shape[-1]
        out = np.empty((4, n // 16), np.uint32)
        m = _u32(mix4)
        self._check(self.lib.hfb200_op_fri_fold(self._h, _ptr(out), _ptr(a), n, _ptr(m)))
        return out

    def bench_lde(self, po2, count, iters):
        ms = C.c_float()
        self._check(self.lib.hfb200_bench_lde(self._h, po2, count, iters, C.byref(ms)))
        return ms.value

    def bench_merkle(self, po2, count, iters):
        ms = C.c_float()
        self._check(self.lib.hfb200_bench_merkle(self._h, po2, count, iters, C.byref(ms)))
        return ms.value

    def control_root(self, po2, code):
        """Control id of (circuit, po2): Merkle root of the committed code group (computed on the GPU)."""
        code = _u32(code)
        out = np.empty(8, np.uint32)
        self._check(self.lib.hfb200_control_root(self._h, po2, _ptr(code), _ptr(out)))
        self._po2 = po2  # the context now holds columns of this size
        return out

    def ir_jit_active(self):
        """(active, compile_ms): whether eval_check of this data-defined circuit runs the NVRTC-specialised kernel."""
        ms = C.c_float()
        a = self.lib.hfb200_ir_jit_active(self._h, C.byref(ms))
        return bool(a), ms.value

    def bench_modmul(self, kind, iters=1 << 15):
        """Modular products per second of instruction sequence `kind` (0 Montgomery, 1 Shoup, 2 S-box chain)."""
        r = C.c_double()
        self._check(self.lib.hfb200_bench_modmul(self._h, kind, iters, C.byref(r)))
        return r.value

    def mark(self, slot):
        """Records device-timeline mark `slot` (0..3) on this context's stream."""
        self._check(self.lib.hfb200_mark(self._h, slot))

    def mark_elapsed(self, slot_a, other, slot_b):
        """Device milliseconds from this context's mark slot_a to `other`'s mark slot_b."""
        ms = C.c_float()
        self._check(self.lib.hfb200_mark_elapsed(self._h, slot_a, other._h, slot_b, C.byref(ms)))
        return ms.value


class Hal:
    """The device HAL (hfb200_hal_*) over a Context: risc0-zkp `Hal` operators on buffers in the context's device memory.

    On a GPU build every buffer is a contiguous torch CUDA tensor of dtype int32 / uint32 on the context's device (its
    data_ptr() goes to the library); in the host emulator, whose device memory is host memory, buffers are contiguous uint32
    numpy arrays.  Shapes follow include/hfb200.h: base-field matrices [count, n], Fp4 buffers [..., 4].  Work is queued on the
    context's stream; call sync() before reading results on the host.  Host Fp4 values (mix, z) are sequences of 4 ints."""

    def __init__(self, ctx):
        self.ctx, self.lib, self._h = ctx, ctx.lib, ctx._h
        self.emulator = b"EMULATOR" in self.lib.hfb200_version()
        st, dev = C.c_void_p(), C.c_int()
        ctx._check(self.lib.hfb200_hal_stream(self._h, C.byref(st), C.byref(dev)))
        self.stream, self.device = st.value, dev.value

    def _a(self, buf, name):
        """Device address of `buf` after the checks the library cannot make (dtype, contiguity, and which memory kind)."""
        if self.emulator:
            if not isinstance(buf, np.ndarray) or buf.dtype != np.uint32 or not buf.flags.c_contiguous:
                raise Hfb200Error("Hal.%s: the host emulator takes contiguous uint32 numpy arrays" % name)
            return buf.ctypes.data
        import torch
        if not isinstance(buf, torch.Tensor) or not buf.is_cuda or buf.device.index != self.device:
            raise Hfb200Error("Hal.%s: expects a torch CUDA tensor on cuda:%d" % (name, self.device))
        if buf.dtype not in (torch.int32, torch.uint32) or not buf.is_contiguous():
            raise Hfb200Error("Hal.%s: expects a contiguous int32 / uint32 tensor" % name)
        return buf.data_ptr()

    def _run(self, e):
        self.ctx._check(e)

    @staticmethod
    def _e4(v):
        return np.ascontiguousarray(np.asarray(v, dtype=np.uint64).reshape(4), dtype=np.uint32)

    def sync(self):
        self._run(self.lib.hfb200_hal_sync(self._h))

    def host_syncs(self):
        return self.lib.hfb200_hal_host_syncs(self._h)

    def batch_interpolate_ntt(self, io):
        count, n = io.shape
        self._run(self.lib.hfb200_hal_batch_interpolate_ntt(self._h, self._a(io, "batch_interpolate_ntt"), count, n))

    def zk_shift(self, io):
        count, n = io.shape
        self._run(self.lib.hfb200_hal_zk_shift(self._h, self._a(io, "zk_shift"), count, n))

    def batch_expand_into_evaluate_ntt(self, out, inp, expand_bits):
        count, n_in = inp.shape
        if tuple(out.shape) != (count, n_in << expand_bits):
            raise Hfb200Error("Hal.batch_expand_into_evaluate_ntt: out must be [count, n_in << expand_bits]")
        self._run(self.lib.hfb200_hal_batch_expand_into_evaluate_ntt(self._h, self._a(out, "expand"), self._a(inp, "expand"), count, n_in, expand_bits))

    def batch_bit_reverse(self, io):
        count, n = io.shape
        self._run(self.lib.hfb200_hal_batch_bit_reverse(self._h, self._a(io, "batch_bit_reverse"), count, n))

    def hash_rows(self, digests, matrix):
        """digests [rows, 8] <- leaf digest of every row of matrix [cols, rows]."""
        cols, rows = matrix.shape
        if tuple(digests.shape) != (rows, 8):
            raise Hfb200Error("Hal.hash_rows: digests must be [rows, 8]")
        self._run(self.lib.hfb200_hal_hash_rows(self._h, self._a(digests, "hash_rows"), self._a(matrix, "hash_rows"), rows, cols))

    def hash_fold(self, io, input_size, output_size):
        """io [2 * rows, 8] heap-layout nodes: level output_size from level input_size."""
        self._run(self.lib.hfb200_hal_hash_fold(self._h, self._a(io, "hash_fold"), input_size, output_size))

    def merkle_tree(self, nodes, matrix):
        """hash_rows into the leaf level of nodes [2 * rows, 8], then every fold: the whole tree through the HAL."""
        rows = matrix.shape[1]
        self.hash_rows(nodes[rows:], matrix)
        size = rows
        while size > 1:
            self.hash_fold(nodes, size, size // 2)
            size //= 2

    def batch_evaluate_any(self, coeffs, which, xs, out):
        """out[j] = sum_k coeffs[which[j]][k] * xs[j]^k; coeffs [poly_count, n], which [count], xs / out [count, 4]."""
        poly_count, n = coeffs.shape
        count = which.shape[0]
        self._run(self.lib.hfb200_hal_batch_evaluate_any(self._h, self._a(coeffs, "batch_evaluate_any"), poly_count, n, self._a(which, "batch_evaluate_any"),
                                                         self._a(xs, "batch_evaluate_any"), self._a(out, "batch_evaluate_any"), count))

    def mix_poly_coeffs(self, out, mix_start, mix, inp, combo_of_col):
        """out [n_combos, n, 4] += mix_start * mix^c * inp[c] into combo combo_of_col[c]; inp [n_cols, n]."""
        n_cols, n = inp.shape
        n_combos = out.shape[0]
        ms, m = self._e4(mix_start), self._e4(mix)
        self._run(self.lib.hfb200_hal_mix_poly_coeffs(self._h, self._a(out, "mix_poly_coeffs"), _ptr(ms), _ptr(m), self._a(inp, "mix_poly_coeffs"),
                                                      self._a(combo_of_col, "mix_poly_coeffs"), n_cols, n, n_combos))

    def poly_divide(self, poly, z, remainder):
        """poly [n, 4] <- quotient of poly / (x - z) (last element 0); remainder [4] (device) <- poly(z)."""
        zz = self._e4(z)
        self._run(self.lib.hfb200_hal_poly_divide(self._h, self._a(poly, "poly_divide"), poly.shape[0], _ptr(zz), self._a(remainder, "poly_divide")))

    def eltwise_add_elem(self, out, x, y):
        self._run(self.lib.hfb200_hal_eltwise_add_elem(self._h, self._a(out, "eltwise_add_elem"), self._a(x, "eltwise_add_elem"), self._a(y, "eltwise_add_elem"), _numel(out)))

    def eltwise_sum_extelem(self, out, inp):
        """out [4, count] <- components of sum_g inp[g]; inp [to_add, count, 4]."""
        to_add, count = inp.shape[0], inp.shape[1]
        self._run(self.lib.hfb200_hal_eltwise_sum_extelem(self._h, self._a(out, "eltwise_sum_extelem"), self._a(inp, "eltwise_sum_extelem"), count, to_add))

    def eltwise_copy_elem(self, out, inp):
        self._run(self.lib.hfb200_hal_eltwise_copy_elem(self._h, self._a(out, "eltwise_copy_elem"), self._a(inp, "eltwise_copy_elem"), _numel(out)))

    def eltwise_zeroize_elem(self, io):
        self._run(self.lib.hfb200_hal_eltwise_zeroize_elem(self._h, self._a(io, "eltwise_zeroize_elem"), _numel(io)))

    def gather_sample(self, dst, src, idx, stride):
        self._run(self.lib.hfb200_hal_gather_sample(self._h, self._a(dst, "gather_sample"), self._a(src, "gather_sample"), idx, _numel(dst), stride))

    def scatter(self, into, index, offsets, values):
        self._run(self.lib.hfb200_hal_scatter(self._h, self._a(into, "scatter"), self._a(index, "scatter"), self._a(offsets, "scatter"),
                                              self._a(values, "scatter"), _numel(index) - 1))

    def prefix_products(self, io):
        """io [n, 4] <- inclusive running product."""
        self._run(self.lib.hfb200_hal_prefix_products(self._h, self._a(io, "prefix_products"), io.shape[0]))

    def fri_fold(self, out, inp, mix):
        """out [4, n/16] <- fold of inp [4, n] by mix ([4], device)."""
        self._run(self.lib.hfb200_hal_fri_fold(self._h, self._a(out, "fri_fold"), self._a(inp, "fri_fold"), inp.shape[1], self._a(mix, "fri_fold")))


def _numel(a):
    return int(a.numel()) if hasattr(a, "numel") and callable(a.numel) else int(a.size)


def device_count(lib=None):
    """Number of CUDA devices (hfb200_device_count); 0 without a device or a driver."""
    lib = lib or load_library()
    n = C.c_int()
    _raise_err(lib, lib.hfb200_device_count(C.byref(n)))
    return n.value


class SegmentHandle:
    """What a Python accum callback of Pool.set_accum may call on the context it is given."""

    def __init__(self, lib, ctx):
        self.lib, self._h = lib, ctx

    def accum_scan(self, kind, first_chain, n_chains, rows):
        _raise_err(self.lib, self.lib.hfb200_segment_accum_scan(self._h, int(kind), first_chain, n_chains, rows))

    def accum_blind(self):
        _raise_err(self.lib, self.lib.hfb200_segment_accum_blind(self._h))


class WitnessHandle:
    """What a Python witgen callback of Pool.set_witgen may call on the context it is given."""

    def __init__(self, lib, ctx):
        self.lib, self._h = lib, ctx

    def scratch(self, nbytes):
        p = C.c_void_p()
        _raise_err(self.lib, self.lib.hfb200_segment_scratch(self._h, nbytes, C.byref(p)))
        return p.value

    def data_blind(self):
        _raise_err(self.lib, self.lib.hfb200_segment_data_blind(self._h))


def verify_segment(seal, code_root, circuit=(16, 192, 48), ir=None, lib=None):
    """`Receipt::verify` for one segment seal (hfb200_verify_segment; host-side like the reference's verifier, no GPU
    needed).  Returns the segment's po2; raises Hfb200Error with the reason when the seal is rejected."""
    lib = lib or load_library()
    seal, code_root = _u32(seal), _u32(code_root)
    if code_root.size != 8:
        raise Hfb200Error("verify_segment: code_root must have 8 words")
    po2 = C.c_uint32()
    if ir is not None:
        taps, steps = _u32(ir["taps"]), _u32(ir["steps"])
        d = _mk_ir(ir, circuit[0], circuit[1], circuit[2], int(ir["n_mix"]), taps.ctypes.data, taps.size // 3, steps.ctypes.data, steps.size // 4, int(ir["ret"]))
        e = lib.hfb200_verify_segment(None, C.byref(d), _ptr(seal), seal.size, _ptr(code_root), C.byref(po2))
    else:
        d = CircuitDesc(circuit[0], circuit[1], circuit[2], 0)
        e = lib.hfb200_verify_segment(C.byref(d), None, _ptr(seal), seal.size, _ptr(code_root), C.byref(po2))
    if e:
        msg = C.cast(e, C.c_char_p).value.decode(errors="replace")
        lib.hfb200_free_error(e)
        raise Hfb200Error(msg)
    return po2.value


def _raise_err(lib, e):
    if e:
        msg = C.cast(e, C.c_char_p).value.decode(errors="replace")
        lib.hfb200_free_error(e)
        raise Hfb200Error(msg)


def digest_bytes(data, lib=None):
    """Poseidon2 digest of a byte string (hfb200_digest_bytes): the journal digest of this path's claims."""
    lib = lib or load_library()
    out = np.zeros(8, np.uint32)
    data = bytes(data)
    _raise_err(lib, lib.hfb200_digest_bytes(data, len(data), _ptr(out)))
    return out


def digest_pair(a, b, lib=None):
    lib = lib or load_library()
    a, b, out = _u32(a), _u32(b), np.zeros(8, np.uint32)
    _raise_err(lib, lib.hfb200_digest_pair(_ptr(a), _ptr(b), _ptr(out)))
    return out


def claim_next_state(pre, index, po2, lib=None):
    lib = lib or load_library()
    pre, out = _u32(pre), np.zeros(8, np.uint32)
    _raise_err(lib, lib.hfb200_claim_next_state(_ptr(pre), index, po2, _ptr(out)))
    return out


def claim_encode(globals_, pre, post, exit_code, output, lib=None):
    """Returns a copy of the 32 globals with the claim words written (hfb200_claim_encode)."""
    lib = lib or load_library()
    g = _u32(globals_).copy()
    c = Claim()
    c.pre[:] = [int(x) for x in pre]; c.post[:] = [int(x) for x in post]; c.output[:] = [int(x) for x in output]
    c.exit_code = int(exit_code)
    _raise_err(lib, lib.hfb200_claim_encode(C.byref(c), _ptr(g)))
    return g


def claim_decode(seal, lib=None):
    lib = lib or load_library()
    seal = _u32(seal)
    c = Claim()
    _raise_err(lib, lib.hfb200_claim_decode(_ptr(seal), seal.size, C.byref(c)))
    return c


def verify_segments(seals, code_roots, circuit=(16, 192, 48), ir=None, threads=0, lib=None):
    """`hfb200_verify_segments`: the segment seals of a composite receipt checked on `threads` host threads (0 = all hardware
    threads).  `code_roots`: one 8-word control id per seal.  Returns the po2 of every seal; raises Hfb200Error naming the
    first rejected seal."""
    lib = lib or load_library()
    seals = [_u32(s) for s in seals]
    roots = np.ascontiguousarray(np.stack([_u32(r) for r in code_roots]) if len(code_roots) else np.zeros((0, 8), np.uint32), dtype=np.uint32)
    n = len(seals)
    if roots.shape != (n, 8):
        raise Hfb200Error("verify_segments: one 8-word control id per seal")
    ptrs = (C.c_void_p * max(n, 1))(*[s.ctypes.data for s in seals])
    lens = (C.c_size_t * max(n, 1))(*[s.size for s in seals])
    po2 = np.zeros(max(n, 1), dtype=np.uint32)
    bad = C.c_size_t(n)
    if ir is not None:
        taps, steps = _u32(ir["taps"]), _u32(ir["steps"])
        d = _mk_ir(ir, circuit[0], circuit[1], circuit[2], int(ir["n_mix"]), taps.ctypes.data, taps.size // 3, steps.ctypes.data, steps.size // 4, int(ir["ret"]))
        e = lib.hfb200_verify_segments(None, C.byref(d), ptrs, lens, n, _ptr(roots) if n else None, _ptr(po2), threads, C.byref(bad))
    else:
        d = CircuitDesc(circuit[0], circuit[1], circuit[2], 0)
        e = lib.hfb200_verify_segments(C.byref(d), None, ptrs, lens, n, _ptr(roots) if n else None, _ptr(po2), threads, C.byref(bad))
    _raise_err(lib, e)
    return [int(x) for x in po2[:n]]


def verify_claims(seals, image_id, journal_bytes, lib=None):
    """The claim chain of `receipt.verify(image_id)` over seals in segment order (hfb200_verify_claims)."""
    lib = lib or load_library()
    seals = [_u32(s) for s in seals]
    n = len(seals)
    ptrs = (C.c_void_p * n)(*[s.ctypes.data for s in seals])
    lens = (C.c_size_t * n)(*[s.size for s in seals])
    image_id = _u32(image_id)
    if image_id.size != 8:
        raise Hfb200Error("verify_claims: image id must have 8 words")
    journal_bytes = bytes(journal_bytes)
    _raise_err(lib, lib.hfb200_verify_claims(ptrs, lens, n, _ptr(image_id), journal_bytes, len(journal_bytes)))


def ir_source(ir, circuit, lib=None):
    """CUDA source that hfb200_init_ir compiles for the eval_check of a data-defined circuit (needs no device)."""
    lib = lib or load_library()
    taps, steps = _u32(ir["taps"]), _u32(ir["steps"])
    desc = _mk_ir(ir, circuit[0], circuit[1], circuit[2], int(ir["n_mix"]), taps.ctypes.data, taps.size // 3, steps.ctypes.data, steps.size // 4, int(ir["ret"]))
    need = C.c_size_t()
    e = lib.hfb200_ir_source(C.byref(desc), None, 0, C.byref(need))
    if e:
        msg = C.cast(e, C.c_char_p).value.decode(errors="replace"); lib.hfb200_free_error(e); raise Hfb200Error(msg)
    buf = C.create_string_buffer(need.value)
    e = lib.hfb200_ir_source(C.byref(desc), buf, need.value, C.byref(need))
    if e:
        msg = C.cast(e, C.c_char_p).value.decode(errors="replace"); lib.hfb200_free_error(e); raise Hfb200Error(msg)
    return buf.value.decode()


class Pool:
    """hfb200_pool: worker contexts on several GPUs fed from one queue of independent segments (no collectives).
    Mirrors the segment loop of upstream's `ProverImpl::prove_session`."""

    def __init__(self, devices=(0,), contexts_per_device=1, max_po2=20, circuit=(16, 192, 48), lib=None, ir=None, deterministic=None):
        self.lib = lib or load_library()
        self.circuit = tuple(int(x) for x in circuit)
        devs = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        self._h = None
        if ir is not None:
            taps, steps = _u32(ir["taps"]), _u32(ir["steps"])
            desc = _mk_ir(ir, self.circuit[0], self.circuit[1], self.circuit[2], int(ir["n_mix"]), taps.ctypes.data, taps.size // 3,
                             steps.ctypes.data, steps.size // 4, int(ir["ret"]))
            e = self.lib.hfb200_pool_create_ir(devs, len(devices), contexts_per_device, max_po2, C.byref(desc), C.byref(h))
        else:
            desc = CircuitDesc(self.circuit[0], self.circuit[1], self.circuit[2], 0)
            e = self.lib.hfb200_pool_create(devs, len(devices), contexts_per_device, max_po2, C.byref(desc), C.byref(h))
        self._raise(e)
        self._h = h
        self.workers = len(devices) * contexts_per_device
        self._raise(self.lib.hfb200_pool_set_blinding(self._h, _default_blinding(deterministic)))
        self.last_attempts = []

    def stats(self):
        st = PoolStats()
        self._raise(self.lib.hfb200_pool_stats(self._h, C.byref(st)))
        return st.as_dict()

    def inject_fault(self, worker, after_jobs=0, kind=0):
        """Test hook (hfb200_pool_inject_fault): kind 0 = device fault (context re-created, job re-queued), 1 = plain failure."""
        self._raise(self.lib.hfb200_pool_inject_fault(self._h, worker, after_jobs, kind))

    def _raise(self, e):
        if e:
            msg = C.cast(e, C.c_char_p).value.decode(errors="replace")
            self.lib.hfb200_free_error(e)
            raise Hfb200Error(msg)

    def set_accum(self, fn, user=None):
        """The caller's step_accum for every job (hfb200_pool_set_accum); None removes it.
        `fn` is either the address (int) of a C function `int fn(void* user, hfb200_ctx*, const hfb200_segment_dev*, size_t job)`
        -- `user` is then passed through as a pointer (int or None) -- or a Python callable fn(ctx, seg, job) with ctx a
        SegmentHandle (accum_scan / accum_blind) and seg the SegmentDev.  A Python callback runs on the worker threads, one at a
        time under the GIL; an exception fails that job only and its text appears in the job's error."""
        self._accum_errors = {}
        if fn is None:
            self._accum_cb = None
            self._raise(self.lib.hfb200_pool_set_accum(self._h, None, None))
            return
        if isinstance(fn, int):
            self._accum_cb = None
            self._raise(self.lib.hfb200_pool_set_accum(self._h, fn, user))
            return
        lib, errors = self.lib, self._accum_errors

        def trampoline(_user, ctx, seg, job):
            try:
                fn(SegmentHandle(lib, ctx), seg.contents, int(job))
                return 0
            except BaseException as e:  # noqa: B036 -- nothing may unwind into the C worker thread
                errors[int(job)] = "%s: %s" % (type(e).__name__, e)
                return 1
        self._accum_cb = ACCUM_FN(trampoline)  # kept alive as long as the pool may call it
        self._raise(self.lib.hfb200_pool_set_accum(self._h, C.cast(self._accum_cb, C.c_void_p).value, None))

    def set_witgen(self, fn, user=None):
        """The caller's witness generator for every job whose data is None (hfb200_pool_set_witgen); None removes it.
        `fn` is either the address (int) of a C function `int fn(void* user, hfb200_ctx*, const hfb200_witness_dev*, size_t job)`
        -- `user` is then passed through as a pointer (int or None) -- or a Python callable fn(ctx, w, job) with ctx a
        WitnessHandle (scratch / data_blind) and w the WitnessDev.  A Python callback runs on the worker threads, one at a time
        under the GIL; an exception fails that job only and its text appears in the job's error."""
        self._witgen_errors = {}
        if fn is None:
            self._witgen_cb = None
            self._raise(self.lib.hfb200_pool_set_witgen(self._h, None, None))
            return
        if isinstance(fn, int):
            self._witgen_cb = None
            self._raise(self.lib.hfb200_pool_set_witgen(self._h, fn, user))
            return
        lib, errors = self.lib, self._witgen_errors

        def trampoline(_user, ctx, w, job):
            try:
                fn(WitnessHandle(lib, ctx), w.contents, int(job))
                return 0
            except BaseException as e:  # noqa: B036 -- nothing may unwind into the C worker thread
                errors[int(job)] = "%s: %s" % (type(e).__name__, e)
                return 1
        self._witgen_cb = WITGEN_FN(trampoline)  # kept alive as long as the pool may call it
        self._raise(self.lib.hfb200_pool_set_witgen(self._h, C.cast(self._witgen_cb, C.c_void_p).value, None))

    def close(self):
        if self._h:
            self.lib.hfb200_pool_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def load_control(self, po2, code):
        """Shared control group of the po2-sized segments: jobs of that po2 may then pass code=None (identical seals)."""
        if not hasattr(self, "_control"):
            self._control = {}
        if code is None:
            self._control.pop(po2, None)
            self._raise(self.lib.hfb200_pool_load_control(self._h, po2, None))
            return
        code = _u32(code)
        if code.size != self.circuit[0] << po2:
            raise Hfb200Error("load_control: control columns do not match (circuit, po2)")
        self._control[po2] = code  # keeps the buffer alive: the library holds the pointer
        self._raise(self.lib.hfb200_pool_load_control(self._h, po2, _ptr(code)))

    def prove(self, jobs, seal_cap, return_errors=False):
        """jobs: list of (po2, globals, code, data, blind_seed) with numpy u32 arrays (code may be None after load_control, data
        None with a witgen callback).
        Returns (seals, devices, ms); raises on the first failed job unless return_errors=True, in which case the result is
        (seals, devices, ms, errors) with errors[i] = None or the job's message (failed jobs have an empty seal; the others are
        proved regardless, like the reference's batch tooling sets failed inputs aside)."""
        n = len(jobs)
        arr = (SegmentJob * n)()
        keep = []
        seals = [np.empty(seal_cap, np.uint32) for _ in range(n)]
        for i, (po2, g, code, data, seed) in enumerate(jobs):
            g = _u32(g)
            code = _u32(code) if code is not None else None
            data = _u32(data) if data is not None else None
            rows = 1 << po2
            if g.size != N_GLOBAL or (data is not None and data.size != self.circuit[1] * rows) or (code is not None and code.size != self.circuit[0] * rows):
                raise Hfb200Error("pool.prove: job %d: trace shape does not match (circuit, po2)" % i)
            keep.append((g, code, data))
            arr[i].po2, arr[i].blind_seed = po2, seed
            arr[i].globals, arr[i].code = g.ctypes.data, (code.ctypes.data if code is not None else None)
            arr[i].data = data.ctypes.data if data is not None else None
            arr[i].seal_out, arr[i].seal_cap = seals[i].ctypes.data, seal_cap
        accum_errors = getattr(self, "_accum_errors", {})
        accum_errors.clear()
        witgen_errors = getattr(self, "_witgen_errors", {})
        witgen_errors.clear()
        e = self.lib.hfb200_pool_prove(self._h, arr, n)
        errs = [None] * n
        for i in range(n):
            if arr[i].error:
                errs[i] = C.cast(arr[i].error, C.c_char_p).value.decode(errors="replace")
                self.lib.hfb200_free_error(arr[i].error)
                # a Python callback's own exception
                if i in witgen_errors and errs[i].startswith("witgen callback returned"):
                    errs[i] += ": " + witgen_errors[i]
                elif i in accum_errors:
                    errs[i] += ": " + accum_errors[i]
        self.last_attempts = [arr[i].attempts for i in range(n)]
        out = ([seals[i][:arr[i].seal_words] if errs[i] is None else seals[i][:0] for i in range(n)], [arr[i].device for i in range(n)],
               [arr[i].ms for i in range(n)])
        if return_errors:
            if e:
                self.lib.hfb200_free_error(e)
            return out + (errs,)
        if e and (accum_errors or witgen_errors):
            self.lib.hfb200_free_error(e)  # the library's message lacks the callback's text: report the job's own
            i = next(k for k in range(n) if errs[k] is not None)
            raise Hfb200Error("job %d: %s" % (i, errs[i]))
        self._raise(e)
        first = [m for m in errs if m is not None]
        if first:
            raise Hfb200Error(first[0])
        return out
