/*
 * hfb200.h -- C ABI of the B200-native STARK segment prover (libhfb200.so).
 *
 * Drop-in boundary for the ONE hot path of element36-io/hyperfridge-r0: the call
 *     let prover = default_prover();                       (/root/reference/host/src/main.rs:420)
 *     prover.prove(env, HYPERFRIDGE_ELF)                   (/root/reference/host/src/main.rs:423)
 * which, per segment, runs risc0-circuit-rv32im 4.0.4 `SegmentProver::prove(&Segment) -> Seal` on top of
 * risc0-zkp 3.0.4's `Hal` / `CircuitHal` traits (/root/reference/Cargo.lock:3087-3223; crates not vendored).
 * The library sits at that `SegmentProver` seam: trace columns in, seal (u32 words) out.
 *
 * Conventions (same as upstream's sys crates, risc0-sys `ffi_wrap`):
 *   - every entry returns `const char*`: NULL = success, otherwise a malloc'd message that the caller
 *     releases with hfb200_free_error().  No exceptions or aborts cross the ABI.
 *   - matrices are column-major u32[w][N] BabyBear residues in MONTGOMERY form (R = 2^32), N = 2^po2.
 *   - a context is single-owner: one host thread <-> one GPU <-> its stream.  Distinct contexts are
 *     independent (one per GPU for multi-GPU operation; segments are independent, no collectives).
 *   - the caller owns every host pointer for the duration of the call; the library owns device memory.
 *   - there is NO CPU fallback: without a CUDA device hfb200_init fails.
 */
#ifndef HFB200_H
#define HFB200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hfb200_ctx hfb200_ctx;

/* Circuit plug-in descriptor.  Replaces the generated rv32im circuit (taps + poly_fp + step_accum of
 * risc0-circuit-rv32im[-sys], /root/reference/Cargo.lock:3087-3132), which is not obtainable here; the
 * built-in plug-in is the declared stand-in "synth-rv32im-shape v1" (DESIGN.md, oracle/circuit.h). */
typedef struct {
    uint32_t w_code;  /* control columns  (>= 5)            default 16  */
    uint32_t w_data;  /* data columns     (multiple of 4)   default 192 */
    uint32_t w_accum; /* accum columns    (multiple of 4)   default 48  */
    uint32_t flags;   /* reserved, 0 */
} hfb200_circuit_desc;

/* Circuit as DATA (SURVEY.md section 8b `hfb200_circuit_register`): what upstream ships as generated code is accepted
 * here as tables, in upstream's own shapes --
 *   taps  : risc0_zkp::taps::TapSet  -- (group, offset, back) sorted; group ids 0 = accum, 1 = code, 2 = data
 *   steps : risc0_zkp::adapter::PolyExtStepDef -- Const / Get / GetGlobal / Add / Sub / Mul / True / AndEqz / AndCond;
 *           fp vars and mix vars are two SSA index spaces, every step pushes one; `ret` = mix var of the result.
 *           CONST a = canonical value | GET a = tap index | GET_GLOBAL a = 0 (globals) / 1 (mix), b = offset |
 *           ADD/SUB/MUL a, b = fp vars | TRUE | AND_EQZ a = mix var, b = fp var | AND_COND a = mix var, b = fp cond, c = inner mix var
 * Limits: <= 4 taps per register, <= 4 distinct back values, <= 8 distinct tap sets.  For a data-defined circuit the
 * witness and the accum columns are the caller's: two-phase API, either on the host (hfb200_segment_begin / _finish with
 * the columns) or on the device (hfb200_segment_begin_dev / _finish_dev, or a pool with hfb200_pool_set_accum);
 * hfb200_witgen_synth / finish(NULL) are refused. */
typedef struct { uint32_t group, offset, back; } hfb200_tap;
typedef struct { uint32_t op, a, b, c; } hfb200_poly_step;
enum { HFB200_OP_CONST = 0, HFB200_OP_GET = 1, HFB200_OP_GET_GLOBAL = 2, HFB200_OP_ADD = 3, HFB200_OP_SUB = 4, HFB200_OP_MUL = 5,
       HFB200_OP_TRUE = 6, HFB200_OP_AND_EQZ = 7, HFB200_OP_AND_COND = 8 };
typedef struct {
    uint32_t w_code, w_data, w_accum; /* group widths */
    uint32_t n_mix;                   /* accum mix elements drawn after the DATA commit (upstream REGCOUNT_MIX) */
    const hfb200_tap* taps;
    size_t n_taps;
    const hfb200_poly_step* steps;
    size_t n_steps;
    uint32_t ret;
    uint8_t info[16];                 /* upstream `CircuitImpl::CIRCUIT_INFO` (risc0-zkp `ProtocolInfo`): hashed into the transcript right
                                         after the proof-system info; all zero = "RV32IM:v2_______" (upstream's rv32im-v2 string) */
} hfb200_circuit_ir;

#define HFB200_N_GLOBAL 32u
#define HFB200_DIGEST_WORDS 8u

/* ---- lifetime ------------------------------------------------------------------------------- */
/* Replaces `segment_prover(hashfn)` / HAL construction.  Allocates the device arena for segments up to
 * 2^max_po2 cycles (12 <= max_po2 <= 22) and registers the circuit. */
const char* hfb200_init(int device, uint32_t max_po2, const hfb200_circuit_desc* circuit, hfb200_ctx** out);
const char* hfb200_init_ir(int device, uint32_t max_po2, const hfb200_circuit_ir* circuit, hfb200_ctx** out);
/* Same, for a circuit given as data.  The constraint polynomial is cut along its top-level AndEqz / AndCond chain into chunks of
 * ~400 steps (HFB200_IR_CHUNK); every chunk becomes one straight-line kernel (its body looped over the rows, so that it runs out of the
 * instruction cache), specialised with NVRTC for sm_100a AND for the segment
 * size (tap offsets become literals): loaded at init for max_po2, for other sizes when first proved.
 * The cubins live in a process-wide cache keyed by a Poseidon2 digest of each chunk's whole NVRTC input (options, prelude,
 * source), so every (circuit, po2) is compiled once per process, on up to 8 host threads; concurrent contexts wait for that
 * one compile.  A size that is not cached while NVRTC is unavailable runs the interpreter kernel (same seals).
 * HFB200_NVRTC_LIB=<path> names the NVRTC library in place of the built-in search list. */
/* The CUDA source of those kernels for po2 = 20 (one thread per LDE row, one kernel per chunk).  Needs no device.  Writes at most
 * `cap` bytes including the terminating NUL; *need = bytes required. */
const char* hfb200_ir_source(const hfb200_circuit_ir* circuit, char* out, size_t cap, size_t* need);
/* 1 when the context's eval_check runs the NVRTC-specialised kernel for its max_po2, 0 when it runs the interpreter kernel
 * (built-in circuit: 0).  *compile_ms (may be NULL) = wall time of the most recent specialisation (sources + cache lookup +
 * NVRTC for the chunks not cached + load). */
int hfb200_ir_jit_active(const hfb200_ctx* ctx, float* compile_ms);
/* Compiles the specialised eval_check kernels of `circuit` for each po2 in po2s (12..22) into the process cache.
 * Needs NVRTC, not a device.  Sizes already cached are not recompiled.
 * bundle_out == NULL and need == NULL: only warm the cache.  need != NULL: *need = bytes of the bundle that serialises every
 * requested specialisation, ready for hfb200_ir_load_kernels.  bundle_out != NULL: that bundle (cap >= *need, else an error).
 * Serialised from the cache, so the same request gives the same bytes.  threads = 0: up to 8 compile threads.
 * Bundle: magic "HFB200KB", format version, arch ("sm_100a"), per (circuit, po2) its (key, cubin) records, then a Poseidon2
 * digest over everything before it.  The host emulator build returns an error. */
const char* hfb200_ir_compile(const hfb200_circuit_ir* circuit, const uint32_t* po2s, size_t n_po2, unsigned threads,
                              void* bundle_out, size_t cap, size_t* need);
/* Adds a bundle's cubins to the process cache.  Needs no device and no NVRTC.  A bundle for another circuit or other
 * code-generation settings loads but never matches.  A malformed bundle (bad magic, version or arch, truncated, digest
 * mismatch) is refused whole, with nothing added.  *specialisations (optional) = (circuit, po2) entries the bundle carries,
 * all of them now cached.  The host emulator build returns an error. */
const char* hfb200_ir_load_kernels(const void* bundle, size_t bytes, size_t* specialisations);
/* NVRTC programs this process has compiled (tests, probes). */
uint64_t hfb200_ir_nvrtc_programs(void);
void hfb200_destroy(hfb200_ctx* ctx);
void hfb200_free_error(const char* msg);

/* Zero-knowledge blinding.  Upstream draws the blinding rows of every proof from a cryptographic RNG (risc0-zkp
 * `Elem::random(&mut thread_rng())`).  The library does the same by DEFAULT: per segment, a 256-bit key from the OS
 * (getrandom) expanded by the ChaCha20 block function on the device (csrc/blind.cuh); the `blind_seed` arguments below are
 * then only mixed into that key and seals are NOT reproducible.  HFB200_BLIND_DETERMINISTIC derives the key from the 64-bit
 * `blind_seed` alone: reproducible seals for parity tests and benchmarks, NOT zero-knowledge against anyone who can guess
 * the seed -- never use it for real statements. */
enum { HFB200_BLIND_OS_ENTROPY = 0, HFB200_BLIND_DETERMINISTIC = 1 };
const char* hfb200_set_blinding(hfb200_ctx* ctx, int mode);
/* Where the Fiat-Shamir transcript (upstream: WriteIOP + Poseidon2Rng on the host) of the ONE-SHOT entries runs for the built-in circuit.
 * 0 (default): on the host, 10 stream synchronisations per segment, each a true dependency.  1: on the device as one-warp kernels,
 * the seal assembled in device memory, ONE synchronisation per segment (csrc/transcript.cuh); identical seals.  Measured ~1 % slower on
 * B200 (a segment's transcript is ~170 sequential Poseidon2 permutations, 3.3 us each on a warp against ~1 us on a host core); for hosts
 * with few cores per GPU.  2: mode 1 replayed as a CUDA GRAPH: the first segment of a (po2, control-reuse) shape runs plainly, the
 * second is captured and instantiated, every later one refills the pinned parameter staging area and issues one cudaGraphLaunch
 * (trace uploads from caller memory stay outside the graph); identical seals; per-stage times are not available for replayed
 * segments (hfb200_last_stats reports ms_device only).  HFB200_DEVICE_TRANSCRIPT=1|2 in the environment selects a mode for
 * contexts that never call this. */
const char* hfb200_set_transcript(hfb200_ctx* ctx, int mode);
/* Hash suite of the context: upstream's `segment_prover(hashfn)` with hashfn "poseidon2" (default) or "sha-256".  It selects the
 * Merkle hash of every tree the context commits (leaves: hash of the row's raw Montgomery words; nodes: hash_pair of two
 * digests) and the transcript's hash and RNG (Poseidon2Rng, or ShaRng).  Digests are 8 words in both suites, so the seal layout,
 * hfb200_seal_words and the checkpoint names stay the same; the control id differs (upstream keeps one control-id table per
 * hashfn).  SHA-256 digest words, read as little-endian bytes, are the standard SHA-256 output bytes.
 *   - valid between segments; a change drops the resident control group (a code == NULL segment then needs hfb200_control_root
 *     again, and a pool re-commits its loaded control group on that context);
 *   - hfb200_control_root, hfb200_op_merkle, the one-shot, two-phase and device entries, the accum / witgen callbacks of a pool
 *     and hfb200_bench_merkle follow the context's suite; the hfb200_hal_* operators name their suite themselves;
 *   - SHA-256 runs the host transcript only: hfb200_set_transcript(ctx, 1 | 2) on a SHA-256 context is an error, so is
 *     switching a context set to mode 1 or 2 to SHA-256, and HFB200_DEVICE_TRANSCRIPT does not apply to SHA-256 contexts;
 *   - seals verify with hfb200_verify_segment_suite / _segments_suite under the same suite;
 *   - the claim digests (hfb200_digest_bytes, hfb200_digest_pair) stay Poseidon2 in both suites. */
enum { HFB200_HASH_POSEIDON2 = 0, HFB200_HASH_SHA256 = 1 };
const char* hfb200_set_hash_suite(hfb200_ctx* ctx, int suite);
/* Segments of this context that were issued as one cudaGraphLaunch (transcript mode 2). */
uint64_t hfb200_graph_launches(const hfb200_ctx* ctx);
const char* hfb200_version(void);

/* Pinned host memory for trace staging (plain pointers are accepted too, just slower over PCIe). */
const char* hfb200_host_alloc(size_t bytes, void** out);
void hfb200_host_free(void* p);

/* ---- the segment prover (replaces SegmentProver::prove) ------------------------------------- */
/* One-shot: host trace in, seal out.  `code` = control columns u32[w_code][N], `data` = witness columns
 * u32[w_data][N] with their blinding rows already filled by the witness generator (upstream's
 * WitnessGenerator does the same); `blind_seed` fixes the blinding noise of the accum group, which the
 * library derives on the device (step_accum).  On success *seal_words = words written.  If seal_cap is too
 * small an error is returned and *seal_words holds the required size. */
const char* hfb200_prove_segment(hfb200_ctx* ctx, uint32_t po2, const uint32_t* globals /*[32]*/,
                                 const uint32_t* code, const uint32_t* data, uint64_t blind_seed,
                                 uint32_t* seal_out, size_t seal_cap, size_t* seal_words);

/* Two-phase form (SURVEY.md section 8b): begin commits CODE and DATA and returns the accum mix
 * (Fiat-Shamir) so an external step_accum can run; finish takes the accum columns (or NULL to let the
 * built-in plug-in compute them on the device) and completes the seal. */
const char* hfb200_segment_begin(hfb200_ctx* ctx, uint32_t po2, const uint32_t* globals, const uint32_t* code,
                                 const uint32_t* data, uint64_t blind_seed, uint32_t* mix_out, size_t mix_cap, size_t* mix_words);
const char* hfb200_segment_finish(hfb200_ctx* ctx, const uint32_t* accum_or_null, uint32_t* seal_out, size_t seal_cap, size_t* seal_words);

/* Two-phase form on DEVICE memory (upstream's GPU path keeps witgen and step_accum on the device).  begin_dev is
 * hfb200_segment_begin plus a description of the segment in flight: the committed columns, the mix and the writable accum
 * columns, all in the context's device memory.  The caller's step_accum writes the accum columns in place, on `stream` or on
 * its own streams; finish_dev then commits them as they stand.  Every pointer stays valid until the segment is finished. */
typedef struct {
    uint32_t po2;            /* N = 2^po2 rows                                                                          */
    uint32_t zk_rows;        /* the last zk_rows rows of DATA and ACCUM are blinding rows (upstream ZK_CYCLES)           */
    uint32_t w_code, w_data, w_accum, n_mix;
    int device;              /* CUDA ordinal of the context                                                            */
    void* stream;            /* the context's cudaStream_t (NULL in the host emulator)                                  */
    const uint32_t* code;    /* device u32[w_code][N]: committed control columns                                        */
    const uint32_t* data;    /* device u32[w_data][N]: committed witness columns                                        */
    const uint32_t* globals; /* device [32]                                                                             */
    const uint32_t* mix;     /* device [n_mix]: the accum mix drawn after the DATA commit                               */
    uint32_t* accum;         /* device u32[w_accum][N]: the caller writes these                                         */
    const uint32_t* mix_host;     /* host copies, owned by the context                                                  */
    const uint32_t* globals_host;
    uint64_t blind_seed;
} hfb200_segment_dev;
/* flags of hfb200_segment_begin_dev: `code` / `data` are device pointers on the context's device, copied device to device on
 * the context's stream (the copy follows the stream's earlier work; anything writing them on other streams must be complete).
 * A pointer that is not device memory of that device is refused before anything is queued. */
enum { HFB200_DEV_INPUTS = 1 };
/* `code == NULL` reuses the resident control group as in hfb200_segment_begin; `data` may be NULL after hfb200_witgen_synth or
 * hfb200_segment_witness_dev (below). */
const char* hfb200_segment_begin_dev(hfb200_ctx* ctx, uint32_t po2, const uint32_t* globals, const uint32_t* code, const uint32_t* data,
                                     uint64_t blind_seed, uint32_t flags, hfb200_segment_dev* out);
/* Completes the segment begun by either begin, from the accum columns as they stand in device memory (no upload, no built-in
 * step_accum).  The caller's accum work must be enqueued on `stream`, or complete on the caller's own streams, before the
 * call.  hfb200_last_stats then reports as ms_accum the device time on the stream from the end of the DATA commit to this
 * call: the caller's kernels AND any idle time of the stream in between. */
const char* hfb200_segment_finish_dev(hfb200_ctx* ctx, uint32_t* seal_out, size_t seal_cap, size_t* seal_words);
/* Device form of risc0-zkp `Hal::prefix_products` (and of the running sums of LogUp-style arguments): an in-place inclusive scan
 * of the Fp4 chains stored in accum columns 4c..4c+3, c in [first_chain, first_chain + n_chains), over rows [0, rows), on the
 * context's stream.  Valid between a begin and its finish. */
enum { HFB200_SCAN_PRODUCT = 0, HFB200_SCAN_SUM = 1 };
const char* hfb200_segment_accum_scan(hfb200_ctx* ctx, int kind, uint32_t first_chain, uint32_t n_chains, size_t rows);
/* Writes the zk_rows blinding rows of every accum column from the segment's blinding key (the rows the built-in step_accum
 * writes; the key itself never leaves the library).  On the context's stream; valid between a begin and its finish. */
const char* hfb200_segment_accum_blind(hfb200_ctx* ctx);
/* Number of CUDA devices.  No device or no driver is a count of 0 (NULL returned), not an error. */
const char* hfb200_device_count(int* out);

/* The witness on DEVICE memory (upstream's GPU prover generates it there: witgen kernels expand the preflight trace into the
 * data columns).  witness_dev lays the context out for po2 (12 <= po2 <= max_po2; the same po2 again keeps a resident control
 * group) and derives the segment's blinding key, once: hfb200_segment_data_blind and the later accum blinding (built-in
 * step_accum or hfb200_segment_accum_blind) both use it.  It then describes the writable DATA columns.  The caller's kernels
 * write them on `stream`; the next hfb200_segment_begin / _begin_dev with data == NULL commits them exactly as they stand (no
 * copy, no upload) and must pass the same po2 and blind_seed.  `code` keeps its rules: host columns (device columns with
 * HFB200_DEV_INPUTS) are copied in, NULL reuses the resident control group of that po2.  An error return of any entry
 * abandons the open witness. */
typedef struct {
    uint32_t po2;            /* N = 2^po2 rows                                                            */
    uint32_t zk_rows;        /* the last zk_rows rows of every DATA column are blinding rows               */
    uint32_t w_code, w_data;
    int device;              /* CUDA ordinal of the context                                               */
    void* stream;            /* the context's cudaStream_t (NULL in the host emulator)                     */
    uint32_t* data;          /* device u32[w_data][N]: the context's resident data columns                 */
} hfb200_witness_dev;
const char* hfb200_segment_witness_dev(hfb200_ctx* ctx, uint32_t po2, uint64_t blind_seed, hfb200_witness_dev* out);
/* Writes rows [N - zk_rows, N) of every DATA column from the segment's key (the rows hfb200_witgen_synth writes there), on
 * the context's stream.  Valid between hfb200_segment_witness_dev and the begin that follows. */
const char* hfb200_segment_data_blind(hfb200_ctx* ctx);
/* Device memory owned by the context, at least `bytes` long, for the caller's compact witness input (e.g. a preflight trace),
 * which the caller copies in itself with cudaMemcpyAsync on the witness's `stream`.  Valid until the segment is finished or
 * abandoned; it grows only when a larger request comes (a grow first waits for the context's stream) and is freed by
 * hfb200_destroy.  Valid to call while a witness is open. */
const char* hfb200_segment_scratch(hfb200_ctx* ctx, size_t bytes, void** out);

/* Witness stand-in on the device (replaces preflight + WitnessGenerator for the synthetic circuit):
 * fills the context's resident code/data columns; globals_out receives the 32 global words. */
const char* hfb200_witgen_synth(hfb200_ctx* ctx, uint32_t po2, uint64_t trace_seed, uint64_t blind_seed, uint32_t* globals_out);
/* Proves the resident trace (inputs already in HBM: the `value` leg of bench.py). The trace stays intact. */
const char* hfb200_prove_resident(hfb200_ctx* ctx, uint64_t blind_seed, uint32_t* seal_out, size_t seal_cap, size_t* seal_words);
/* Copies resident columns back (group: 0 accum, 1 code, 2 data), for parity tests of witgen/step_accum. */
const char* hfb200_read_group(hfb200_ctx* ctx, uint32_t group, uint32_t* out, size_t cap_words);

/* Seal length in words for (circuit, po2) -- what upstream's Vec<u32> seal would hold.  Defined for 12 <= po2 <= 22, the sizes
 * hfb200_init accepts as max_po2, whatever this context's own max_po2; returns 0 for any other po2 and for ctx == NULL. */
size_t hfb200_seal_words(const hfb200_ctx* ctx, uint32_t po2);

/* ---- transcript checkpoints of the last proved segment (parity tests) ------------------------ */
/* names: globals_hash code_root data_root accum_mix accum_root poly_mix check_root z hash_u deep_mix
 *        final_poly_hash fri_root_<r> fri_mix_<r> fri_final_hash query_positions */
const char* hfb200_checkpoint(hfb200_ctx* ctx, const char* name, uint32_t* out, size_t cap, size_t* n_words);

/* ---- verification ---------------------------------------------------------------------------- */
/* `Receipt::verify` for one segment seal (the reference's uses: /root/reference/host/src/main.rs:622-624,
 * /root/reference/verifier/src/main.rs:124-126).  Mirrors risc0-zkp `verify::Verifier::verify` + the circuit's
 * constraint polynomial at the DEEP point; runs on the host like upstream's verifier and needs no device or context.
 * Exactly one of `circuit` (built-in stand-in circuit) / `ir` (data-defined circuit) is non-NULL.  `code_root` = the 8-word
 * control id of (circuit, po2), e.g. hfb200_control_root or the "code_root" checkpoint of a trusted proof.
 * Returns NULL when the seal is valid, else the reason. */
const char* hfb200_verify_segment(const hfb200_circuit_desc* circuit, const hfb200_circuit_ir* ir, const uint32_t* seal, size_t seal_words,
                                  const uint32_t* code_root /*[8]*/, uint32_t* po2_out);
/* The same over the n segment seals of a composite receipt, fanned out over up to `threads` host threads (0 = one per hardware
 * thread; the seals are independent).  `code_roots` = n x 8 words (the control id of each seal's po2), `po2_out` (optional) = n
 * words.  Returns NULL when every seal is valid; otherwise the reason of the FIRST failing seal (lowest index), prefixed
 * "segment <i>: ", and `*first_bad` (optional) = i (n when all verify). */
const char* hfb200_verify_segments(const hfb200_circuit_desc* circuit, const hfb200_circuit_ir* ir, const uint32_t* const* seals,
                                   const size_t* seal_words, size_t n, const uint32_t* code_roots /*[n][8]*/, uint32_t* po2_out /*[n] or NULL*/,
                                   unsigned threads, size_t* first_bad);
/* hfb200_verify_segment / hfb200_verify_segments for seals of hash suite `suite` (HFB200_HASH_*); `code_root(s)` must be control
 * ids of that suite.  The two entries above are these with HFB200_HASH_POSEIDON2. */
const char* hfb200_verify_segment_suite(const hfb200_circuit_desc* circuit, const hfb200_circuit_ir* ir, const uint32_t* seal, size_t seal_words,
                                        const uint32_t* code_root /*[8]*/, uint32_t* po2_out, int suite);
const char* hfb200_verify_segments_suite(const hfb200_circuit_desc* circuit, const hfb200_circuit_ir* ir, const uint32_t* const* seals,
                                         const size_t* seal_words, size_t n, const uint32_t* code_roots /*[n][8]*/, uint32_t* po2_out /*[n] or NULL*/,
                                         unsigned threads, size_t* first_bad, int suite);
/* ---- receipt claims: the rest of `receipt.verify(image_id)` (host only; no device, no context) -------------------------
 * Upstream's Receipt::verify also decodes each segment's ReceiptClaim from the seal's globals, chains pre/post state digests
 * from the image id and ties the journal digest to the last claim's output (/root/reference/verifier/src/main.rs:124-126 trusts
 * the journal after this call).  Globals layout used here (the rv32im-v2 layout is not obtainable; this is the stand-in's):
 *   word 1 = exit code (0 Halted / 1 SystemSplit), words 8..15 = pre-state, 16..23 = post-state, 24..31 = output (journal)
 *   digest, zero unless last.  Digests are Poseidon2 digests: 8 field elements in Montgomery form.
 * The globals are part of every seal and are absorbed first into the Fiat-Shamir transcript, so a seal that verifies carries
 * exactly the claim its prover was given. */
typedef struct { uint32_t pre[8], post[8], output[8]; uint32_t exit_code; } hfb200_claim;
enum { HFB200_EXIT_HALTED = 0, HFB200_EXIT_SYSTEM_SPLIT = 1 };
/* Poseidon2 digest of a byte string (length, then 3 bytes per field element): the journal digest. */
const char* hfb200_digest_bytes(const uint8_t* bytes, size_t n, uint32_t* out8);
/* Poseidon2 hash_pair of two digests. */
const char* hfb200_digest_pair(const uint32_t* a8, const uint32_t* b8, uint32_t* out8);
/* Writes / reads the claim words of a 32-word globals array (a seal starts with its globals). */
const char* hfb200_claim_encode(const hfb200_claim* claim, uint32_t* globals /*[32]*/);
const char* hfb200_claim_decode(const uint32_t* seal, size_t seal_words, hfb200_claim* out);
/* Executor stand-in: the post-state that follows `pre` after segment `index` of size po2 (upstream: digest of the memory image). */
const char* hfb200_claim_next_state(const uint32_t* pre8, uint32_t index, uint32_t po2, uint32_t* post8);
/* The claim part of Receipt::verify over n seals in segment order (each already accepted by hfb200_verify_segment): segment 0
 * starts from image_id, every segment continues from its predecessor's post-state, only the last one halts, and its output equals
 * hfb200_digest_bytes(journal).  Returns NULL or the reason. */
const char* hfb200_verify_claims(const uint32_t* const* seals, const size_t* seal_words, size_t n, const uint32_t* image_id8,
                                 const uint8_t* journal, size_t journal_len);

/* ---- the hash suites' host primitives (host only; no device, no context) ------------------------------------------------
 * The pieces of the transcript and of the verifier of each suite (HFB200_HASH_*), for known-answer tests and for hosts that
 * recompute a digest.  hfb200_sha256: the standard, padded SHA-256 of a byte string as digest words (little-endian bytes =
 * the standard output).  hfb200_hash_elems: the suite's hash of n words (hash_elem_slice: Merkle leaves, the transcript
 * header, hash_u).  hfb200_hash_pair: the suite's hash of two digests (Merkle nodes).  hfb200_rng_script: runs the suite's
 * transcript RNG (Poseidon2Rng or ShaRng) from its initial state through n_ops ops, ops[2i] = 0: mix(the next 8 words of
 * `digests`), 1: random_elem (Montgomery form), 2: random_bits(ops[2i + 1] in 1..31); every draw is appended to out
 * (cap words), *n_out = draws written. */
const char* hfb200_sha256(const uint8_t* bytes, size_t n, uint32_t* out8);
const char* hfb200_hash_elems(int suite, const uint32_t* elems, size_t n, uint32_t* out8);
const char* hfb200_hash_pair(int suite, const uint32_t* a8, const uint32_t* b8, uint32_t* out8);
const char* hfb200_rng_script(int suite, const uint32_t* ops, size_t n_ops, const uint32_t* digests, size_t n_digests, uint32_t* out, size_t cap,
                              size_t* n_out);

/* Control id: Merkle root of the x4 LDE of the code (control) columns, u32[w_code][2^po2] on the host, in the context's hash suite.
 * The committed control group stays resident: until the context sees another po2 or another `code` pointer, segments may
 * pass code == NULL to hfb200_prove_segment / hfb200_segment_begin and reuse it (the control columns depend on
 * (circuit, po2) only; the seal is bit-identical to the one produced with the columns passed again). */
const char* hfb200_control_root(hfb200_ctx* ctx, uint32_t po2, const uint32_t* code, uint32_t* root_out /*[8]*/);

/* ---- measurement ------------------------------------------------------------------------------ */
typedef struct {
    float ms_total;        /* whole segment, host wall clock from entry to seal bytes on host                 */
    float ms_device;       /* CUDA-event time, first enqueue to last kernel, on the context's stream          */
    float ms_h2d;          /* host->device trace copies (0 for resident)                                  */
    float ms_ntt_main;     /* iNTT+zk_shift and expand+NTT (LDE) of code+data+accum columns               */
    float ms_hash_main;    /* Poseidon2 leaf hashing + tree folds of code+data+accum                      */
    float ms_accum;        /* step_accum (after hfb200_segment_finish_dev: stream time from the DATA commit to the call,  */
                           /* the caller's accum kernels and any idle time together)                                      */
    float ms_check;        /* eval_check + check-group commit                                             */
    float ms_deep;         /* DEEP evaluations + quotient                                                 */
    float ms_fri;          /* FRI rounds + query openings                                                 */
    uint64_t launches;     /* kernels launched for the segment                                            */
    uint64_t ntt_main_bytes; /* algorithmic bytes of ms_ntt_main: 28 * w * N (8 iNTT + 20 LDE)            */
    uint64_t host_syncs;   /* stream synchronisations of the segment (each one a transcript dependency: a root, the tap  */
                           /* evaluations, the final FRI coefficients, the openings)                                       */
} hfb200_stats;
/* Tracing (SURVEY.md section 5): every stage is an NVTX range on the enqueuing host thread ("hfb200:commit_code", "...:commit_data",
 * "...:commit_accum", "...:check", "...:deep", "...:fri"), visible in nsys; with HFB200_METRICS=<file|stderr> in the environment every
 * proved segment appends one JSON line {po2, columns, device, stage ms, launches, host_syncs, ntt_main_bytes, ntt_main_gbs[, hbm_peak_gbs,
 * ntt_main_frac when HFB200_HBM_PEAK_GBS is set]}. */
const char* hfb200_last_stats(hfb200_ctx* ctx, hfb200_stats* out);
uint64_t hfb200_total_launches(const hfb200_ctx* ctx);

/* ---- multi-GPU: a pool of contexts fed from one queue of independent segments --------------------------------- */
/* Replaces the segment loop of upstream's `ProverImpl::prove_session` (sequential there).  One worker thread per
 * (device, slot); whole segments are handed out longest-first (by po2); no collective, only seals return.  Seals depend
 * on (trace, blind_seed) only, so the result is identical for any number of devices.  A pool proves data-defined circuits
 * once it has an accum callback (hfb200_pool_set_accum); without one their jobs are refused (step_accum is the caller's). */
typedef struct hfb200_pool hfb200_pool;
typedef struct {
    uint32_t po2;
    const uint32_t* globals; /* [32] */
    const uint32_t* code;    /* u32[w_code][N]  host */
    const uint32_t* data;    /* u32[w_data][N]  host; NULL = from the pool's witgen callback (hfb200_pool_set_witgen) */
    uint64_t blind_seed;
    uint32_t* seal_out;      /* caller buffer, seal_cap words */
    size_t seal_cap;
    size_t seal_words;       /* out */
    const char* error;       /* out: NULL or malloc'd message (hfb200_free_error) */
    int device;              /* out: device that proved the job */
    float ms;                /* out: host wall time of the job (last attempt) */
    int attempts;            /* out: times the job was started (> 1: re-queued after a CUDA error on another context) */
} hfb200_segment_job;
const char* hfb200_pool_create(const int* devices, int n_devices, int contexts_per_device, uint32_t max_po2,
                               const hfb200_circuit_desc* circuit, hfb200_pool** out);
/* Same for a circuit given as data (every worker context is an hfb200_init_ir context; the tables are copied). */
const char* hfb200_pool_create_ir(const int* devices, int n_devices, int contexts_per_device, uint32_t max_po2,
                                  const hfb200_circuit_ir* circuit, hfb200_pool** out);
/* Blinding mode of every worker context (see hfb200_set_blinding; default HFB200_BLIND_OS_ENTROPY). */
const char* hfb200_pool_set_blinding(hfb200_pool* pool, int mode);
/* Hash suite of every worker context (see hfb200_set_hash_suite; default HFB200_HASH_POSEIDON2).  Kept by the pool: a context
 * re-created after a device fault gets it again.  Not while hfb200_pool_prove runs. */
const char* hfb200_pool_set_hash_suite(hfb200_pool* pool, int suite);
/* Proves all jobs; returns NULL when every job succeeded, else the first failed job's error (every failed job keeps its own
 * message in jobs[i].error).  Failure handling (the reference's batch behaviour, /root/reference/data/watchdog.sh:58-83: a
 * failed input is set aside and the rest continue): a shape / argument error fails that job only; a CUDA error makes the
 * worker destroy and re-create its context (the context is retired if that fails) and puts the job back on the queue for any
 * healthy context, at most 3 attempts; jobs left when no healthy context remains fail with that reason.  The number of
 * contexts in flight per device follows the queue depth (min(contexts_per_device, ceil(jobs per device / 2))). */
const char* hfb200_pool_prove(hfb200_pool* pool, hfb200_segment_job* jobs, size_t n_jobs);
typedef struct {
    size_t contexts;            /* worker contexts created */
    size_t contexts_retired;    /* contexts that could not be re-created after a CUDA error */
    uint64_t faults;            /* CUDA errors seen by workers since pool creation */
    uint64_t retries;           /* jobs put back on the queue */
    uint64_t contexts_recreated;
} hfb200_pool_stats_t;
const char* hfb200_pool_stats(const hfb200_pool* pool, hfb200_pool_stats_t* out);
/* Test hook: worker `worker` lets `after_jobs` more jobs pass, then reports a failure INSTEAD of proving its next job.
 * kind 0 = a device fault ("CUDA error ..."): exercises context re-creation + re-queue; kind 1 = a non-device failure: the
 * job fails, nothing is retried.  Nothing is injected unless this is called. */
const char* hfb200_pool_inject_fault(hfb200_pool* pool, size_t worker, uint64_t after_jobs, int kind);
/* Shared control group for the jobs of one po2 (opt-in): `code` = u32[w_code][2^po2], caller-owned, must stay valid while the pool
 * may use it (NULL forgets it).  Jobs of that po2 may then carry code == NULL: every worker context commits the control group once
 * per load (each call starts a new generation, so a reload -- same pointer or not -- is re-committed by every worker before its
 * next code == NULL job) and reuses it; seals are identical to the ones produced with the columns passed per job. */
const char* hfb200_pool_load_control(hfb200_pool* pool, uint32_t po2, const uint32_t* code);
/* The caller's step_accum for every job of the pool (both kinds of pool; on a built-in pool it replaces the built-in one).  Each
 * job then runs hfb200_segment_begin_dev (host inputs, as jobs carry them), fn on the worker thread (the context's device is
 * current; `job` = index into the jobs array), hfb200_segment_finish_dev.  Callbacks run concurrently, one per worker, and may
 * call only hfb200_segment_accum_scan / _accum_blind on the `ctx` they are given (plus their own kernels on seg->stream).  A
 * nonzero return fails that job only ("accum callback returned <rc>"), is not retried, and leaves the context usable; a CUDA
 * error takes the device-fault path above.  fn = NULL removes the callback. */
typedef int (*hfb200_accum_fn)(void* user, hfb200_ctx* ctx, const hfb200_segment_dev* seg, size_t job);
const char* hfb200_pool_set_accum(hfb200_pool* pool, hfb200_accum_fn fn, void* user);
/* The caller's witness generator for every job with data == NULL (without one such jobs are refused).  Each of them runs
 * hfb200_segment_witness_dev, fn on the worker thread (the context's device is current), begin with data == NULL (job.code as
 * usual, NULL = the pool's shared control group), the accum stage (the accum callback if set, else the built-in step_accum; a
 * pool over a data-defined circuit without an accum callback refuses the job) and finish.  Jobs with data keep their path.
 * Callbacks run concurrently, one per worker, and may call only hfb200_segment_scratch / _data_blind on the `ctx` they are given
 * (plus their own kernels and cudaMemcpyAsync on w->stream).  A nonzero return fails that job only ("witgen callback returned
 * <rc>"), is not retried, and leaves the context usable; a CUDA error takes the device-fault path, so the callback runs again
 * on a NEW context: it must rebuild its device state (the scratch contents included) from host input.  fn = NULL removes it. */
typedef int (*hfb200_witgen_fn)(void* user, hfb200_ctx* ctx, const hfb200_witness_dev* w, size_t job);
const char* hfb200_pool_set_witgen(hfb200_pool* pool, hfb200_witgen_fn fn, void* user);
void hfb200_pool_destroy(hfb200_pool* pool);

/* ---- HAL-level operators (second seam: risc0-zkp `Hal` methods), host buffers in/out ----------- */
/* Hal::batch_interpolate_ntt (+ Hal::zk_shift when zk_shift != 0): natural-order evaluations ->
 * bit-reversed coefficients, in place, `count` columns of n = 2^k. */
const char* hfb200_op_interpolate_ntt(hfb200_ctx* ctx, uint32_t* io, size_t count, size_t n, int zk_shift);
/* Hal::batch_expand_into_evaluate_ntt(out, in, count, expand_bits): bit-reversed coefficients ->
 * natural-order evaluations on the 2^expand_bits larger domain (expand_bits in {0, 2}). */
const char* hfb200_op_expand_ntt(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, size_t n_in, uint32_t expand_bits);
/* The fused production path of commit_group: trace columns -> LDE evaluations (no coefficient round trip). */
const char* hfb200_op_lde(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, size_t n_in);
/* Hal::hash_rows + Hal::hash_fold: full Merkle tree (heap layout, 2*rows digests) of a column-major matrix, in the context's hash suite. */
const char* hfb200_op_merkle(hfb200_ctx* ctx, const uint32_t* matrix, size_t rows, size_t cols, uint32_t* nodes_out);
/* poseidon2_mix on `n` independent 24-word states. */
const char* hfb200_op_poseidon2(hfb200_ctx* ctx, uint32_t* states, size_t n);
/* Hal::fri_fold: 4 x n bit-reversed coefficient columns -> 4 x n/16. mix = one Fp4. */
const char* hfb200_op_fri_fold(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t n, const uint32_t* mix4);
/* Device-only timing of the main-group NTT/LDE pipeline on resident synthetic columns (roofline probe):
 * runs the fused trace->LDE pipeline over `count` columns of 2^po2 `iters` times, returns avg ms. */
const char* hfb200_bench_lde(hfb200_ctx* ctx, uint32_t po2, uint32_t count, uint32_t iters, float* ms_avg);
const char* hfb200_bench_merkle(hfb200_ctx* ctx, uint32_t po2, uint32_t count, uint32_t iters, float* ms_avg);
/* Integer-multiply roofline probe (the bound of Poseidon2 and of the NTT butterflies on sm_100a): sustained rate of a
 * modular-multiply sequence over every SM, 8 independent chains per thread.  kind 0 = Montgomery product, 1 = Shoup
 * constant product, 2 = the x^7 S-box chain (4 products per step).  Returns products per second. */
const char* hfb200_bench_modmul(hfb200_ctx* ctx, int kind, uint32_t iters, double* products_per_s);
/* Device-timeline marks for whole-job timing across several contexts of one device: hfb200_mark records CUDA event
 * `slot` (0..3) on the context's stream; hfb200_mark_elapsed returns the device time from mark (a, slot_a) to mark
 * (b, slot_b) after both have completed (a and b may be the same or different contexts of the same device). */
const char* hfb200_mark(hfb200_ctx* ctx, int slot);
const char* hfb200_mark_elapsed(hfb200_ctx* a, int slot_a, hfb200_ctx* b, int slot_b, float* ms);

/* ---- device HAL: risc0-zkp `Hal` operators on caller DEVICE buffers ------------------------------------------------
 * The second seam (upstream's `Prover`, `MerkleTreeProver` and `fri_prove` are written against `risc0_zkp::hal::Hal`): the
 * operators a `Hal` implementation needs, on device memory the caller owns (INTEGRATION.md sketches `impl Hal for B200Hal`).
 *   - any context works (one made with max_po2 = 12 is cheap); sizes are bounded by the kernels, not by max_po2;
 *   - every buffer pointer must be device memory of the context's device: sizes are checked first, then pointers, and a
 *     refused call queues nothing;
 *   - work is enqueued on the context's stream (hfb200_hal_stream) and the call returns without synchronising; results are
 *     visible to later work on that stream, and to the host after hfb200_hal_sync;
 *   - operators that need scratch (batch_evaluate_any, mix_poly_coeffs, poly_divide, prefix_products) use a buffer owned by
 *     the context that grows when a larger request comes (a grow first waits for the stream) and is freed by hfb200_destroy.
 * Layouts: base-field matrices column-major u32[count][n] (Montgomery form); Fp4 buffers hold 4 consecutive words per element
 * (upstream's Buffer<ExtElem>), c0 + c1 x + c2 x^2 + c3 x^3 with x^4 = -11. */
/* The context's cudaStream_t (NULL in the host emulator) and device ordinal (device may be NULL). */
const char* hfb200_hal_stream(hfb200_ctx* ctx, void** stream, int* device);
/* Waits for everything queued on the context's stream. */
const char* hfb200_hal_sync(hfb200_ctx* ctx);
/* Stream synchronisations the context has made since it was created: the segment prover's transcript waits, hfb200_hal_sync
 * and the waits of a scratch grow.  A sequence of HAL calls that needs no larger scratch leaves it unchanged. */
uint64_t hfb200_hal_host_syncs(const hfb200_ctx* ctx);
/* Hal::batch_interpolate_ntt: per column, natural-order evaluations on the 2^k-th roots of unity -> coefficients in
 * bit-reversed order (scaled by 1/n), in place.  n = 2^k, 2 <= n <= 2^24. */
const char* hfb200_hal_batch_interpolate_ntt(hfb200_ctx* ctx, uint32_t* io, size_t count, size_t n);
/* Hal::zk_shift: the coefficient at bit-reversed position i (true index j = bitrev(i)) times 3^j, so f(x) -> f(3x).
 * n = 2^k <= 2^24. */
const char* hfb200_hal_zk_shift(hfb200_ctx* ctx, uint32_t* io, size_t count, size_t n);
/* Hal::batch_expand_into_evaluate_ntt: bit-reversed coefficients u32[count][n_in] -> natural-order evaluations
 * u32[count][n_in << expand_bits] on the 2^expand_bits times larger domain.  expand_bits in {0, 2}; 2 <= n_in,
 * n_in << expand_bits <= 2^24; out and in must not overlap. */
const char* hfb200_hal_batch_expand_into_evaluate_ntt(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, size_t n_in, uint32_t expand_bits);
/* Hal::batch_bit_reverse: io[c][i] <-> io[c][bitrev(i)] per column, in place.  n = 2^k <= 2^31. */
const char* hfb200_hal_batch_bit_reverse(hfb200_ctx* ctx, uint32_t* io, size_t count, size_t n);
/* Hal::hash_rows: digests[r] (8 words) = Poseidon2 sponge over row r of the column-major matrix u32[cols][rows], 16 elements
 * per absorption, zero padded (the leaves of hfb200_op_merkle and of the segment prover's trees).  Any rows >= 1; digests
 * 16-byte aligned. */
const char* hfb200_hal_hash_rows(hfb200_ctx* ctx, uint32_t* digests, const uint32_t* matrix, size_t rows, size_t cols);
/* Hal::hash_fold: io[output_size + i] = hash_pair(io[input_size + 2i], io[input_size + 2i + 1]) for i < output_size, digests
 * of 8 words, input_size = 2 * output_size: one level of the heap layout of hfb200_op_merkle (node 1 = root).  16-byte aligned. */
const char* hfb200_hal_hash_fold(hfb200_ctx* ctx, uint32_t* io, size_t input_size, size_t output_size);
/* hfb200_hal_hash_rows / _hash_fold of the SHA-256 suite (upstream's Hal with HashSuite = Sha256HashSuite), whatever the
 * context's own suite; same shapes, checks and stream rules.  sha_rows: digests[r] = SHA-256 compressions from the IV over row
 * r's words as little-endian bytes, 16 words per block, the last block zero-filled, no length block; sha_fold: hash_pair =
 * one compression of the 64 bytes of the two child digests.  Digest words are the byte-swapped state words. */
const char* hfb200_hal_sha_rows(hfb200_ctx* ctx, uint32_t* digests, const uint32_t* matrix, size_t rows, size_t cols);
const char* hfb200_hal_sha_fold(hfb200_ctx* ctx, uint32_t* io, size_t input_size, size_t output_size);
/* Hal::batch_evaluate_any: out[j] = sum_{k < n} coeffs[which[j]][k] * xs[j]^k for j < count, coeffs u32[poly_count][n]
 * (natural order), which u32[count] (each < poly_count), xs and out Fp4[count].  count <= 262140. */
const char* hfb200_hal_batch_evaluate_any(hfb200_ctx* ctx, const uint32_t* coeffs, size_t poly_count, size_t n, const uint32_t* which,
                                          const uint32_t* xs, uint32_t* out, size_t count);
/* Hal::mix_poly_coeffs (the DEEP combos): out[combo_of_col[c]][i] += mix_start * mix^c * in[c][i] for c < n_cols, i < n;
 * in u32[n_cols][n], combo_of_col u32[n_cols] (each < n_combos), out Fp4[n_combos][n].  mix_start and mix are HOST Fp4 values
 * (4 words each, read during the call).  n_cols <= 8192. */
const char* hfb200_hal_mix_poly_coeffs(hfb200_ctx* ctx, uint32_t* out, const uint32_t* mix_start, const uint32_t* mix, const uint32_t* in,
                                       const uint32_t* combo_of_col, size_t n_cols, size_t n, size_t n_combos);
/* risc0-zkp poly_divide: synthetic division of the Fp4 polynomial poly[0..n) (natural order) by (x - z), in place:
 * afterwards poly[k] = r_{k+1} with r_k = poly[k] + z r_{k+1}, r_n = 0 (poly[0..n-1) is the quotient, poly[n-1] = 0), and
 * remainder_out (device, one Fp4) = r_0 = p(z).  z is a HOST Fp4 value.  Runs as a parallel scan over the affine maps
 * r -> c + z r.  1 <= n <= 2^30. */
const char* hfb200_hal_poly_divide(hfb200_ctx* ctx, uint32_t* poly, size_t n, const uint32_t* z, uint32_t* remainder_out);
/* Hal::eltwise_add_elem: out[i] = x[i] + y[i], i < count. */
const char* hfb200_hal_eltwise_add_elem(hfb200_ctx* ctx, uint32_t* out, const uint32_t* x, const uint32_t* y, size_t count);
/* Hal::eltwise_sum_extelem: s_i = sum_{g < to_add} in[g * count + i] over Fp4 in[to_add * count]; out u32[4][count] holds the
 * four components: out[k * count + i] = s_i.c_k. */
const char* hfb200_hal_eltwise_sum_extelem(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, size_t to_add);
/* Hal::eltwise_copy_elem: out[i] = in[i], i < count (one cudaMemcpyAsync). */
const char* hfb200_hal_eltwise_copy_elem(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count);
/* Hal::eltwise_zeroize_elem: io[i] = 0, i < count. */
const char* hfb200_hal_eltwise_zeroize_elem(hfb200_ctx* ctx, uint32_t* io, size_t count);
/* Hal::gather_sample: dst[i] = src[idx + i * stride], i < size. */
const char* hfb200_hal_gather_sample(hfb200_ctx* ctx, uint32_t* dst, const uint32_t* src, size_t idx, size_t size, size_t stride);
/* Hal::scatter: for every cycle c < count, into[offsets[j]] = values[j] for j in [index[c], index[c + 1]); index u32[count + 1]. */
const char* hfb200_hal_scatter(hfb200_ctx* ctx, uint32_t* into, const uint32_t* index, const uint32_t* offsets, const uint32_t* values, size_t count);
/* Hal::prefix_products: io[i] <- io[0] * io[1] * ... * io[i] over Fp4[n], in place (two-pass block scan). */
const char* hfb200_hal_prefix_products(hfb200_ctx* ctx, uint32_t* io, size_t n);
/* Hal::fri_fold: in = 4 component columns u32[4][n] of Fp4 coefficients in bit-reversed order -> out u32[4][n/16],
 * out[.][idx] = sum_{i < 16} mix^i * in[.][bitrev4(i) * n/16 + idx]; mix = one Fp4 in DEVICE memory.  n a multiple of 16. */
const char* hfb200_hal_fri_fold(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t n, const uint32_t* mix);

#ifdef __cplusplus
}
#endif
#endif /* HFB200_H */
