//! Raw bindings of `include/hfb200.h`.  Error convention is the one of upstream's sys crates
//! (`risc0_sys::ffi_wrap`): NULL = success, otherwise a malloc'd C string released with `hfb200_free_error`.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_uint, c_void};

#[repr(C)]
pub struct hfb200_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct hfb200_pool {
    _private: [u8; 0],
}

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct hfb200_circuit_desc {
    pub w_code: u32,
    pub w_data: u32,
    pub w_accum: u32,
    pub flags: u32,
}

/// Circuit as data: upstream's TapSet and PolyExtStepDef flattened to u32 tables (include/hfb200.h).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct hfb200_tap {
    pub group: u32,
    pub offset: u32,
    pub back: u32,
}
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct hfb200_poly_step {
    pub op: u32,
    pub a: u32,
    pub b: u32,
    pub c: u32,
}
#[repr(C)]
pub struct hfb200_circuit_ir {
    pub w_code: u32,
    pub w_data: u32,
    pub w_accum: u32,
    pub n_mix: u32,
    pub taps: *const hfb200_tap,
    pub n_taps: usize,
    pub steps: *const hfb200_poly_step,
    pub n_steps: usize,
    pub ret: u32,
    /// upstream `CircuitImpl::CIRCUIT_INFO` (16 bytes); all zero selects "RV32IM:v2_______"
    pub info: [u8; 16],
}

#[repr(C)]
pub struct hfb200_segment_job {
    pub po2: u32,
    pub globals: *const u32,
    pub code: *const u32,
    pub data: *const u32,
    pub blind_seed: u64,
    pub seal_out: *mut u32,
    pub seal_cap: usize,
    pub seal_words: usize,
    pub error: *const c_char,
    pub device: c_int,
    pub ms: f32,
    pub attempts: c_int,
}

/// What upstream's `ReceiptClaim` boils down to on this path (include/hfb200.h: receipt claims).
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct hfb200_claim {
    pub pre: [u32; 8],
    pub post: [u32; 8],
    pub output: [u32; 8],
    pub exit_code: u32,
}
pub const HFB200_EXIT_HALTED: u32 = 0;
pub const HFB200_EXIT_SYSTEM_SPLIT: u32 = 1;
pub const HFB200_BLIND_OS_ENTROPY: c_int = 0;
pub const HFB200_BLIND_DETERMINISTIC: c_int = 1;

/// The segment in flight between `hfb200_segment_begin_dev` and `hfb200_segment_finish_dev`: device pointers of the committed
/// columns, the mix and the writable accum columns (valid until the segment is finished), and the context's stream.
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct hfb200_segment_dev {
    pub po2: u32,
    /// the last `zk_rows` rows of DATA and ACCUM are blinding rows
    pub zk_rows: u32,
    pub w_code: u32,
    pub w_data: u32,
    pub w_accum: u32,
    pub n_mix: u32,
    pub device: c_int,
    /// the context's `cudaStream_t` (null in the host emulator)
    pub stream: *mut c_void,
    pub code: *const u32,
    pub data: *const u32,
    pub globals: *const u32,
    pub mix: *const u32,
    pub accum: *mut u32,
    pub mix_host: *const u32,
    pub globals_host: *const u32,
    pub blind_seed: u64,
}
pub const HFB200_DEV_INPUTS: u32 = 1;
pub const HFB200_SCAN_PRODUCT: c_int = 0;
pub const HFB200_SCAN_SUM: c_int = 1;
/// The caller's step_accum for every job of a pool (`hfb200_pool_set_accum`); nonzero fails the job.
pub type hfb200_accum_fn =
    Option<unsafe extern "C" fn(user: *mut c_void, ctx: *mut hfb200_ctx, seg: *const hfb200_segment_dev, job: usize) -> c_int>;

/// The writable DATA columns between `hfb200_segment_witness_dev` and the begin (data = null) that commits them as they stand.
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct hfb200_witness_dev {
    pub po2: u32,
    /// the last `zk_rows` rows of every DATA column are blinding rows (`hfb200_segment_data_blind`)
    pub zk_rows: u32,
    pub w_code: u32,
    pub w_data: u32,
    pub device: c_int,
    /// the context's `cudaStream_t` (null in the host emulator)
    pub stream: *mut c_void,
    /// device u32[w_data][N]: the context's resident data columns
    pub data: *mut u32,
}
/// The caller's witness generator for every pool job with `data` = null (`hfb200_pool_set_witgen`); nonzero fails the job.
pub type hfb200_witgen_fn =
    Option<unsafe extern "C" fn(user: *mut c_void, ctx: *mut hfb200_ctx, w: *const hfb200_witness_dev, job: usize) -> c_int>;

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct hfb200_pool_stats_t {
    pub contexts: usize,
    pub contexts_retired: usize,
    pub faults: u64,
    pub retries: u64,
    pub contexts_recreated: u64,
}

extern "C" {
    pub fn hfb200_init(device: c_int, max_po2: u32, circuit: *const hfb200_circuit_desc, out: *mut *mut hfb200_ctx) -> *const c_char;
    pub fn hfb200_init_ir(device: c_int, max_po2: u32, circuit: *const hfb200_circuit_ir, out: *mut *mut hfb200_ctx) -> *const c_char;
    /// CUDA source of the eval_check kernel `hfb200_init_ir` specialises with NVRTC (no device needed).
    pub fn hfb200_ir_source(circuit: *const hfb200_circuit_ir, out: *mut c_char, cap: usize, need: *mut usize) -> *const c_char;
    /// 1 when the context's eval_check runs the NVRTC-specialised kernel (0: interpreter kernel / built-in circuit).
    pub fn hfb200_ir_jit_active(ctx: *const hfb200_ctx, compile_ms: *mut f32) -> c_int;
    pub fn hfb200_destroy(ctx: *mut hfb200_ctx);
    pub fn hfb200_free_error(msg: *const c_char);
    /// Seal length in words for `po2`; 0 for po2 outside [12, 22].
    pub fn hfb200_seal_words(ctx: *const hfb200_ctx, po2: u32) -> usize;
    pub fn hfb200_prove_segment(
        ctx: *mut hfb200_ctx, po2: u32, globals: *const u32, code: *const u32, data: *const u32, blind_seed: u64,
        seal_out: *mut u32, seal_cap: usize, seal_words: *mut usize,
    ) -> *const c_char;
    pub fn hfb200_segment_begin(
        ctx: *mut hfb200_ctx, po2: u32, globals: *const u32, code: *const u32, data: *const u32, blind_seed: u64,
        mix_out: *mut u32, mix_cap: usize, mix_words: *mut usize,
    ) -> *const c_char;
    pub fn hfb200_segment_finish(ctx: *mut hfb200_ctx, accum_or_null: *const u32, seal_out: *mut u32, seal_cap: usize, seal_words: *mut usize) -> *const c_char;
    /// `hfb200_segment_begin`, then `out` describes the segment in device memory; flags: `HFB200_DEV_INPUTS` (code / data are
    /// device pointers on the context's device).
    pub fn hfb200_segment_begin_dev(
        ctx: *mut hfb200_ctx, po2: u32, globals: *const u32, code: *const u32, data: *const u32, blind_seed: u64, flags: u32,
        out: *mut hfb200_segment_dev,
    ) -> *const c_char;
    /// Commits the accum columns as they stand in device memory and completes the seal.
    pub fn hfb200_segment_finish_dev(ctx: *mut hfb200_ctx, seal_out: *mut u32, seal_cap: usize, seal_words: *mut usize) -> *const c_char;
    /// `Hal::prefix_products` (kind `HFB200_SCAN_PRODUCT`) or running sums (`HFB200_SCAN_SUM`) of the Fp4 chains in accum columns
    /// 4c..4c+3, rows [0, rows), in place on the context's stream.
    pub fn hfb200_segment_accum_scan(ctx: *mut hfb200_ctx, kind: c_int, first_chain: u32, n_chains: u32, rows: usize) -> *const c_char;
    /// The accum group's blinding rows from the segment's blinding key.
    pub fn hfb200_segment_accum_blind(ctx: *mut hfb200_ctx) -> *const c_char;
    /// Number of CUDA devices; 0 (and success) without a device or a driver.
    pub fn hfb200_device_count(out: *mut c_int) -> *const c_char;
    pub fn hfb200_pool_set_accum(pool: *mut hfb200_pool, f: hfb200_accum_fn, user: *mut c_void) -> *const c_char;
    /// Lays the context out for `po2`, derives the segment's blinding key and describes the writable DATA columns.
    pub fn hfb200_segment_witness_dev(ctx: *mut hfb200_ctx, po2: u32, blind_seed: u64, out: *mut hfb200_witness_dev) -> *const c_char;
    /// The DATA group's blinding rows from the segment's blinding key (between witness_dev and the begin).
    pub fn hfb200_segment_data_blind(ctx: *mut hfb200_ctx) -> *const c_char;
    /// Device memory owned by the context for the caller's compact witness input; valid until the segment ends.
    pub fn hfb200_segment_scratch(ctx: *mut hfb200_ctx, bytes: usize, out: *mut *mut c_void) -> *const c_char;
    pub fn hfb200_pool_set_witgen(pool: *mut hfb200_pool, f: hfb200_witgen_fn, user: *mut c_void) -> *const c_char;
    pub fn hfb200_pool_create(
        devices: *const c_int, n_devices: c_int, contexts_per_device: c_int, max_po2: u32, circuit: *const hfb200_circuit_desc,
        out: *mut *mut hfb200_pool,
    ) -> *const c_char;
    pub fn hfb200_pool_create_ir(
        devices: *const c_int, n_devices: c_int, contexts_per_device: c_int, max_po2: u32, circuit: *const hfb200_circuit_ir,
        out: *mut *mut hfb200_pool,
    ) -> *const c_char;
    pub fn hfb200_pool_set_blinding(pool: *mut hfb200_pool, mode: c_int) -> *const c_char;
    pub fn hfb200_pool_stats(pool: *const hfb200_pool, out: *mut hfb200_pool_stats_t) -> *const c_char;
    pub fn hfb200_set_blinding(ctx: *mut hfb200_ctx, mode: c_int) -> *const c_char;
    pub fn hfb200_pool_prove(pool: *mut hfb200_pool, jobs: *mut hfb200_segment_job, n_jobs: usize) -> *const c_char;
    pub fn hfb200_digest_bytes(bytes: *const u8, n: usize, out8: *mut u32) -> *const c_char;
    pub fn hfb200_digest_pair(a8: *const u32, b8: *const u32, out8: *mut u32) -> *const c_char;
    pub fn hfb200_claim_encode(claim: *const hfb200_claim, globals: *mut u32) -> *const c_char;
    pub fn hfb200_claim_decode(seal: *const u32, seal_words: usize, out: *mut hfb200_claim) -> *const c_char;
    pub fn hfb200_claim_next_state(pre8: *const u32, index: u32, po2: u32, post8: *mut u32) -> *const c_char;
    pub fn hfb200_verify_claims(
        seals: *const *const u32, seal_words: *const usize, n: usize, image_id8: *const u32, journal: *const u8, journal_len: usize,
    ) -> *const c_char;
    pub fn hfb200_pool_load_control(pool: *mut hfb200_pool, po2: u32, code: *const u32) -> *const c_char;
    pub fn hfb200_pool_destroy(pool: *mut hfb200_pool);
    /// `Receipt::verify` for one segment seal (host code, no device needed).  Exactly one of `circuit` / `ir` is non-null.
    pub fn hfb200_verify_segment(
        circuit: *const hfb200_circuit_desc, ir: *const hfb200_circuit_ir, seal: *const u32, seal_words: usize,
        code_root: *const u32, po2_out: *mut u32,
    ) -> *const c_char;
    /// The same over the `n` segment seals of a composite receipt on up to `threads` host threads (0 = all); reports the first
    /// failing seal.  `code_roots`: n x 8 words, `po2_out`: n words or null, `first_bad`: optional.
    pub fn hfb200_verify_segments(
        circuit: *const hfb200_circuit_desc, ir: *const hfb200_circuit_ir, seals: *const *const u32, seal_words: *const usize, n: usize,
        code_roots: *const u32, po2_out: *mut u32, threads: c_uint, first_bad: *mut usize,
    ) -> *const c_char;
    /// Where the Fiat-Shamir transcript runs: 0 host (default), 1 device, 2 device replayed as a CUDA graph.  Identical seals.
    pub fn hfb200_set_transcript(ctx: *mut hfb200_ctx, mode: c_int) -> *const c_char;
    pub fn hfb200_graph_launches(ctx: *const hfb200_ctx) -> u64;
    /// Control id of (circuit, po2): Merkle root of the committed control columns, computed on the GPU.
    pub fn hfb200_control_root(ctx: *mut hfb200_ctx, po2: u32, code: *const u32, root_out: *mut u32) -> *const c_char;

    // ---- device HAL: risc0-zkp `Hal` operators on caller device buffers (include/hfb200.h states each one's semantics) ----
    // Every pointer is device memory of the context's device; work goes on the context's stream, nothing synchronises until
    // hfb200_hal_sync.  Fp4 buffers: 4 consecutive u32 per element.
    pub fn hfb200_hal_stream(ctx: *mut hfb200_ctx, stream: *mut *mut c_void, device: *mut c_int) -> *const c_char;
    pub fn hfb200_hal_sync(ctx: *mut hfb200_ctx) -> *const c_char;
    pub fn hfb200_hal_host_syncs(ctx: *const hfb200_ctx) -> u64;
    pub fn hfb200_hal_batch_interpolate_ntt(ctx: *mut hfb200_ctx, io: *mut u32, count: usize, n: usize) -> *const c_char;
    pub fn hfb200_hal_zk_shift(ctx: *mut hfb200_ctx, io: *mut u32, count: usize, n: usize) -> *const c_char;
    pub fn hfb200_hal_batch_expand_into_evaluate_ntt(
        ctx: *mut hfb200_ctx, out: *mut u32, input: *const u32, count: usize, n_in: usize, expand_bits: u32,
    ) -> *const c_char;
    pub fn hfb200_hal_batch_bit_reverse(ctx: *mut hfb200_ctx, io: *mut u32, count: usize, n: usize) -> *const c_char;
    pub fn hfb200_hal_hash_rows(ctx: *mut hfb200_ctx, digests: *mut u32, matrix: *const u32, rows: usize, cols: usize) -> *const c_char;
    pub fn hfb200_hal_hash_fold(ctx: *mut hfb200_ctx, io: *mut u32, input_size: usize, output_size: usize) -> *const c_char;
    pub fn hfb200_hal_batch_evaluate_any(
        ctx: *mut hfb200_ctx, coeffs: *const u32, poly_count: usize, n: usize, which: *const u32, xs: *const u32, out: *mut u32, count: usize,
    ) -> *const c_char;
    /// `mix_start` / `mix`: HOST Fp4 values (4 words each).
    pub fn hfb200_hal_mix_poly_coeffs(
        ctx: *mut hfb200_ctx, out: *mut u32, mix_start: *const u32, mix: *const u32, input: *const u32, combo_of_col: *const u32,
        n_cols: usize, n: usize, n_combos: usize,
    ) -> *const c_char;
    /// `z`: HOST Fp4 value; `remainder_out`: one device Fp4.
    pub fn hfb200_hal_poly_divide(ctx: *mut hfb200_ctx, poly: *mut u32, n: usize, z: *const u32, remainder_out: *mut u32) -> *const c_char;
    pub fn hfb200_hal_eltwise_add_elem(ctx: *mut hfb200_ctx, out: *mut u32, x: *const u32, y: *const u32, count: usize) -> *const c_char;
    pub fn hfb200_hal_eltwise_sum_extelem(ctx: *mut hfb200_ctx, out: *mut u32, input: *const u32, count: usize, to_add: usize) -> *const c_char;
    pub fn hfb200_hal_eltwise_copy_elem(ctx: *mut hfb200_ctx, out: *mut u32, input: *const u32, count: usize) -> *const c_char;
    pub fn hfb200_hal_eltwise_zeroize_elem(ctx: *mut hfb200_ctx, io: *mut u32, count: usize) -> *const c_char;
    pub fn hfb200_hal_gather_sample(ctx: *mut hfb200_ctx, dst: *mut u32, src: *const u32, idx: usize, size: usize, stride: usize) -> *const c_char;
    pub fn hfb200_hal_scatter(
        ctx: *mut hfb200_ctx, into: *mut u32, index: *const u32, offsets: *const u32, values: *const u32, count: usize,
    ) -> *const c_char;
    pub fn hfb200_hal_prefix_products(ctx: *mut hfb200_ctx, io: *mut u32, n: usize) -> *const c_char;
    /// `mix`: one Fp4 in DEVICE memory.
    pub fn hfb200_hal_fri_fold(ctx: *mut hfb200_ctx, out: *mut u32, input: *const u32, n: usize, mix: *const u32) -> *const c_char;
}

/// Same contract as `risc0_sys::ffi_wrap`.
pub fn ffi_wrap<F: FnOnce() -> *const c_char>(f: F) -> anyhow::Result<()> {
    let e = f();
    if e.is_null() {
        return Ok(());
    }
    let msg = unsafe { std::ffi::CStr::from_ptr(e) }.to_string_lossy().into_owned();
    unsafe { hfb200_free_error(e) };
    Err(anyhow::anyhow!(msg))
}
