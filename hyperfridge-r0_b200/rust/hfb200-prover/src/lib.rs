//! `b200_prover()` -- the one-line replacement for `default_prover()` at `/root/reference/host/src/main.rs:420`;
//! `prover.prove(env, HYPERFRIDGE_ELF)` (`:423`) and everything after it (`receipt.journal`, `serde_json::to_string(&receipt)`,
//! `receipt.verify(HYPERFRIDGE_ID)`, `:250-267`, `:622-624`) stay as they are.
//!
//! UNCOMPILED SOURCE: the build image has no Rust toolchain and the risc0 crates are not vendored
//! (`/root/reference/Cargo.lock:3087-3229`).  Everything that touches `hfb200_sys` is exact against `include/hfb200.h`;
//! the upstream items (`ExecutorImpl`, `Segment`, `SegmentProver`, `SegmentReceipt`, `CompositeReceipt`, `TAPSET`, `POLY_EXT_DEF`,
//! `WitnessGenerator`, `step_accum`) are written from recollection of risc0-zkvm 3.0.5 / risc0-circuit-rv32im 4.0.4 and are
//! marked `// [upstream]` where a maintainer must check the exact path or signature.
//!
//! What runs where:
//!   upstream CPU (unchanged)   executor (ELF -> Session -> Segments), preflight + witness generation, `step_accum`,
//!                              `SegmentReceipt` / `CompositeReceipt` / `Receipt` constructors, `Receipt::verify`
//!   libhfb200 (B200)           `SegmentProver::prove`: commits, eval_check, DEEP-ALI, FRI, openings, transcript -> seal words
//!
//! The seals verify against `risc0_zkvm` once libhfb200 carries the verified Poseidon2 `M_INT_DIAG` row (DESIGN.md section 1);
//! the rv32im-v2 circuit itself needs no library change: it is registered below as DATA (`hfb200_init_ir` / `hfb200_pool_create_ir`)
//! from upstream's own `TAPSET` and `POLY_EXT_DEF` tables.
use anyhow::{anyhow, bail, Result};
use hfb200_sys as sys;
use std::rc::Rc;

// [upstream] risc0-zkvm 3.0.5 public API (host/src/main.rs uses exactly these: default_prover, ExecutorEnv, Receipt)
use risc0_zkvm::{
    CompositeReceipt, ExecutorEnv, ExecutorImpl, InnerReceipt, ProveInfo, Prover, ProverOpts, Receipt, Segment, SegmentReceipt, Session,
    SessionStats, VerifierContext,
};
// [upstream] risc0-circuit-rv32im 4.0.4: the segment seam and the circuit tables
use risc0_circuit_rv32im::{
    prove::{witgen::WitnessGenerator, Seal, SegmentProver},
    zirgen::{poly_ext::DEF as POLY_EXT_DEF, taps::TAPSET, CircuitImpl},
    REGCOUNT_ACCUM, REGCOUNT_CODE, REGCOUNT_DATA, REGCOUNT_GLOBAL, REGCOUNT_MIX,
};
use risc0_zkp::adapter::{PolyExtStep, PolyExtStepDef};
use risc0_zkp::taps::TapSet;

/// upstream's `TapSet` -> `hfb200_tap[]`: (group, offset, back) in `TapSet::taps()` order; group ids are the library's
/// (0 accum, 1 code, 2 data), the same numbering risc0-zkp uses for `REGISTER_GROUP_{ACCUM, CODE, DATA}`.
fn flatten_taps(taps: &TapSet<'static>) -> Vec<sys::hfb200_tap> {
    taps.taps().map(|t| sys::hfb200_tap { group: t.group() as u32, offset: t.offset() as u32, back: t.back() as u32 }).collect()
}

/// upstream's `PolyExtStepDef` -> `hfb200_poly_step[]`, one entry per step, same two SSA index spaces (fp vars / mix vars).
fn flatten_poly(def: &PolyExtStepDef) -> (Vec<sys::hfb200_poly_step>, u32) {
    let op = |op: u32, a: usize, b: usize, c: usize| sys::hfb200_poly_step { op, a: a as u32, b: b as u32, c: c as u32 };
    let steps = def
        .block
        .iter()
        .map(|s| match *s {
            PolyExtStep::Const(v) => op(0, v as usize, 0, 0),             // canonical value
            PolyExtStep::ConstExt(..) => unreachable!("rv32im-v2 constraints use base-field constants only"), // [upstream] check
            PolyExtStep::Get(tap) => op(1, tap, 0, 0),
            PolyExtStep::GetGlobal(base, offset) => op(2, base, offset, 0), // 0 = globals, 1 = mix
            PolyExtStep::Add(a, b) => op(3, a, b, 0),
            PolyExtStep::Sub(a, b) => op(4, a, b, 0),
            PolyExtStep::Mul(a, b) => op(5, a, b, 0),
            PolyExtStep::True => op(6, 0, 0, 0),
            PolyExtStep::AndEqz(x, val) => op(7, x, val, 0),
            PolyExtStep::AndCond(x, cond, inner) => op(8, x, cond, inner),
        })
        .collect();
    (steps, def.ret as u32)
}

/// The circuit as the library wants it; owns the flattened tables for the lifetime of the pool.
struct CircuitTables {
    taps: Vec<sys::hfb200_tap>,
    steps: Vec<sys::hfb200_poly_step>,
    ret: u32,
}
impl CircuitTables {
    fn rv32im_v2() -> Self {
        let taps = flatten_taps(TAPSET);
        let (steps, ret) = flatten_poly(&POLY_EXT_DEF);
        Self { taps, steps, ret }
    }
    fn ir(&self) -> sys::hfb200_circuit_ir {
        sys::hfb200_circuit_ir {
            w_code: REGCOUNT_CODE as u32,
            w_data: REGCOUNT_DATA as u32,
            w_accum: REGCOUNT_ACCUM as u32,
            n_mix: REGCOUNT_MIX as u32,
            taps: self.taps.as_ptr(),
            n_taps: self.taps.len(),
            steps: self.steps.as_ptr(),
            n_steps: self.steps.len(),
            ret: self.ret,
            info: CircuitImpl::CIRCUIT_INFO.0, // the same 16 bytes upstream's prover and verifier hash into the transcript
        }
    }
}

/// One hfb200_ctx: one host thread <-> one GPU.  Implements upstream's `SegmentProver` with the TWO-PHASE form of the C ABI,
/// because the accum columns are upstream's to compute (`step_accum` needs the mix drawn after the DATA commit).
pub struct B200SegmentProver {
    ctx: *mut sys::hfb200_ctx,
    _tables: CircuitTables, // hfb200_init_ir copies nothing it needs later, but keep the tables alive with the context anyway
}

impl B200SegmentProver {
    pub fn new(device: i32, max_po2: u32) -> Result<Self> {
        let tables = CircuitTables::rv32im_v2();
        let ir = tables.ir();
        let mut ctx = std::ptr::null_mut();
        sys::ffi_wrap(|| unsafe { sys::hfb200_init_ir(device, max_po2, &ir, &mut ctx) })?;
        // default blinding = OS entropy per segment (include/hfb200.h); nothing to configure for production use
        Ok(Self { ctx, _tables: tables })
    }

    /// Column-major u32 Montgomery trace in, seal words out (what upstream's `Seal = Vec<u32>` holds).
    /// `accum_fn(mix) -> accum columns` is upstream's `step_accum`.
    pub fn prove_trace(
        &self, po2: u32, globals: &[u32], code: &[u32], data: &[u32], accum_fn: impl FnOnce(&[u32]) -> Result<Vec<u32>>,
    ) -> Result<Vec<u32>> {
        let n = 1usize << po2;
        if globals.len() != REGCOUNT_GLOBAL || code.len() != REGCOUNT_CODE * n || data.len() != REGCOUNT_DATA * n {
            bail!("trace shape does not match (rv32im-v2, po2 = {po2})");
        }
        let mut mix = vec![0u32; REGCOUNT_MIX];
        let mut mix_words = 0usize;
        sys::ffi_wrap(|| unsafe {
            sys::hfb200_segment_begin(self.ctx, po2, globals.as_ptr(), code.as_ptr(), data.as_ptr(), 0, mix.as_mut_ptr(), mix.len(), &mut mix_words)
        })?;
        mix.truncate(mix_words);
        let accum = accum_fn(&mix)?;
        if accum.len() != REGCOUNT_ACCUM * n {
            bail!("step_accum returned {} words, expected {}", accum.len(), REGCOUNT_ACCUM * n);
        }
        let cap = unsafe { sys::hfb200_seal_words(self.ctx, po2) };
        let mut seal = vec![0u32; cap];
        let mut words = 0usize;
        sys::ffi_wrap(|| unsafe { sys::hfb200_segment_finish(self.ctx, accum.as_ptr(), seal.as_mut_ptr(), cap, &mut words) })?;
        seal.truncate(words);
        Ok(seal)
    }

    /// Control id of (circuit, po2): commits the control columns once and keeps them on the device, so the segments that
    /// follow may pass an empty `code` slice (identical seals, no per-segment control commitment).
    pub fn load_control(&self, po2: u32, code: &[u32]) -> Result<[u32; 8]> {
        let mut root = [0u32; 8];
        sys::ffi_wrap(|| unsafe { sys::hfb200_control_root(self.ctx, po2, code.as_ptr(), root.as_mut_ptr()) })?;
        Ok(root)
    }
}

impl Drop for B200SegmentProver {
    fn drop(&mut self) {
        unsafe { sys::hfb200_destroy(self.ctx) }
    }
}

// [upstream] risc0_circuit_rv32im::prove::SegmentProver { fn prove(&self, segment: &Segment) -> Result<Seal>; }
impl SegmentProver for B200SegmentProver {
    fn prove(&self, segment: &risc0_circuit_rv32im::execute::Segment) -> Result<Seal> {
        // upstream CPU code, unchanged: preflight replays the segment, the witness generator fills code / data / global
        // (column-major Montgomery u32, blinding rows included) -- exactly the layout of include/hfb200.h
        let trace = segment.preflight()?;                                       // [upstream] execute::Segment::preflight
        let po2 = segment.po2 as u32;
        let witgen = WitnessGenerator::new(po2 as usize, &trace)?;              // [upstream] prove::witgen (CPU hal)
        let (global, code, data) = (witgen.global.as_u32_slice(), witgen.code.as_u32_slice(), witgen.data.as_u32_slice());
        self.prove_trace(po2, global, code, data, |mix| {
            // [upstream] CircuitImpl::step_accum over the CPU hal: accum columns from (code, data, global, mix)
            let accum = witgen.accum(&CircuitImpl, mix)?;
            Ok(accum.as_u32_slice().to_vec())
        })
    }
}

/// `Prover` over B200SegmentProver: upstream executor -> segments -> one seal per segment on the GPU -> upstream receipt types.
pub struct B200Prover {
    devices: Vec<i32>,
    max_po2: u32,
}

impl B200Prover {
    pub fn new(devices: Vec<i32>, max_po2: u32) -> Self {
        Self { devices, max_po2 }
    }

    fn prove_session(&self, ctx: &VerifierContext, session: &Session) -> Result<ProveInfo> {
        // Segments are independent (SURVEY.md section 8e): one worker thread and one context per GPU, segments handed out
        // from a shared index; no collective, only the seals return.  (The pool of include/hfb200.h -- hfb200_pool_prove with
        // hfb200_pool_set_accum -- carries upstream's step_accum once it runs on the device: a callback that launches
        // rv32im-sys's accum kernel on seg.stream.  That kernel is not part of this crate, so segments go through the host
        // two-phase path of B200SegmentProver here.)
        let n = session.segments.len();
        let next = std::sync::atomic::AtomicUsize::new(0);
        let seals: Vec<std::sync::Mutex<Option<Result<Seal>>>> = (0..n).map(|_| std::sync::Mutex::new(None)).collect();
        std::thread::scope(|scope| {
            for &device in &self.devices {
                let (next, seals, max_po2) = (&next, &seals, self.max_po2);
                scope.spawn(move || {
                    let prover = match B200SegmentProver::new(device, max_po2) {
                        Ok(p) => p,
                        Err(_) => return, // this GPU is unusable: the other workers take its share
                    };
                    loop {
                        let i = next.fetch_add(1, std::sync::atomic::Ordering::Relaxed);
                        if i >= n {
                            break;
                        }
                        let res = session.segments[i].resolve().and_then(|seg| prover.prove(&seg.inner)); // [upstream] SegmentRef::resolve
                        *seals[i].lock().unwrap() = Some(res);
                    }
                });
            }
        });
        let mut segments = Vec::with_capacity(n);
        for (i, cell) in seals.into_iter().enumerate() {
            let seal = cell.into_inner().unwrap().ok_or_else(|| anyhow!("segment {i}: no healthy GPU left"))??;
            let seg = session.segments[i].resolve()?;
            // [upstream] the claim is decoded from the seal's globals by upstream's own code path, exactly as for its CPU/CUDA provers
            let claim = risc0_zkvm::receipt::segment::decode_receipt_claim_from_seal(&seal)?;
            segments.push(SegmentReceipt {
                seal,
                index: seg.index as u32,
                hashfn: "poseidon2".into(),
                verifier_parameters: ctx.segment_verifier_parameters()?.digest(),
                claim,
            });
        }
        let composite = CompositeReceipt { segments, assumption_receipts: vec![], verifier_parameters: ctx.composite_verifier_parameters().digest() };
        let receipt = Receipt::new(InnerReceipt::Composite(composite), session.journal.clone().unwrap_or_default().bytes);
        receipt.verify_integrity_with_context(ctx)?; // upstream's verifier, as upstream's provers do before returning
        Ok(ProveInfo { receipt, stats: session.stats() })
    }
}

// [upstream] risc0_zkvm::Prover: `prove(env, elf)` is the provided method that calls prove_with_ctx with defaults
impl Prover for B200Prover {
    fn get_name(&self) -> String {
        "b200".into()
    }

    fn prove_with_ctx(&self, env: ExecutorEnv<'_>, ctx: &VerifierContext, elf: &[u8], opts: &ProverOpts) -> Result<ProveInfo> {
        if opts.hashfn != "poseidon2" {
            bail!("b200 prover: only the default poseidon2 hash suite is on the GPU path (asked for {})", opts.hashfn);
        }
        if !matches!(opts.receipt_kind, risc0_zkvm::ReceiptKind::Composite) {
            bail!("b200 prover: succinct / groth16 receipts need the recursion circuit; compress the composite receipt with upstream");
        }
        let mut exec = ExecutorImpl::from_elf(env, elf)?; // upstream executor, unchanged
        let session = exec.run()?;
        self.prove_session(ctx, &session)
    }

    fn compress(&self, _opts: &ProverOpts, _receipt: &Receipt) -> Result<Receipt> {
        bail!("b200 prover: receipt compression (lift / join / identity_p254) is upstream's recursion prover")
    }
}

/// `let prover = hfb200_prover::b200_prover();` replaces `default_prover()` (`/root/reference/host/src/main.rs:420`).
/// Devices: HFB200_DEVICES="0,1,..." or every visible GPU; segment size: the executor's default po2 = 20, prover limit 22.
pub fn b200_prover() -> Rc<dyn Prover> {
    let devices = std::env::var("HFB200_DEVICES")
        .ok()
        .map(|s| s.split(',').filter_map(|x| x.trim().parse().ok()).collect::<Vec<i32>>())
        .filter(|v| !v.is_empty())
        .unwrap_or_else(|| (0..visible_gpus()).collect());
    Rc::new(B200Prover::new(devices, 22))
}

fn visible_gpus() -> i32 {
    // a count is a query: no device or no driver is 0 GPUs, not an error (the prover then fails when it creates a context)
    let mut n: std::os::raw::c_int = 0;
    let e = unsafe { sys::hfb200_device_count(&mut n) };
    if !e.is_null() {
        unsafe { sys::hfb200_free_error(e) };
        return 1;
    }
    n.max(1)
}

/// `SegmentReceipt::verify_integrity` for the seals this library emits (host code, no GPU needed): `check_code` of upstream's
/// verifier becomes the comparison against `control_id` (one entry of the per-po2 control-id table).
pub fn verify_seal(seal: &[u32], control_id: &[u32; 8]) -> Result<u32> {
    let tables = CircuitTables::rv32im_v2();
    let ir = tables.ir();
    let mut po2 = 0u32;
    sys::ffi_wrap(|| unsafe { sys::hfb200_verify_segment(std::ptr::null(), &ir, seal.as_ptr(), seal.len(), control_id.as_ptr(), &mut po2) })?;
    Ok(po2)
}

/// All segment seals of a composite receipt in one call, fanned out over the host's threads (`hfb200_verify_segments`);
/// `control_ids[i]` is the control id of seal i's po2.  Returns the po2 of every seal; the error names the first rejected seal.
pub fn verify_seals(seals: &[&[u32]], control_ids: &[[u32; 8]]) -> Result<Vec<u32>> {
    anyhow::ensure!(seals.len() == control_ids.len(), "one control id per seal");
    let tables = CircuitTables::rv32im_v2();
    let ir = tables.ir();
    let ptrs: Vec<*const u32> = seals.iter().map(|s| s.as_ptr()).collect();
    let lens: Vec<usize> = seals.iter().map(|s| s.len()).collect();
    let roots: Vec<u32> = control_ids.iter().flat_map(|d| d.iter().copied()).collect();
    let mut po2 = vec![0u32; seals.len()];
    let mut first_bad = 0usize;
    sys::ffi_wrap(|| unsafe {
        sys::hfb200_verify_segments(std::ptr::null(), &ir, ptrs.as_ptr(), lens.as_ptr(), seals.len(), roots.as_ptr(), po2.as_mut_ptr(), 0, &mut first_bad)
    })?;
    Ok(po2)
}
