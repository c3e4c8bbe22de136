// C ABI of libhfb200.so (see include/hfb200.h for the boundary contract and reference citations).
#include "../../include/hfb200.h"
#include "prover.cuh"
#include "probe.cuh"
#include "verify.cuh"
#include "hal.cuh"
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <deque>
#include <map>
#include <memory>
#include <thread>

using namespace hf;

struct hfb200_ctx {
    Prover p;
    std::vector<uint32_t> seal;
#ifndef HFB200_EMU
    cudaEvent_t marks[4] = {nullptr, nullptr, nullptr, nullptr};
#endif
    // device HAL (hfb200_hal_*): scratch of the operators that need it, grown on demand, freed by hfb200_destroy
    void* hal_scratch = nullptr;
    size_t hal_scratch_cap = 0;
};

// the one message that is NOT malloc'd (returned when malloc itself fails); hfb200_free_error recognises it by address
static const char kOomMessage[] = "hfb200: out of memory while reporting an error";
static const char* dup_err(const std::string& s) {
    char* m = (char*)std::malloc(s.size() + 1);
    if (!m) return kOomMessage;
    std::memcpy(m, s.c_str(), s.size() + 1);
    return m;
}
#define API_TRY try {
#define API_CATCH } catch (const std::exception& e) { return dup_err(e.what()); } catch (...) { return dup_err("hfb200: unknown error"); } return nullptr;

// An error return must not leave copies from (or to) caller memory in flight: drain both streams before reporting it.
#define API_CATCH_QUIESCE(ctx_) } catch (const std::exception& e) { if (ctx_) (ctx_)->p.quiesce(); return dup_err(e.what()); } catch (...) { if (ctx_) (ctx_)->p.quiesce(); return dup_err("hfb200: unknown error"); } return nullptr;

static const char* emit_seal(hfb200_ctx* ctx, uint32_t* seal_out, size_t seal_cap, size_t* seal_words) {
    if (seal_words) *seal_words = ctx->seal.size();
    if (seal_cap < ctx->seal.size() || !seal_out) return dup_err("seal buffer too small: need " + std::to_string(ctx->seal.size()) + " words");
    std::memcpy(seal_out, ctx->seal.data(), ctx->seal.size() * 4);
    return nullptr;
}

extern "C" {

const char* hfb200_version(void) {
#ifdef HFB200_EMU
    return "hfb200 0.1 (HOST EMULATOR - test build, not a product)";
#else
    return "hfb200 0.1 (sm_100a)";
#endif
}

void hfb200_free_error(const char* msg) { if (msg && msg != kOomMessage) std::free((void*)msg); }

const char* hfb200_init(int device, uint32_t max_po2, const hfb200_circuit_desc* c, hfb200_ctx** out) {
    API_TRY
    if (!out) throw Err("hfb200_init: out is NULL");
    *out = nullptr;
    hfb200_circuit_desc d = c ? *c : hfb200_circuit_desc{16, 192, 48, 0};
    hfb200_ctx* ctx = new hfb200_ctx();
    try { ctx->p.init(device, max_po2, d.w_code, d.w_data, d.w_accum); } catch (...) { delete ctx; throw; }
    *out = ctx;
    API_CATCH
}
const char* hfb200_init_ir(int device, uint32_t max_po2, const hfb200_circuit_ir* c, hfb200_ctx** out) {
    API_TRY
    if (!out || !c) throw Err("hfb200_init_ir: NULL argument");
    *out = nullptr;
    static_assert(sizeof(hfb200_tap) == sizeof(IrTap) && sizeof(hfb200_poly_step) == sizeof(IrStep), "IR layouts must match");
    hfb200_ctx* ctx = new hfb200_ctx();
    try {
        ctx->p.init(device, max_po2, c->w_code, c->w_data, c->w_accum, reinterpret_cast<const IrTap*>(c->taps), c->n_taps,
                    reinterpret_cast<const IrStep*>(c->steps), c->n_steps, c->ret, c->n_mix, c->info);
    } catch (...) { delete ctx; throw; }
    *out = ctx;
    API_CATCH
}
const char* hfb200_ir_source(const hfb200_circuit_ir* c, char* out, size_t cap, size_t* need) {
    API_TRY
    if (!c) throw Err("hfb200_ir_source: NULL circuit");
    GenericCircuitHost g;
    g.init(nullptr, c->w_code, c->w_data, c->w_accum, c->n_mix, reinterpret_cast<const IrTap*>(c->taps), c->n_taps,
           reinterpret_cast<const IrStep*>(c->steps), c->n_steps, c->ret);
    const std::string src = jit_source(g);
    if (need) *need = src.size() + 1;
    if (out && cap) { const size_t n = std::min(cap - 1, src.size()); std::memcpy(out, src.data(), n); out[n] = 0; }
    API_CATCH
}
int hfb200_ir_jit_active(const hfb200_ctx* ctx, float* compile_ms) {
    if (!ctx) return 0;
    if (compile_ms) *compile_ms = ctx->p.jit.compile_ms;
    return ctx->p.jit.ready ? 1 : 0;
}
const char* hfb200_ir_compile(const hfb200_circuit_ir* c, const uint32_t* po2s, size_t n_po2, unsigned threads, void* bundle_out, size_t cap,
                              size_t* need) {
    API_TRY
#ifdef HFB200_EMU
    (void)c; (void)po2s; (void)n_po2; (void)threads; (void)bundle_out; (void)cap; (void)need;
    throw Err("hfb200_ir_compile: the host emulator build has no sm_100a kernels to compile");
#else
    if (!c || (!po2s && n_po2)) throw Err("hfb200_ir_compile: NULL argument");
    if (need) *need = 0;
    for (size_t i = 0; i < n_po2; i++) if (po2s[i] < MIN_PO2 || po2s[i] > MAX_PO2) throw Err("po2 must be in [12, 22]");
    GenericCircuitHost g;  // the checks of hfb200_init_ir, without a device
    g.init(nullptr, c->w_code, c->w_data, c->w_accum, c->n_mix, reinterpret_cast<const IrTap*>(c->taps), c->n_taps,
           reinterpret_cast<const IrStep*>(c->steps), c->n_steps, c->ret);
    std::vector<uint32_t> sizes(po2s, po2s + n_po2);  // ascending, each once: the bundle does not depend on the request's order
    std::sort(sizes.begin(), sizes.end());
    sizes.erase(std::unique(sizes.begin(), sizes.end()), sizes.end());
    std::vector<JitSpec> specs;
    std::vector<std::vector<JitCubin>> bins;
    for (uint32_t po2 : sizes) {
        specs.push_back(jit_spec(g, po2, threads));
        bins.push_back(JitCache::get().fetch(specs.back(), threads));
        for (const JitCubin& b : bins.back())
            if (!b) { std::string why; JitCache::get().nvrtc(&why); throw Err("hfb200_ir_compile: po2 " + std::to_string(po2) + " is not cached and NVRTC is unavailable: " + why); }
    }
    if (!bundle_out && !need) return nullptr;
    const std::string b = jit_bundle(specs, bins, threads);
    if (need) *need = b.size();
    if (bundle_out) {
        if (cap < b.size()) throw Err("hfb200_ir_compile: bundle buffer too small: need " + std::to_string(b.size()) + " bytes");
        std::memcpy(bundle_out, b.data(), b.size());
    }
#endif
    API_CATCH
}
const char* hfb200_ir_load_kernels(const void* bundle, size_t bytes, size_t* specialisations) {
    API_TRY
    if (specialisations) *specialisations = 0;
#ifdef HFB200_EMU
    (void)bundle; (void)bytes;
    throw Err("hfb200_ir_load_kernels: the host emulator build runs no sm_100a kernels");
#else
    if (!bundle && bytes) throw Err("hfb200_ir_load_kernels: NULL bundle");
    size_t n = 0;
    const auto recs = jit_parse_bundle(static_cast<const uint8_t*>(bundle), bytes, &n);
    JitCache::get().add(recs);
    if (specialisations) *specialisations = n;
#endif
    API_CATCH
}
uint64_t hfb200_ir_nvrtc_programs(void) {
#ifdef HFB200_EMU
    return 0;
#else
    return JitCache::get().programs.load();
#endif
}
void hfb200_destroy(hfb200_ctx* ctx) {
    if (!ctx) return;
#ifndef HFB200_EMU
    for (auto& m : ctx->marks) if (m) { cudaEventDestroy(m); m = nullptr; }
#endif
    try { ctx->p.dev.free(ctx->hal_scratch); ctx->p.destroy(); } catch (...) {}
    delete ctx;
}

const char* hfb200_set_blinding(hfb200_ctx* ctx, int mode) {
    API_TRY
    if (!ctx) throw Err("hfb200_set_blinding: NULL ctx");
    if (mode != BLIND_OS_ENTROPY && mode != BLIND_DETERMINISTIC) throw Err("hfb200_set_blinding: mode must be HFB200_BLIND_OS_ENTROPY or HFB200_BLIND_DETERMINISTIC");
    if (ctx->p.begun) throw Err("hfb200_set_blinding: a segment is in flight");
    ctx->p.blind_mode = mode;
    API_CATCH
}

const char* hfb200_set_transcript(hfb200_ctx* ctx, int on_device) {
    API_TRY
    if (!ctx) throw Err("hfb200_set_transcript: NULL ctx");
    if (ctx->p.begun) throw Err("hfb200_set_transcript: a segment is in flight");
    if (on_device < 0 || on_device > 2) throw Err("hfb200_set_transcript: mode must be 0 (host), 1 (device) or 2 (device + CUDA-graph replay)");
    if (on_device >= 1 && ctx->p.hash_suite == HASH_SHA256) throw Err("hfb200_set_transcript: the SHA-256 suite runs the host transcript only");
    ctx->p.transcript_mode = on_device;
    API_CATCH
}

const char* hfb200_set_hash_suite(hfb200_ctx* ctx, int suite) {
    API_TRY
    if (!ctx) throw Err("hfb200_set_hash_suite: NULL ctx");
    try { ctx->p.set_hash_suite(suite); } catch (const Err& e) { throw Err(std::string("hfb200_set_hash_suite: ") + e.what()); }
    API_CATCH
}

uint64_t hfb200_graph_launches(const hfb200_ctx* ctx) { return ctx ? ctx->p.graph_launches : 0; }

const char* hfb200_host_alloc(size_t bytes, void** out) {
    API_TRY
    if (!out) throw Err("hfb200_host_alloc: out is NULL");
    *out = nullptr;
#ifndef HFB200_EMU
    CUDA_CHECK(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
#else
    *out = std::malloc(bytes);
#endif
    API_CATCH
}
void hfb200_host_free(void* p) {
#ifndef HFB200_EMU
    cudaFreeHost(p);
#else
    std::free(p);
#endif
}

const char* hfb200_prove_segment(hfb200_ctx* ctx, uint32_t po2, const uint32_t* globals, const uint32_t* code, const uint32_t* data,
                                 uint64_t blind_seed, uint32_t* seal_out, size_t seal_cap, size_t* seal_words) {
    API_TRY
    if (!ctx || !globals || !data) throw Err("hfb200_prove_segment: NULL argument");
    if (ctx->p.device_transcript()) ctx->p.prove_device(po2, globals, code, data, blind_seed, ctx->seal);
    else { ctx->p.begin(po2, globals, code, data, blind_seed); ctx->p.finish(nullptr, ctx->seal); }
    if (const char* e = emit_seal(ctx, seal_out, seal_cap, seal_words)) return e;
    API_CATCH_QUIESCE(ctx)
}

const char* hfb200_segment_begin(hfb200_ctx* ctx, uint32_t po2, const uint32_t* globals, const uint32_t* code, const uint32_t* data,
                                 uint64_t blind_seed, uint32_t* mix_out, size_t mix_cap, size_t* mix_words) {
    API_TRY
    if (!ctx || !globals) throw Err("hfb200_segment_begin: NULL argument");
    ctx->p.begin(po2, globals, code, data, blind_seed);
    if (mix_words) *mix_words = ctx->p.mix.size();
    if (mix_out) {
        if (mix_cap < ctx->p.mix.size()) throw Err("mix buffer too small");
        std::memcpy(mix_out, ctx->p.mix.data(), ctx->p.mix.size() * 4);
    }
    API_CATCH_QUIESCE(ctx)
}
const char* hfb200_segment_finish(hfb200_ctx* ctx, const uint32_t* accum_or_null, uint32_t* seal_out, size_t seal_cap, size_t* seal_words) {
    API_TRY
    if (!ctx) throw Err("hfb200_segment_finish: NULL ctx");
    ctx->p.finish(accum_or_null, ctx->seal);
    if (const char* e = emit_seal(ctx, seal_out, seal_cap, seal_words)) return e;
    API_CATCH_QUIESCE(ctx)
}

const char* hfb200_segment_begin_dev(hfb200_ctx* ctx, uint32_t po2, const uint32_t* globals, const uint32_t* code, const uint32_t* data,
                                     uint64_t blind_seed, uint32_t flags, hfb200_segment_dev* out) {
    API_TRY
    if (!ctx || !globals || !out) throw Err("hfb200_segment_begin_dev: NULL argument");
    if (flags & ~(uint32_t)HFB200_DEV_INPUTS) throw Err("hfb200_segment_begin_dev: unknown flags");
    Prover& p = ctx->p;
    p.begin_dev(po2, globals, code, data, blind_seed, (flags & HFB200_DEV_INPUTS) != 0);
    hfb200_segment_dev s{};
    s.po2 = p.po2; s.zk_rows = ZK_CYCLES;
    s.w_code = p.cir.cd.w_code; s.w_data = p.cir.cd.w_data; s.w_accum = p.cir.cd.w_accum; s.n_mix = (uint32_t)p.mix.size();
    s.device = p.device_id;
    s.stream = (void*)p.dev.stream;
    s.code = p.tr[GROUP_CODE]; s.data = p.tr[GROUP_DATA]; s.globals = p.d_globals; s.mix = p.d_mix; s.accum = p.tr[GROUP_ACCUM];
    s.mix_host = p.mix.data(); s.globals_host = p.globals;
    s.blind_seed = blind_seed;
    *out = s;
    API_CATCH_QUIESCE(ctx)
}
const char* hfb200_segment_finish_dev(hfb200_ctx* ctx, uint32_t* seal_out, size_t seal_cap, size_t* seal_words) {
    API_TRY
    if (!ctx) throw Err("hfb200_segment_finish_dev: NULL ctx");
    ctx->p.finish(nullptr, ctx->seal, true);
    if (const char* e = emit_seal(ctx, seal_out, seal_cap, seal_words)) return e;
    API_CATCH_QUIESCE(ctx)
}
// argument errors leave the segment in flight (nothing was queued); the caller may still finish or abandon it
const char* hfb200_segment_accum_scan(hfb200_ctx* ctx, int kind, uint32_t first_chain, uint32_t n_chains, size_t rows) {
    API_TRY
    if (!ctx) throw Err("hfb200_segment_accum_scan: NULL ctx");
    ctx->p.accum_scan(kind, first_chain, n_chains, rows);
    API_CATCH
}
const char* hfb200_segment_accum_blind(hfb200_ctx* ctx) {
    API_TRY
    if (!ctx) throw Err("hfb200_segment_accum_blind: NULL ctx");
    ctx->p.accum_blind();
    API_CATCH
}
const char* hfb200_segment_witness_dev(hfb200_ctx* ctx, uint32_t po2, uint64_t blind_seed, hfb200_witness_dev* out) {
    API_TRY
    if (!ctx || !out) throw Err("hfb200_segment_witness_dev: NULL argument");
    Prover& p = ctx->p;
    p.witness_dev(po2, blind_seed);
    hfb200_witness_dev w{};
    w.po2 = p.po2; w.zk_rows = ZK_CYCLES;
    w.w_code = p.cir.cd.w_code; w.w_data = p.cir.cd.w_data;
    w.device = p.device_id;
    w.stream = (void*)p.dev.stream;
    w.data = p.tr[GROUP_DATA];
    *out = w;
    API_CATCH
}
const char* hfb200_segment_data_blind(hfb200_ctx* ctx) {
    API_TRY
    if (!ctx) throw Err("hfb200_segment_data_blind: NULL ctx");
    ctx->p.data_blind();
    API_CATCH
}
const char* hfb200_segment_scratch(hfb200_ctx* ctx, size_t bytes, void** out) {
    API_TRY
    if (!ctx || !out) throw Err("hfb200_segment_scratch: NULL argument");
    *out = ctx->p.segment_scratch(bytes);
    API_CATCH
}
const char* hfb200_device_count(int* out) {
    API_TRY
    if (!out) throw Err("hfb200_device_count: out is NULL");
    *out = 0;
#ifndef HFB200_EMU
    int n = 0;
    const cudaError_t e = cudaGetDeviceCount(&n);
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) { cudaGetLastError(); return nullptr; }  // a count of zero
    CUDA_CHECK(e);
    *out = n;
#else
    *out = 1;
#endif
    API_CATCH
}

const char* hfb200_witgen_synth(hfb200_ctx* ctx, uint32_t po2, uint64_t trace_seed, uint64_t blind_seed, uint32_t* globals_out) {
    API_TRY
    if (!ctx || !globals_out) throw Err("hfb200_witgen_synth: NULL argument");
    ctx->p.witgen(po2, trace_seed, blind_seed, globals_out);
    API_CATCH
}
const char* hfb200_prove_resident(hfb200_ctx* ctx, uint64_t blind_seed, uint32_t* seal_out, size_t seal_cap, size_t* seal_words) {
    API_TRY
    if (!ctx) throw Err("hfb200_prove_resident: NULL ctx");
    if (!ctx->p.have_trace) throw Err("hfb200_prove_resident: no resident trace (call hfb200_witgen_synth)");
    uint32_t g[N_GLOBAL];
    std::memcpy(g, ctx->p.globals, sizeof g);
    if (ctx->p.device_transcript()) ctx->p.prove_device(ctx->p.po2, g, nullptr, nullptr, blind_seed, ctx->seal);
    else { ctx->p.begin(ctx->p.po2, g, nullptr, nullptr, blind_seed); ctx->p.finish(nullptr, ctx->seal); }
    if (const char* e = emit_seal(ctx, seal_out, seal_cap, seal_words)) return e;
    API_CATCH_QUIESCE(ctx)
}
const char* hfb200_read_group(hfb200_ctx* ctx, uint32_t group, uint32_t* out, size_t cap_words) {
    API_TRY
    if (!ctx || group > 2 || !ctx->p.tr[group]) throw Err("hfb200_read_group: bad argument");
    ctx->p.bind();
    const size_t words = (size_t)ctx->p.cir.group_width((int)group) << ctx->p.po2;
    if (cap_words < words) throw Err("hfb200_read_group: buffer too small");
    ctx->p.dev.d2h(out, ctx->p.tr[group], words * 4);
    ctx->p.dev.sync();
    API_CATCH
}

size_t hfb200_seal_words(const hfb200_ctx* ctx, uint32_t po2) { return ctx && po2 >= MIN_PO2 && po2 <= MAX_PO2 ? ctx->p.seal_words(po2) : 0; }

const char* hfb200_checkpoint(hfb200_ctx* ctx, const char* name, uint32_t* out, size_t cap, size_t* n_words) {
    API_TRY
    if (!ctx || !name) throw Err("hfb200_checkpoint: NULL argument");
    for (auto& kv : ctx->p.cps)
        if (kv.first == name) {
            if (n_words) *n_words = kv.second.size();
            if (out) { if (cap < kv.second.size()) throw Err("checkpoint buffer too small"); std::memcpy(out, kv.second.data(), kv.second.size() * 4); }
            return nullptr;
        }
    throw Err(std::string("no such checkpoint: ") + name);
    API_CATCH
}

const char* hfb200_last_stats(hfb200_ctx* ctx, hfb200_stats* out) {
    API_TRY
    if (!ctx || !out) throw Err("hfb200_last_stats: NULL argument");
    const Stats& s = ctx->p.stats;
    out->ms_total = s.ms_total; out->ms_device = s.ms_device; out->ms_h2d = s.ms_h2d; out->ms_ntt_main = s.ms_ntt_main; out->ms_hash_main = s.ms_hash_main;
    out->ms_accum = s.ms_accum; out->ms_check = s.ms_check; out->ms_deep = s.ms_deep; out->ms_fri = s.ms_fri;
    out->launches = s.launches; out->ntt_main_bytes = s.ntt_main_bytes; out->host_syncs = s.host_syncs;
    API_CATCH
}
uint64_t hfb200_total_launches(const hfb200_ctx* ctx) { return ctx ? ctx->p.dev.launches : 0; }

// ---- multi-GPU pool ---------------------------------------------------------------------------------
} // extern "C"
// Replaces the (sequential) segment loop of upstream's `ProverImpl::prove_session`.  Failure behaviour follows the reference's
// batch tooling (/root/reference/data/watchdog.sh:58-83: a failed input is set aside, the rest continue) and its prover call
// site (/root/reference/host/src/main.rs:327-330: the error is surfaced, not swallowed):
//   * an argument / shape error fails that job only; it is never retried;
//   * a CUDA error poisons the context that saw it: the context is destroyed and re-created (the device is retired for this
//     pool if that fails), and the job goes back to the queue for any healthy worker, at most HFB200_POOL_MAX_ATTEMPTS times;
//   * jobs left when no healthy context remains fail with that reason.
static constexpr int HFB200_POOL_MAX_ATTEMPTS = 3;
struct hfb200_pool {
    struct Slot { hfb200_ctx* ctx = nullptr; int device = 0; bool retired = false; uint64_t faults = 0; };
    std::vector<Slot> slots;
    struct Control { const uint32_t* code; uint64_t gen; };
    std::map<uint32_t, Control> control;  // po2 -> caller-owned control columns + the load that installed them
    uint64_t next_gen = 1;
    // what is needed to re-create a context after a fault
    uint32_t max_po2 = 0;
    hfb200_circuit_desc desc{};
    bool is_ir = false;
    std::vector<IrTap> ir_taps; std::vector<IrStep> ir_steps; uint32_t ir_ret = 0, ir_n_mix = 0; uint8_t ir_info[16] = {0};
    int blind_mode = BLIND_OS_ENTROPY;
    int hash_suite = HASH_POSEIDON2;
    // the caller's step_accum (hfb200_pool_set_accum): jobs then run begin_dev -> accum_fn -> finish_dev
    hfb200_accum_fn accum_fn = nullptr;
    void* accum_user = nullptr;
    // the caller's witness generator (hfb200_pool_set_witgen): jobs with data == NULL then run witness_dev -> witgen_fn -> begin ...
    hfb200_witgen_fn witgen_fn = nullptr;
    void* witgen_user = nullptr;
    // test hook (hfb200_pool_inject_fault): worker `w` reports a CUDA error instead of proving its n-th job from now
    std::mutex inject_mu;
    std::map<size_t, std::pair<uint64_t, int>> inject;  // worker -> (jobs to let pass, kind)
    uint64_t total_faults = 0, total_retries = 0, contexts_recreated = 0;

    hfb200_ctx* make_ctx(int device) const {
        hfb200_ctx* ctx = new hfb200_ctx();
        try {
            if (is_ir) ctx->p.init(device, max_po2, desc.w_code, desc.w_data, desc.w_accum, ir_taps.data(), ir_taps.size(), ir_steps.data(), ir_steps.size(), ir_ret, ir_n_mix, ir_info);
            else ctx->p.init(device, max_po2, desc.w_code, desc.w_data, desc.w_accum);
            ctx->p.blind_mode = blind_mode;
            ctx->p.set_hash_suite(hash_suite);
        } catch (...) { try { ctx->p.destroy(); } catch (...) {} delete ctx; throw; }
        return ctx;
    }
    void drop_ctx(Slot& sl) {
        if (!sl.ctx) return;
#ifndef HFB200_EMU
        cudaSetDevice(sl.device);
#endif
        hfb200_destroy(sl.ctx);
        sl.ctx = nullptr;
    }
    ~hfb200_pool() { for (auto& sl : slots) drop_ctx(sl); }
};

static void pool_fill(hfb200_pool* pool, const int* devices, int n_devices, int contexts_per_device) {
    // contexts are created up front, serially (cudaSetDevice is per thread); on failure the pool's destructor releases the
    // contexts already made (arenas, streams, events)
    for (int i = 0; i < n_devices; i++)
        for (int s_ = 0; s_ < contexts_per_device; s_++) {
            hfb200_pool::Slot sl;
            sl.device = devices[i];
            sl.ctx = pool->make_ctx(devices[i]);
            pool->slots.push_back(sl);
        }
}
static bool is_device_fault(const char* msg) { return msg && std::strncmp(msg, "CUDA error", 10) == 0; }
// One job through the device seam: begin_dev (the job's host inputs), the caller's step_accum on this worker thread, finish_dev.
// A nonzero return of the callback fails the job (never retried) and abandons the segment: the stream is drained so that the
// context is usable for the next job.  If draining it reports a CUDA error, the callback met a device fault: the worker takes
// the device-fault path (context re-created, job re-queued).
static const char* abandon_after_callback(hfb200_ctx* ctx, const char* which, int rc) {
#ifndef HFB200_EMU
    cudaSetDevice(ctx->p.device_id);
    const cudaError_t e = cudaStreamSynchronize(ctx->p.dev.stream);
    ctx->p.quiesce();
    if (e != cudaSuccess)
        return dup_err(std::string("CUDA error ") + cudaGetErrorName(e) + " after the " + which + " callback: " + cudaGetErrorString(e));
#else
    ctx->p.quiesce();
#endif
    return dup_err(std::string(which) + " callback returned " + std::to_string(rc));
}
static const char* prove_job_with_accum(hfb200_pool* pool, hfb200_ctx* ctx, hfb200_segment_job& j, size_t idx) {
    hfb200_segment_dev seg;
    if (const char* e = hfb200_segment_begin_dev(ctx, j.po2, j.globals, j.code, j.data, j.blind_seed, 0, &seg)) return e;
    const int rc = pool->accum_fn(pool->accum_user, ctx, &seg, idx);
    if (rc != 0) return abandon_after_callback(ctx, "accum", rc);
    return hfb200_segment_finish_dev(ctx, j.seal_out, j.seal_cap, &j.seal_words);
}
// A job with data == NULL through the witness seam: witness_dev, the caller's witness generator on this worker thread, then the
// accum stage (the accum callback, or the built-in step_accum of a built-in pool).  Failures as in prove_job_with_accum.
static const char* prove_job_with_witgen(hfb200_pool* pool, hfb200_ctx* ctx, hfb200_segment_job& j, size_t idx) {
    hfb200_witness_dev w;
    if (const char* e = hfb200_segment_witness_dev(ctx, j.po2, j.blind_seed, &w)) return e;
    const int rc = pool->witgen_fn(pool->witgen_user, ctx, &w, idx);
    if (rc != 0) return abandon_after_callback(ctx, "witgen", rc);
    if (pool->accum_fn) return prove_job_with_accum(pool, ctx, j, idx);
    if (const char* e = hfb200_segment_begin(ctx, j.po2, j.globals, j.code, nullptr, j.blind_seed, nullptr, 0, nullptr)) return e;
    return hfb200_segment_finish(ctx, nullptr, j.seal_out, j.seal_cap, &j.seal_words);
}
static const char* control_root_impl(hfb200_ctx* ctx, uint32_t po2, const uint32_t* code, uint32_t* root_out, uint64_t gen);
extern "C" {

const char* hfb200_pool_create(const int* devices, int n_devices, int contexts_per_device, uint32_t max_po2,
                               const hfb200_circuit_desc* c, hfb200_pool** out) {
    API_TRY
    if (!out || !devices || n_devices <= 0 || contexts_per_device <= 0) throw Err("hfb200_pool_create: bad argument");
    *out = nullptr;
    std::unique_ptr<hfb200_pool> pool(new hfb200_pool());
    pool->desc = c ? *c : hfb200_circuit_desc{16, 192, 48, 0};
    pool->max_po2 = max_po2;
    pool_fill(pool.get(), devices, n_devices, contexts_per_device);
    *out = pool.release();
    API_CATCH
}
const char* hfb200_pool_create_ir(const int* devices, int n_devices, int contexts_per_device, uint32_t max_po2,
                                  const hfb200_circuit_ir* c, hfb200_pool** out) {
    API_TRY
    if (!out || !devices || !c || n_devices <= 0 || contexts_per_device <= 0) throw Err("hfb200_pool_create_ir: bad argument");
    *out = nullptr;
    std::unique_ptr<hfb200_pool> pool(new hfb200_pool());
    pool->desc = hfb200_circuit_desc{c->w_code, c->w_data, c->w_accum, 0};
    pool->max_po2 = max_po2;
    pool->is_ir = true;
    const IrTap* t = reinterpret_cast<const IrTap*>(c->taps);
    const IrStep* st = reinterpret_cast<const IrStep*>(c->steps);
    pool->ir_taps.assign(t, t + c->n_taps);
    pool->ir_steps.assign(st, st + c->n_steps);
    pool->ir_ret = c->ret; pool->ir_n_mix = c->n_mix; std::memcpy(pool->ir_info, c->info, 16);
    pool_fill(pool.get(), devices, n_devices, contexts_per_device);
    *out = pool.release();
    API_CATCH
}
const char* hfb200_pool_set_blinding(hfb200_pool* pool, int mode) {
    API_TRY
    if (!pool) throw Err("hfb200_pool_set_blinding: NULL pool");
    if (mode != BLIND_OS_ENTROPY && mode != BLIND_DETERMINISTIC) throw Err("hfb200_pool_set_blinding: bad mode");
    pool->blind_mode = mode;
    for (auto& sl : pool->slots) if (sl.ctx) sl.ctx->p.blind_mode = mode;
    API_CATCH
}
const char* hfb200_pool_set_hash_suite(hfb200_pool* pool, int suite) {
    API_TRY
    if (!pool) throw Err("hfb200_pool_set_hash_suite: NULL pool");
    if (!hash_suite_valid(suite)) throw Err("hfb200_pool_set_hash_suite: suite must be HFB200_HASH_POSEIDON2 (0) or HFB200_HASH_SHA256 (1)");
    for (auto& sl : pool->slots) if (sl.ctx) sl.ctx->p.set_hash_suite(suite);
    pool->hash_suite = suite;
    API_CATCH
}
const char* hfb200_pool_inject_fault(hfb200_pool* pool, size_t worker, uint64_t after_jobs, int kind) {
    API_TRY
    if (!pool || worker >= pool->slots.size() || kind < 0 || kind > 1) throw Err("hfb200_pool_inject_fault: bad argument");
    std::lock_guard<std::mutex> lock(pool->inject_mu);
    pool->inject[worker] = std::make_pair(after_jobs, kind);
    API_CATCH
}
const char* hfb200_pool_stats(const hfb200_pool* pool, hfb200_pool_stats_t* out) {
    API_TRY
    if (!pool || !out) throw Err("hfb200_pool_stats: NULL argument");
    out->contexts = pool->slots.size();
    out->contexts_retired = 0;
    for (const auto& sl : pool->slots) if (sl.retired) out->contexts_retired++;
    out->faults = pool->total_faults; out->retries = pool->total_retries; out->contexts_recreated = pool->contexts_recreated;
    API_CATCH
}

const char* hfb200_pool_prove(hfb200_pool* pool, hfb200_segment_job* jobs, size_t n_jobs) {
    API_TRY
    if (!pool || (!jobs && n_jobs)) throw Err("hfb200_pool_prove: bad argument");
    std::vector<size_t> order(n_jobs);
    for (size_t i = 0; i < n_jobs; i++) { order[i] = i; jobs[i].error = nullptr; jobs[i].seal_words = 0; jobs[i].device = -1; jobs[i].ms = 0; jobs[i].attempts = 0; }
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return jobs[a].po2 > jobs[b].po2; });  // longest first
    // argument checks up front: a mis-shaped job must not reach cudaMemcpyAsync
    for (size_t i = 0; i < n_jobs; i++) {
        hfb200_segment_job& j = jobs[i];
        if (!j.globals || (!j.data && !pool->witgen_fn) || !j.seal_out) { j.error = dup_err("job has a NULL globals / data / seal_out pointer"); continue; }
        if (!j.data && pool->is_ir && !pool->accum_fn) {
            j.error = dup_err("data-defined circuit: step_accum is the caller's (install an accum callback with hfb200_pool_set_accum)");
            continue;
        }
        if (j.po2 < MIN_PO2 || j.po2 > pool->max_po2) { j.error = dup_err("job po2 " + std::to_string(j.po2) + " outside [12, " + std::to_string(pool->max_po2) + "]"); continue; }
        const size_t need = hfb200_seal_words(pool->slots.empty() ? nullptr : pool->slots[0].ctx, j.po2);
        if (need && j.seal_cap < need) { j.seal_words = need; j.error = dup_err("seal buffer too small: need " + std::to_string(need) + " words"); }
    }
    std::mutex mu;
    std::condition_variable cv;
    std::deque<size_t> pending;
    for (size_t k = 0; k < n_jobs; k++) if (!jobs[order[k]].error) pending.push_back(order[k]);
    size_t inflight = 0;
    // contexts in flight per device follow the queue depth: extra contexts only hide copies and host round trips of OTHER
    // segments; with fewer jobs than contexts they would split the SMs between segments that could have run back to back
    std::map<int, size_t> per_device_cap;
    {
        std::map<int, size_t> live;
        for (const auto& sl : pool->slots) if (!sl.retired) live[sl.device]++;
        const size_t n_dev = live.empty() ? 1 : live.size();
        const size_t jobs_per_device = (pending.size() + n_dev - 1) / n_dev;
        for (const auto& kv : live) per_device_cap[kv.first] = std::max<size_t>(1, std::min(kv.second, (jobs_per_device + 1) / 2));
    }
    std::vector<char> taken(pool->slots.size(), 0);  // slots that have (had) a worker thread in this call
    auto worker = [&](size_t w) {
        for (;;) {
            hfb200_pool::Slot& sl = pool->slots[w];
#ifndef HFB200_EMU
            cudaSetDevice(sl.device);
#endif
            size_t idx;
            {
                std::unique_lock<std::mutex> lock(mu);
                cv.wait(lock, [&] { return !pending.empty() || inflight == 0; });
                if (pending.empty()) return;  // nothing queued and nothing in flight that could come back
                idx = pending.front(); pending.pop_front();
                inflight++;
            }
            hfb200_segment_job& j = jobs[idx];
            const auto t0 = std::chrono::steady_clock::now();
            j.attempts++;
            const char* err = nullptr;
            int injected = -1;
            {
                std::lock_guard<std::mutex> lock(pool->inject_mu);
                auto it = pool->inject.find(w);
                if (it != pool->inject.end()) { if (it->second.first == 0) { injected = it->second.second; pool->inject.erase(it); } else it->second.first--; }
            }
            if (injected == 0) err = dup_err("CUDA error cudaErrorLaunchFailure (injected by hfb200_pool_inject_fault)");
            else if (injected == 1) err = dup_err("injected non-device failure");
            if (!err && !j.code) {
                // shared control group: (re)commit it on this context when the resident one is not the current load for this po2
                const auto it = pool->control.find(j.po2);
                if (it == pool->control.end()) err = dup_err("code is NULL and no control group was loaded for this po2 (hfb200_pool_load_control)");
                else if (!(sl.ctx->p.control_cached && sl.ctx->p.po2 == j.po2 && sl.ctx->p.control_gen == it->second.gen)) {
                    uint32_t root[8];
                    err = control_root_impl(sl.ctx, j.po2, it->second.code, root, it->second.gen);
                }
            }
            if (!err && !j.data) err = prove_job_with_witgen(pool, sl.ctx, j, idx);
            else if (!err && pool->accum_fn) err = prove_job_with_accum(pool, sl.ctx, j, idx);
            else if (!err) err = hfb200_prove_segment(sl.ctx, j.po2, j.globals, j.code, j.data, j.blind_seed, j.seal_out, j.seal_cap, &j.seal_words);
            j.device = sl.device;
            j.ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
            bool requeue = false, retire = false;
            if (err && is_device_fault(err)) {
                // the context (streams, in-flight work, possibly the whole device) is suspect: rebuild it before anything else runs on it
                pool->drop_ctx(sl);
                try { sl.ctx = pool->make_ctx(sl.device); } catch (...) { sl.ctx = nullptr; retire = true; }
                requeue = j.attempts < HFB200_POOL_MAX_ATTEMPTS;
            }
            {
                std::lock_guard<std::mutex> lock(mu);
                if (err && is_device_fault(err)) { pool->total_faults++; sl.faults++; if (!retire) pool->contexts_recreated++; }
                if (requeue) { hfb200_free_error(err); err = nullptr; pool->total_retries++; pending.push_back(idx); }
                j.error = err;
                if (retire) sl.retired = true;
                inflight--;
            }
            cv.notify_all();
            if (retire) {
                // this slot is gone: carry on as the worker of a spare healthy slot (one the queue-depth cap left idle), if any
                std::lock_guard<std::mutex> lock(mu);
                size_t spare = pool->slots.size();
                for (size_t k = 0; k < pool->slots.size(); k++) if (!taken[k] && !pool->slots[k].retired && pool->slots[k].ctx) { spare = k; break; }
                if (spare == pool->slots.size()) return;
                taken[spare] = 1;
                w = spare;
            }
        }
    };
    std::vector<std::thread> th;
    std::map<int, size_t> started;
    for (size_t w = 0; w < pool->slots.size(); w++) {
        const auto& sl = pool->slots[w];
        if (sl.retired || !sl.ctx) continue;
        if (started[sl.device] >= per_device_cap[sl.device]) continue;
        started[sl.device]++;
        taken[w] = 1;
        th.emplace_back(worker, w);
    }
    for (auto& t : th) t.join();
    for (size_t idx : pending) if (!jobs[idx].error) jobs[idx].error = dup_err("no healthy context left in the pool (every worker retired after CUDA errors)");
    for (size_t i = 0; i < n_jobs; i++)
        if (jobs[i].error) return dup_err(std::string("job ") + std::to_string(i) + ": " + jobs[i].error);
    API_CATCH
}

const char* hfb200_pool_load_control(hfb200_pool* pool, uint32_t po2, const uint32_t* code) {
    API_TRY
    if (!pool) throw Err("hfb200_pool_load_control: NULL pool");
    // every load gets a new generation: a worker whose resident control group came from an earlier load (even of the same
    // pointer: the caller may have rewritten the columns) re-commits it before its next code == NULL job
    if (code) pool->control[po2] = hfb200_pool::Control{code, pool->next_gen++}; else pool->control.erase(po2);
    API_CATCH
}

const char* hfb200_pool_set_accum(hfb200_pool* pool, hfb200_accum_fn fn, void* user) {
    API_TRY
    if (!pool) throw Err("hfb200_pool_set_accum: NULL pool");
    pool->accum_fn = fn;
    pool->accum_user = fn ? user : nullptr;
    API_CATCH
}

const char* hfb200_pool_set_witgen(hfb200_pool* pool, hfb200_witgen_fn fn, void* user) {
    API_TRY
    if (!pool) throw Err("hfb200_pool_set_witgen: NULL pool");
    pool->witgen_fn = fn;
    pool->witgen_user = fn ? user : nullptr;
    API_CATCH
}

void hfb200_pool_destroy(hfb200_pool* pool) { delete pool; }

// ---- HAL-level operators ------------------------------------------------------------------------
struct DevBuf {
    Dev& d; uint32_t* p;
    DevBuf(Dev& dev, size_t words) : d(dev), p((uint32_t*)dev.alloc(words * 4)) {}
    ~DevBuf() { d.free(p); }
};

const char* hfb200_op_interpolate_ntt(hfb200_ctx* ctx, uint32_t* io, size_t count, size_t n, int zk_shift) {
    API_TRY
    if (!ctx || !io) throw Err("op_interpolate_ntt: NULL argument");
    ctx->p.bind();
    Dev& d = ctx->p.dev;
    const int lg = ilog2(n);
    if ((1ull << lg) != n || lg > 24 || count == 0) throw Err("op_interpolate_ntt: bad size");
    DevBuf b(d, count * n);
    d.h2d(b.p, io, count * n * 4);
    ctx->p.ntt.interpolate(b.p, n, b.p, n, (uint32_t)count, lg, zk_shift != 0);
    d.d2h(io, b.p, count * n * 4);
    d.sync();
    API_CATCH
}
const char* hfb200_op_expand_ntt(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, size_t n_in, uint32_t expand_bits) {
    API_TRY
    if (!ctx || !out || !in) throw Err("op_expand_ntt: NULL argument");
    ctx->p.bind();
    Dev& d = ctx->p.dev;
    const int lg = ilog2(n_in);
    if ((1ull << lg) != n_in || lg + (int)expand_bits > 24 || (expand_bits != 0 && expand_bits != 2) || count == 0) throw Err("op_expand_ntt: bad size");
    DevBuf bi(d, count * n_in), bo(d, (count * n_in) << expand_bits);
    d.h2d(bi.p, in, count * n_in * 4);
    ctx->p.ntt.expand_evaluate(bi.p, n_in, bo.p, n_in << expand_bits, (uint32_t)count, lg, (int)expand_bits);
    d.d2h(out, bo.p, ((count * n_in) << expand_bits) * 4);
    d.sync();
    API_CATCH
}
const char* hfb200_op_lde(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, size_t n_in) {
    API_TRY
    if (!ctx || !out || !in) throw Err("op_lde: NULL argument");
    ctx->p.bind();
    Dev& d = ctx->p.dev;
    const int lg = ilog2(n_in);
    if ((1ull << lg) != n_in || lg > 22 || count == 0) throw Err("op_lde: bad size");
    DevBuf bi(d, count * n_in), bs(d, count * n_in), bo(d, count * n_in * 4);
    d.h2d(bi.p, in, count * n_in * 4);
    ctx->p.ntt.lde(bi.p, n_in, bo.p, n_in * 4, bs.p, (uint32_t)count, lg);
    d.d2h(out, bo.p, count * n_in * 16);
    d.sync();
    API_CATCH
}
const char* hfb200_op_merkle(hfb200_ctx* ctx, const uint32_t* matrix, size_t rows, size_t cols, uint32_t* nodes_out) {
    API_TRY
    if (!ctx || !matrix || !nodes_out) throw Err("op_merkle: NULL argument");
    ctx->p.bind();
    Dev& d = ctx->p.dev;
    if ((1ull << ilog2(rows)) != rows || rows < 2 || cols == 0) throw Err("op_merkle: rows must be a power of two >= 2");
    DevBuf bm(d, rows * cols), bn(d, 2 * rows * 8);
    d.h2d(bm.p, matrix, rows * cols * 4);
    d.zero(bn.p, 8 * 4);
    ctx->p.merkle.build(bm.p, rows, (uint32_t)rows, (uint32_t)cols, bn.p);
    d.d2h(nodes_out, bn.p, 2 * rows * 8 * 4);
    d.sync();
    API_CATCH
}
const char* hfb200_op_poseidon2(hfb200_ctx* ctx, uint32_t* states, size_t n) {
    API_TRY
    if (!ctx || (!states && n)) throw Err("op_poseidon2: NULL argument");
    ctx->p.bind();
    Dev& d = ctx->p.dev;
    DevBuf b(d, n * 24);
    d.h2d(b.p, states, n * 24 * 4);
    ctx->p.merkle.permute(b.p, (uint32_t)n);
    d.d2h(states, b.p, n * 24 * 4);
    d.sync();
    API_CATCH
}
#if P2_PHASE_PROBE && !defined(HFB200_EMU)
// Phase probe builds only (tools/p2_phase_probe.py): out[0..n) = the cycle sums of g_p2_probe, out[n] = permutations
// sampled, n = 4 + 3 P2TC_BLOCKS phases written to *n_phases.  Clears the counters.
const char* hfb200_p2_probe_read(hfb200_ctx* ctx, unsigned long long* out, uint32_t* n_phases) {
    API_TRY
    if (!ctx || !out || !n_phases) throw Err("p2_probe_read: NULL argument");
    ctx->p.bind();
    ctx->p.dev.sync();
    CUDA_CHECK(cudaMemcpyFromSymbol(out, hf::g_p2_probe, sizeof(unsigned long long) * (hf::P2_PROBE_N + 1)));
    static const unsigned long long zero[hf::P2_PROBE_N + 1] = {};
    CUDA_CHECK(cudaMemcpyToSymbol(hf::g_p2_probe, zero, sizeof zero));
    *n_phases = hf::P2_PROBE_N;
    API_CATCH
}
#endif
const char* hfb200_op_fri_fold(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t n, const uint32_t* mix4) {
    API_TRY
    if (!ctx || !out || !in || !mix4) throw Err("op_fri_fold: NULL argument");
    ctx->p.bind();
    Dev& d = ctx->p.dev;
    if (n < 16 || (n & 15)) throw Err("op_fri_fold: n must be a multiple of 16");
    DevBuf bi(d, 4 * n), bo(d, 4 * n / 16);
    d.h2d(bi.p, in, 4 * n * 4);
    FriFoldArgs fa{};
    fa.in = bi.p; fa.out = bo.p; fa.n = (uint32_t)n;
    const E4 fm = e4(mix4[0], mix4[1], mix4[2], mix4[3]);
    { E4 cur = e4_one(); for (int i = 0; i < 16; i++) { fa.mixpow[i] = cur; cur = e4_mul(cur, fm); } }
    d.launch<FriFoldKernel, 256, 1>((unsigned)((n / 16 + 255) / 256), 1, 256, 0, fa);
    d.d2h(out, bo.p, (4 * n / 16) * 4);
    d.sync();
    API_CATCH
}

// ---- device HAL: risc0-zkp `Hal` operators on caller device buffers ------------------------------------------------------
// Every entry checks its sizes, then its pointers, before anything is queued; the work goes on the context's stream and the
// call returns without waiting for it.
} // extern "C"
static void hal_ptr(const hfb200_ctx* ctx, const void* p, const char* fn, const char* what) {
    if (!p) throw Err(std::string(fn) + ": " + what + " is NULL");
#ifndef HFB200_EMU
    cudaPointerAttributes a{};
    const cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) cudaGetLastError();  // not a pointer the driver knows: clear the error, refuse below
    if (e != cudaSuccess || a.type != cudaMemoryTypeDevice || a.device != ctx->p.device_id)
        throw Err(std::string(fn) + ": " + what + " is not device memory of device " + std::to_string(ctx->p.device_id));
#else
    (void)ctx;
#endif
}
static void hal_aligned16(const void* p, const char* fn, const char* what) {
    if (reinterpret_cast<uintptr_t>(p) & 15u) throw Err(std::string(fn) + ": " + what + " must be 16-byte aligned");
}
// log2 of a power of two n in [lo, 2^max_lg]
static int hal_po2(size_t n, size_t lo, int max_lg, const char* fn, const char* what) {
    if (n < lo || (n & (n - 1)) || ilog2(n) > max_lg)
        throw Err(std::string(fn) + ": " + what + " = " + std::to_string(n) + " is not a power of two in [" + std::to_string(lo) + ", 2^" + std::to_string(max_lg) + "]");
    return ilog2(n);
}
static void hal_limit(size_t v, size_t lo, size_t hi, const char* fn, const char* what) {
    if (v < lo || v > hi) throw Err(std::string(fn) + ": " + what + " = " + std::to_string(v) + " outside [" + std::to_string(lo) + ", " + std::to_string(hi) + "]");
}
static hfb200_ctx* hal_ctx(hfb200_ctx* ctx, const char* fn) {
    if (!ctx) throw Err(std::string(fn) + ": NULL ctx");
    ctx->p.bind();
    return ctx;
}
// context-owned scratch: grows when a larger request comes (after the stream's earlier users are done), never shrinks
static void* hal_scratch(hfb200_ctx* ctx, size_t bytes) {
    if (bytes > ctx->hal_scratch_cap) {
        if (ctx->hal_scratch) { ctx->p.sync(); ctx->p.dev.free(ctx->hal_scratch); ctx->hal_scratch = nullptr; ctx->hal_scratch_cap = 0; }
        bytes = std::max<size_t>(bytes, (size_t)1 << 20);
        ctx->hal_scratch = ctx->p.dev.alloc(bytes);
        ctx->hal_scratch_cap = bytes;
    }
    return ctx->hal_scratch;
}
static unsigned hal_blocks(uint64_t items) { return (unsigned)((items + HAL_T - 1) / HAL_T); }
static constexpr size_t HAL_MAX_ELEMS = (size_t)1 << 34;  // words per buffer (64 GB)
static E4 hal_e4(const uint32_t* h) { for (int k = 0; k < 4; k++) if (h[k] >= P) throw Err("Fp4 argument holds a non-canonical field element"); return e4(h[0], h[1], h[2], h[3]); }
extern "C" {

const char* hfb200_hal_stream(hfb200_ctx* ctx, void** stream, int* device) {
    API_TRY
    static const char* fn = "hfb200_hal_stream";
    hal_ctx(ctx, fn);
    if (!stream) throw Err(std::string(fn) + ": stream is NULL");
    *stream = (void*)ctx->p.dev.stream;
    if (device) *device = ctx->p.device_id;
    API_CATCH
}
const char* hfb200_hal_sync(hfb200_ctx* ctx) {
    API_TRY
    hal_ctx(ctx, "hfb200_hal_sync")->p.sync();
    API_CATCH
}
uint64_t hfb200_hal_host_syncs(const hfb200_ctx* ctx) { return ctx ? ctx->p.host_syncs : 0; }

const char* hfb200_hal_batch_interpolate_ntt(hfb200_ctx* ctx, uint32_t* io, size_t count, size_t n) {
    API_TRY
    static const char* fn = "hfb200_hal_batch_interpolate_ntt";
    hal_ctx(ctx, fn);
    const int lg = hal_po2(n, 2, 24, fn, "n");
    hal_limit(count, 1, HAL_MAX_ELEMS >> lg, fn, "count");
    hal_ptr(ctx, io, fn, "io");
    ctx->p.ntt.interpolate(io, n, io, n, (uint32_t)count, lg, false);
    API_CATCH
}
const char* hfb200_hal_zk_shift(hfb200_ctx* ctx, uint32_t* io, size_t count, size_t n) {
    API_TRY
    static const char* fn = "hfb200_hal_zk_shift";
    hal_ctx(ctx, fn);
    const int lg = hal_po2(n, 1, 24, fn, "n");
    hal_limit(count, 1, HAL_MAX_ELEMS >> lg, fn, "count");
    hal_ptr(ctx, io, fn, "io");
    const RootTables& rt = ctx->p.ntt.rt;
    ctx->p.dev.launch<HalZkShiftKernel, HAL_T, 1>(hal_blocks((uint64_t)count << lg), 1, HAL_T, 0, io, (uint64_t)count << lg, (uint32_t)lg, rt.p3_lo, rt.p3_hi);
    API_CATCH
}
const char* hfb200_hal_batch_expand_into_evaluate_ntt(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, size_t n_in, uint32_t expand_bits) {
    API_TRY
    static const char* fn = "hfb200_hal_batch_expand_into_evaluate_ntt";
    hal_ctx(ctx, fn);
    if (expand_bits != 0 && expand_bits != 2) throw Err(std::string(fn) + ": expand_bits = " + std::to_string(expand_bits) + " is not supported (0 or 2)");
    const int lg = hal_po2(n_in, 2, 24 - (int)expand_bits, fn, "n_in");
    hal_limit(count, 1, HAL_MAX_ELEMS >> (lg + expand_bits), fn, "count");
    hal_ptr(ctx, out, fn, "out");
    hal_ptr(ctx, in, fn, "in");
    const uintptr_t o0 = (uintptr_t)out, o1 = o0 + ((count * n_in) << expand_bits) * 4, i0 = (uintptr_t)in, i1 = i0 + count * n_in * 4;
    if (o0 < i1 && i0 < o1) throw Err(std::string(fn) + ": out and in overlap");
    ctx->p.ntt.expand_evaluate(in, n_in, out, (uint64_t)n_in << expand_bits, (uint32_t)count, lg, (int)expand_bits);
    API_CATCH
}
const char* hfb200_hal_batch_bit_reverse(hfb200_ctx* ctx, uint32_t* io, size_t count, size_t n) {
    API_TRY
    static const char* fn = "hfb200_hal_batch_bit_reverse";
    hal_ctx(ctx, fn);
    const int lg = hal_po2(n, 1, 31, fn, "n");
    hal_limit(count, 1, HAL_MAX_ELEMS >> lg, fn, "count");
    hal_ptr(ctx, io, fn, "io");
    ctx->p.dev.launch<HalBitRevKernel, HAL_T, 1>(hal_blocks((uint64_t)count << lg), 1, HAL_T, 0, io, (uint64_t)count << lg, (uint32_t)lg);
    API_CATCH
}
const char* hfb200_hal_hash_rows(hfb200_ctx* ctx, uint32_t* digests, const uint32_t* matrix, size_t rows, size_t cols) {
    API_TRY
    static const char* fn = "hfb200_hal_hash_rows";
    hal_ctx(ctx, fn);
    hal_limit(rows, 1, 0xFFFFFFFFull, fn, "rows");
    hal_limit(cols, 1, HAL_MAX_ELEMS / rows, fn, "cols");
    hal_ptr(ctx, digests, fn, "digests");
    hal_ptr(ctx, matrix, fn, "matrix");
    hal_aligned16(digests, fn, "digests");
    ctx->p.merkle.hash_rows(HASH_POSEIDON2, matrix, rows, (uint32_t)rows, (uint32_t)cols, digests);
    API_CATCH
}
const char* hfb200_hal_hash_fold(hfb200_ctx* ctx, uint32_t* io, size_t input_size, size_t output_size) {
    API_TRY
    static const char* fn = "hfb200_hal_hash_fold";
    hal_ctx(ctx, fn);
    hal_limit(output_size, 1, 0x7FFFFFFFull, fn, "output_size");
    if (input_size != 2 * output_size) throw Err(std::string(fn) + ": input_size must be 2 * output_size");
    hal_ptr(ctx, io, fn, "io");
    hal_aligned16(io, fn, "io");
    ctx->p.merkle.fold_level(HASH_POSEIDON2, io, (uint32_t)output_size);
    API_CATCH
}
const char* hfb200_hal_sha_rows(hfb200_ctx* ctx, uint32_t* digests, const uint32_t* matrix, size_t rows, size_t cols) {
    API_TRY
    static const char* fn = "hfb200_hal_sha_rows";
    hal_ctx(ctx, fn);
    hal_limit(rows, 1, 0xFFFFFFFFull, fn, "rows");
    hal_limit(cols, 1, HAL_MAX_ELEMS / rows, fn, "cols");
    hal_ptr(ctx, digests, fn, "digests");
    hal_ptr(ctx, matrix, fn, "matrix");
    hal_aligned16(digests, fn, "digests");
    ctx->p.merkle.hash_rows(HASH_SHA256, matrix, rows, (uint32_t)rows, (uint32_t)cols, digests);
    API_CATCH
}
const char* hfb200_hal_sha_fold(hfb200_ctx* ctx, uint32_t* io, size_t input_size, size_t output_size) {
    API_TRY
    static const char* fn = "hfb200_hal_sha_fold";
    hal_ctx(ctx, fn);
    hal_limit(output_size, 1, 0x7FFFFFFFull, fn, "output_size");
    if (input_size != 2 * output_size) throw Err(std::string(fn) + ": input_size must be 2 * output_size");
    hal_ptr(ctx, io, fn, "io");
    hal_aligned16(io, fn, "io");
    ctx->p.merkle.fold_level(HASH_SHA256, io, (uint32_t)output_size);
    API_CATCH
}
const char* hfb200_hal_batch_evaluate_any(hfb200_ctx* ctx, const uint32_t* coeffs, size_t poly_count, size_t n, const uint32_t* which,
                                          const uint32_t* xs, uint32_t* out, size_t count) {
    API_TRY
    static const char* fn = "hfb200_hal_batch_evaluate_any";
    hal_ctx(ctx, fn);
    hal_limit(n, 1, HAL_MAX_ELEMS, fn, "n");
    hal_limit(poly_count, 1, HAL_MAX_ELEMS / n, fn, "poly_count");
    hal_limit(count, 1, (size_t)65535 * HAL_EV_PTS, fn, "count");
    hal_ptr(ctx, coeffs, fn, "coeffs");
    hal_ptr(ctx, which, fn, "which");
    hal_ptr(ctx, xs, fn, "xs");
    hal_ptr(ctx, out, fn, "out");
    const uint32_t nblk = (uint32_t)((n + HAL_EV_RPB - 1) / HAL_EV_RPB);
    E4* partial = (E4*)hal_scratch(ctx, (size_t)count * nblk * sizeof(E4));
    Dev& d = ctx->p.dev;
    d.launch<HalEvalKernel, HAL_T, 1>(nblk, (unsigned)((count + HAL_EV_PTS - 1) / HAL_EV_PTS), HAL_T, (size_t)HAL_EV_PTS * HAL_T * sizeof(E4),
                                      coeffs, (uint64_t)n, which, xs, (uint64_t)count, partial);
    d.launch<HalEvalReduceKernel, HAL_T, 1>(hal_blocks(count), 1, HAL_T, 0, (const E4*)partial, nblk, (uint64_t)count, out);
    API_CATCH
}
const char* hfb200_hal_mix_poly_coeffs(hfb200_ctx* ctx, uint32_t* out, const uint32_t* mix_start, const uint32_t* mix, const uint32_t* in,
                                       const uint32_t* combo_of_col, size_t n_cols, size_t n, size_t n_combos) {
    API_TRY
    static const char* fn = "hfb200_hal_mix_poly_coeffs";
    hal_ctx(ctx, fn);
    hal_limit(n, 1, HAL_MAX_ELEMS, fn, "n");
    hal_limit(n_cols, 1, 8192, fn, "n_cols");
    hal_limit(n_combos, 1, HAL_MAX_ELEMS / 4 / n, fn, "n_combos");
    if (!mix_start || !mix) throw Err(std::string(fn) + ": mix_start / mix is NULL");
    const E4 ms = hal_e4(mix_start), m = hal_e4(mix);
    hal_ptr(ctx, out, fn, "out");
    hal_ptr(ctx, in, fn, "in");
    hal_ptr(ctx, combo_of_col, fn, "combo_of_col");
    E4* w = (E4*)hal_scratch(ctx, n_cols * sizeof(E4));
    Dev& d = ctx->p.dev;
    d.launch<HalMixPowKernel, HAL_T, 1>(hal_blocks(n_cols), 1, HAL_T, 0, w, (uint32_t)n_cols, ms, m);
    d.launch<HalMixPolyKernel, HAL_T, 1>(hal_blocks(n), 1, HAL_T, n_cols * (sizeof(E4) + 4), out, (const E4*)w, in, combo_of_col, (uint32_t)n_cols, (uint64_t)n);
    API_CATCH
}
} // extern "C"
template <class Op>
static void hal_scan(hfb200_ctx* ctx, const HalScanArgs& a) {
    using T = typename Op::T;
    const uint32_t nblk = (uint32_t)((a.n + HAL_SC_RPB - 1) / HAL_SC_RPB);
    T* partial = (T*)hal_scratch(ctx, (size_t)nblk * sizeof(T));
    Dev& d = ctx->p.dev;
    const size_t sm = 2 * HAL_T * sizeof(T);
    d.launch<HalScanKernel<Op>, HAL_T, 1>(nblk, 1, HAL_T, sm, a, partial, 0);
    d.launch<HalScanOffsetsKernel<Op>, HAL_T, 1>(1, 1, HAL_T, sm, partial, nblk);
    d.launch<HalScanKernel<Op>, HAL_T, 1>(nblk, 1, HAL_T, sm, a, partial, 1);
}
extern "C" {
const char* hfb200_hal_poly_divide(hfb200_ctx* ctx, uint32_t* poly, size_t n, const uint32_t* z, uint32_t* remainder_out) {
    API_TRY
    static const char* fn = "hfb200_hal_poly_divide";
    hal_ctx(ctx, fn);
    hal_limit(n, 1, (size_t)1 << 30, fn, "n");
    if (!z) throw Err(std::string(fn) + ": z is NULL");
    const E4 zz = hal_e4(z);
    hal_ptr(ctx, poly, fn, "poly");
    hal_ptr(ctx, remainder_out, fn, "remainder_out");
    HalScanArgs a{poly, (uint64_t)n, zz, remainder_out};
    hal_scan<DivScan>(ctx, a);
    API_CATCH
}
const char* hfb200_hal_prefix_products(hfb200_ctx* ctx, uint32_t* io, size_t n) {
    API_TRY
    static const char* fn = "hfb200_hal_prefix_products";
    hal_ctx(ctx, fn);
    hal_limit(n, 1, (size_t)1 << 30, fn, "n");
    hal_ptr(ctx, io, fn, "io");
    HalScanArgs a{io, (uint64_t)n, e4_zero(), nullptr};
    hal_scan<ProdScan>(ctx, a);
    API_CATCH
}
const char* hfb200_hal_eltwise_add_elem(hfb200_ctx* ctx, uint32_t* out, const uint32_t* x, const uint32_t* y, size_t count) {
    API_TRY
    static const char* fn = "hfb200_hal_eltwise_add_elem";
    hal_ctx(ctx, fn);
    hal_limit(count, 1, HAL_MAX_ELEMS, fn, "count");
    hal_ptr(ctx, out, fn, "out"); hal_ptr(ctx, x, fn, "x"); hal_ptr(ctx, y, fn, "y");
    ctx->p.dev.launch<HalAddElemKernel, HAL_T, 1>(hal_blocks(count), 1, HAL_T, 0, out, x, y, (uint64_t)count);
    API_CATCH
}
const char* hfb200_hal_eltwise_sum_extelem(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count, size_t to_add) {
    API_TRY
    static const char* fn = "hfb200_hal_eltwise_sum_extelem";
    hal_ctx(ctx, fn);
    hal_limit(count, 1, HAL_MAX_ELEMS / 4, fn, "count");
    hal_limit(to_add, 1, HAL_MAX_ELEMS / 4 / count, fn, "to_add");
    hal_ptr(ctx, out, fn, "out"); hal_ptr(ctx, in, fn, "in");
    ctx->p.dev.launch<HalSumExtKernel, HAL_T, 1>(hal_blocks(count), 1, HAL_T, 0, out, in, (uint64_t)count, (uint32_t)to_add);
    API_CATCH
}
const char* hfb200_hal_eltwise_copy_elem(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t count) {
    API_TRY
    static const char* fn = "hfb200_hal_eltwise_copy_elem";
    hal_ctx(ctx, fn);
    hal_limit(count, 1, HAL_MAX_ELEMS, fn, "count");
    hal_ptr(ctx, out, fn, "out"); hal_ptr(ctx, in, fn, "in");
    ctx->p.dev.d2d(out, in, count * 4);
    API_CATCH
}
const char* hfb200_hal_eltwise_zeroize_elem(hfb200_ctx* ctx, uint32_t* io, size_t count) {
    API_TRY
    static const char* fn = "hfb200_hal_eltwise_zeroize_elem";
    hal_ctx(ctx, fn);
    hal_limit(count, 1, HAL_MAX_ELEMS, fn, "count");
    hal_ptr(ctx, io, fn, "io");
    ctx->p.dev.zero(io, count * 4);
    API_CATCH
}
const char* hfb200_hal_gather_sample(hfb200_ctx* ctx, uint32_t* dst, const uint32_t* src, size_t idx, size_t size, size_t stride) {
    API_TRY
    static const char* fn = "hfb200_hal_gather_sample";
    hal_ctx(ctx, fn);
    hal_limit(size, 1, HAL_MAX_ELEMS, fn, "size");
    hal_limit(stride, 1, HAL_MAX_ELEMS, fn, "stride");
    hal_limit(size - 1, 0, HAL_MAX_ELEMS / stride, fn, "size - 1 (times stride)");
    hal_limit(idx, 0, HAL_MAX_ELEMS - (size - 1) * stride, fn, "idx");
    hal_ptr(ctx, dst, fn, "dst"); hal_ptr(ctx, src, fn, "src");
    ctx->p.dev.launch<HalGatherKernel, HAL_T, 1>(hal_blocks(size), 1, HAL_T, 0, dst, src, (uint64_t)idx, (uint64_t)size, (uint64_t)stride);
    API_CATCH
}
const char* hfb200_hal_scatter(hfb200_ctx* ctx, uint32_t* into, const uint32_t* index, const uint32_t* offsets, const uint32_t* values, size_t count) {
    API_TRY
    static const char* fn = "hfb200_hal_scatter";
    hal_ctx(ctx, fn);
    hal_limit(count, 1, HAL_MAX_ELEMS, fn, "count");
    hal_ptr(ctx, into, fn, "into"); hal_ptr(ctx, index, fn, "index"); hal_ptr(ctx, offsets, fn, "offsets"); hal_ptr(ctx, values, fn, "values");
    ctx->p.dev.launch<HalScatterKernel, HAL_T, 1>(hal_blocks(count), 1, HAL_T, 0, into, index, offsets, values, (uint64_t)count);
    API_CATCH
}
const char* hfb200_hal_fri_fold(hfb200_ctx* ctx, uint32_t* out, const uint32_t* in, size_t n, const uint32_t* mix) {
    API_TRY
    static const char* fn = "hfb200_hal_fri_fold";
    hal_ctx(ctx, fn);
    if (n < 16 || (n & 15) || n > HAL_MAX_ELEMS / 4) throw Err(std::string(fn) + ": n = " + std::to_string(n) + " must be a positive multiple of 16");
    hal_ptr(ctx, out, fn, "out"); hal_ptr(ctx, in, fn, "in"); hal_ptr(ctx, mix, fn, "mix");
    ctx->p.dev.launch<HalFriFoldKernel, HAL_T, 1>(hal_blocks(n / 16), 1, HAL_T, 16 * sizeof(E4), out, in, (uint64_t)n, mix);
    API_CATCH
}

const char* hfb200_bench_lde(hfb200_ctx* ctx, uint32_t po2, uint32_t count, uint32_t iters, float* ms_avg) {
    API_TRY
    if (!ctx || !ms_avg) throw Err("bench_lde: NULL argument");
    Prover& p = ctx->p;
    p.bind();
    p.layout(po2);
    if (count == 0 || count > p.cir.cd.w_data) throw Err("bench_lde: count must be in [1, w_data]");
    if (!p.have_trace) throw Err("bench_lde: call hfb200_witgen_synth first");
    const size_t N = (size_t)1 << po2;
    Timer t; t.init(p.dev.stream);
    p.ntt.lde(p.tr[GROUP_DATA], N, p.ev[GROUP_DATA], 4 * N, p.scratch, count, (int)po2);  // warm-up
    t.start();
    for (uint32_t i = 0; i < iters; i++) p.ntt.lde(p.tr[GROUP_DATA], N, p.ev[GROUP_DATA], 4 * N, p.scratch, count, (int)po2);
    t.stop();
    *ms_avg = t.ms() / (iters ? iters : 1);
    t.destroy();
    API_CATCH
}
const char* hfb200_bench_merkle(hfb200_ctx* ctx, uint32_t po2, uint32_t count, uint32_t iters, float* ms_avg) {
    API_TRY
    if (!ctx || !ms_avg) throw Err("bench_merkle: NULL argument");
    Prover& p = ctx->p;
    p.bind();
    p.layout(po2);
    if (count == 0 || count > p.cir.cd.w_data) throw Err("bench_merkle: count must be in [1, w_data]");
    const size_t D = (size_t)4 << po2;
    Timer t; t.init(p.dev.stream);
    p.merkle.build(p.ev[GROUP_DATA], D, (uint32_t)D, count, p.nodes[GROUP_DATA]);
    t.start();
    for (uint32_t i = 0; i < iters; i++) p.merkle.build(p.ev[GROUP_DATA], D, (uint32_t)D, count, p.nodes[GROUP_DATA]);
    t.stop();
    *ms_avg = t.ms() / (iters ? iters : 1);
    t.destroy();
    API_CATCH
}

const char* hfb200_verify_segment(const hfb200_circuit_desc* c, const hfb200_circuit_ir* ir, const uint32_t* seal, size_t seal_words,
                                  const uint32_t* code_root, uint32_t* po2_out) {
    return hfb200_verify_segment_suite(c, ir, seal, seal_words, code_root, po2_out, HASH_POSEIDON2);
}
const char* hfb200_verify_segment_suite(const hfb200_circuit_desc* c, const hfb200_circuit_ir* ir, const uint32_t* seal, size_t seal_words,
                                        const uint32_t* code_root, uint32_t* po2_out, int suite) {
    API_TRY
    if ((c == nullptr) == (ir == nullptr)) throw Err("hfb200_verify_segment: pass exactly one of circuit / ir");
    if (!seal || !code_root) throw Err("hfb200_verify_segment: NULL seal or code_root");
    if (!hash_suite_valid(suite)) throw Err("hfb200_verify_segment: suite must be HFB200_HASH_POSEIDON2 (0) or HFB200_HASH_SHA256 (1)");
    VCircuit vc;
    if (c) vc.init_builtin(c->w_code, c->w_data, c->w_accum);
    else vc.init_ir(ir->w_code, ir->w_data, ir->w_accum, ir->n_mix, reinterpret_cast<const IrTap*>(ir->taps), ir->n_taps,
                    reinterpret_cast<const IrStep*>(ir->steps), ir->n_steps, ir->ret, ir->info);
    verify_segment(vc, seal, seal_words, code_root, po2_out, suite);
    API_CATCH
}
// n seals at once on up to `threads` host threads (0 = one per hardware thread): what `receipt.verify` does over the segment
// receipts of a composite receipt; the seals are independent, so this is plain fan-out.  The FIRST failing seal (lowest index)
// is reported, prefixed with its index; `first_bad` receives that index (or n when all verify).
const char* hfb200_verify_segments(const hfb200_circuit_desc* c, const hfb200_circuit_ir* ir, const uint32_t* const* seals, const size_t* seal_words,
                                   size_t n, const uint32_t* code_roots, uint32_t* po2_out, unsigned threads, size_t* first_bad) {
    return hfb200_verify_segments_suite(c, ir, seals, seal_words, n, code_roots, po2_out, threads, first_bad, HASH_POSEIDON2);
}
const char* hfb200_verify_segments_suite(const hfb200_circuit_desc* c, const hfb200_circuit_ir* ir, const uint32_t* const* seals, const size_t* seal_words,
                                         size_t n, const uint32_t* code_roots, uint32_t* po2_out, unsigned threads, size_t* first_bad, int suite) {
    API_TRY
    if ((c == nullptr) == (ir == nullptr)) throw Err("hfb200_verify_segments: pass exactly one of circuit / ir");
    if (n && (!seals || !seal_words || !code_roots)) throw Err("hfb200_verify_segments: NULL argument");
    if (!hash_suite_valid(suite)) throw Err("hfb200_verify_segments: suite must be HFB200_HASH_POSEIDON2 (0) or HFB200_HASH_SHA256 (1)");
    if (first_bad) *first_bad = n;
    VCircuit vc;
    if (c) vc.init_builtin(c->w_code, c->w_data, c->w_accum);
    else vc.init_ir(ir->w_code, ir->w_data, ir->w_accum, ir->n_mix, reinterpret_cast<const IrTap*>(ir->taps), ir->n_taps,
                    reinterpret_cast<const IrStep*>(ir->steps), ir->n_steps, ir->ret, ir->info);
    p2_host_consts();
    unsigned nt = threads ? threads : std::thread::hardware_concurrency();
    if (nt == 0) nt = 1;
    if (nt > n) nt = (unsigned)n;
    std::vector<std::string> errs(n);
    std::vector<char> bad(n, 0);
    std::atomic<size_t> next{0};
    auto work = [&]() {
        for (size_t i = next.fetch_add(1); i < n; i = next.fetch_add(1)) {
            try {
                if (!seals[i]) throw Err("NULL seal");
                uint32_t po2 = 0;
                verify_segment(vc, seals[i], seal_words[i], code_roots + 8 * i, &po2, suite);
                if (po2_out) po2_out[i] = po2;
            } catch (const std::exception& e) { errs[i] = e.what(); bad[i] = 1; } catch (...) { errs[i] = "unknown error"; bad[i] = 1; }
        }
    };
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < nt; t++) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
    for (size_t i = 0; i < n; i++) if (bad[i]) { if (first_bad) *first_bad = i; throw Err("segment " + std::to_string(i) + ": " + errs[i]); }
    API_CATCH
}
// ---- receipt claims (host only) ------------------------------------------------------------------------------------------
// Upstream's `Receipt::verify(image_id)` (/root/reference/host/src/main.rs:622-624, /root/reference/verifier/src/main.rs:124-126)
// does more than check seals: it decodes each segment's ReceiptClaim from the seal's globals, chains pre/post state digests from
// the image id, and ties the journal digest to the last claim's output.  The same structure, over this library's globals layout:
//   word 0       tied to the trace by the circuit (built-in stand-in)            word 1      exit code (0 Halted, 1 SystemSplit)
//   words 8..15  pre-state digest     words 16..23  post-state digest            words 24..31  output (journal) digest, 0 if not last
// Digests are Poseidon2 digests (8 field elements, Montgomery form), so every word is a valid global.
static Digest8 digest_bytes_impl(const uint8_t* bytes, size_t n) {
    if (n >= P) throw Err("hfb200_digest_bytes: input too long");
    return host_digest_bytes(bytes, n);
}
static Digest8 digest_pair_impl(const uint32_t* a, const uint32_t* b) {
    p2_host_consts();
    uint32_t st[24] = {0};
    for (int i = 0; i < 8; i++) { st[i] = a[i]; st[8 + i] = b[i]; }
    p2_mix(st);
    Digest8 d; for (int i = 0; i < 8; i++) d.w[i] = st[i];
    return d;
}
static void claim_check_words(const uint32_t* w, const char* what) {
    for (int i = 0; i < 8; i++) if (w[i] >= P) throw Err(std::string("claim: ") + what + " digest holds a non-canonical field element");
}
const char* hfb200_digest_bytes(const uint8_t* bytes, size_t n, uint32_t* out8) {
    API_TRY
    if ((!bytes && n) || !out8) throw Err("hfb200_digest_bytes: NULL argument");
    const Digest8 d = digest_bytes_impl(bytes, n);
    std::memcpy(out8, d.w, 32);
    API_CATCH
}
const char* hfb200_digest_pair(const uint32_t* a8, const uint32_t* b8, uint32_t* out8) {
    API_TRY
    if (!a8 || !b8 || !out8) throw Err("hfb200_digest_pair: NULL argument");
    claim_check_words(a8, "left"); claim_check_words(b8, "right");
    const Digest8 d = digest_pair_impl(a8, b8);
    std::memcpy(out8, d.w, 32);
    API_CATCH
}
const char* hfb200_claim_encode(const hfb200_claim* c, uint32_t* globals) {
    API_TRY
    if (!c || !globals) throw Err("hfb200_claim_encode: NULL argument");
    if (c->exit_code > 1) throw Err("hfb200_claim_encode: exit_code must be HFB200_EXIT_HALTED or HFB200_EXIT_SYSTEM_SPLIT");
    claim_check_words(c->pre, "pre"); claim_check_words(c->post, "post"); claim_check_words(c->output, "output");
    globals[1] = c->exit_code ? ONE : 0u;
    std::memcpy(globals + 8, c->pre, 32); std::memcpy(globals + 16, c->post, 32); std::memcpy(globals + 24, c->output, 32);
    API_CATCH
}
const char* hfb200_claim_decode(const uint32_t* seal, size_t seal_words, hfb200_claim* out) {
    API_TRY
    if (!seal || !out) throw Err("hfb200_claim_decode: NULL argument");
    if (seal_words < N_GLOBAL + 1) throw Err("hfb200_claim_decode: seal truncated");
    if (seal[1] != 0u && seal[1] != ONE) throw Err("claim: exit code word is neither Halted nor SystemSplit");
    out->exit_code = seal[1] == ONE ? 1u : 0u;
    std::memcpy(out->pre, seal + 8, 32); std::memcpy(out->post, seal + 16, 32); std::memcpy(out->output, seal + 24, 32);
    claim_check_words(out->pre, "pre"); claim_check_words(out->post, "post"); claim_check_words(out->output, "output");
    API_CATCH
}
const char* hfb200_claim_next_state(const uint32_t* pre8, uint32_t index, uint32_t po2, uint32_t* post8) {
    API_TRY
    if (!pre8 || !post8) throw Err("hfb200_claim_next_state: NULL argument");
    claim_check_words(pre8, "pre");
    // executor stand-in (SURVEY.md section 8f N1 is not built): upstream's post-state is the digest of the memory image after the
    // segment; here it is a hash chain over (segment index, po2), so that order and count of the segments are bound
    const uint8_t tag[8] = {(uint8_t)index, (uint8_t)(index >> 8), (uint8_t)(index >> 16), (uint8_t)(index >> 24), (uint8_t)po2, 's', 'e', 'g'};
    const Digest8 t = digest_bytes_impl(tag, sizeof tag);
    const Digest8 d = digest_pair_impl(pre8, t.w);
    std::memcpy(post8, d.w, 32);
    API_CATCH
}
const char* hfb200_verify_claims(const uint32_t* const* seals, const size_t* seal_words, size_t n, const uint32_t* image_id8,
                                 const uint8_t* journal, size_t journal_len) {
    API_TRY
    if (!seals || !seal_words || !image_id8 || (!journal && journal_len)) throw Err("hfb200_verify_claims: NULL argument");
    if (n == 0) throw Err("verify: composite receipt without segments");
    const Digest8 jd = digest_bytes_impl(journal, journal_len);
    uint32_t expect_pre[8];
    std::memcpy(expect_pre, image_id8, 32);
    const uint32_t zero[8] = {0};
    for (size_t i = 0; i < n; i++) {
        hfb200_claim c;
        if (const char* e = hfb200_claim_decode(seals[i], seal_words[i], &c)) { const std::string m(e); hfb200_free_error(e); throw Err("segment " + std::to_string(i) + ": " + m); }
        if (std::memcmp(c.pre, expect_pre, 32) != 0)
            throw Err(i == 0 ? std::string("verify: segment 0 does not start from the image id (wrong program, or not the first segment)")
                             : "verify: segment " + std::to_string(i) + " does not continue from the post-state of segment " + std::to_string(i - 1));
        const bool last = i + 1 == n;
        if (!last) {
            if (c.exit_code != 1u) throw Err("verify: segment " + std::to_string(i) + " halts before the last segment");
            if (std::memcmp(c.output, zero, 32) != 0) throw Err("verify: segment " + std::to_string(i) + " carries an output digest but is not the last segment");
        } else {
            if (c.exit_code != 0u) throw Err("verify: the last segment does not halt (receipt truncated)");
            if (std::memcmp(c.output, jd.w, 32) != 0) throw Err("verify: journal digest does not match the claim of the last segment (journal altered)");
        }
        std::memcpy(expect_pre, c.post, 32);
    }
    API_CATCH
}

// ---- the hash suites' host primitives (the ones the transcript and the verifier use) ----------------------------------
static void suite_arg(int suite, const char* fn) {
    if (!hash_suite_valid(suite)) throw Err(std::string(fn) + ": suite must be HFB200_HASH_POSEIDON2 (0) or HFB200_HASH_SHA256 (1)");
}
const char* hfb200_sha256(const uint8_t* bytes, size_t n, uint32_t* out8) {
    API_TRY
    if ((!bytes && n) || !out8) throw Err("hfb200_sha256: NULL argument");
    sha256_bytes(bytes, n, out8);
    API_CATCH
}
const char* hfb200_hash_elems(int suite, const uint32_t* elems, size_t n, uint32_t* out8) {
    API_TRY
    suite_arg(suite, "hfb200_hash_elems");
    if ((!elems && n) || !out8) throw Err("hfb200_hash_elems: NULL argument");
    const Digest8 d = suite_hash_elems(suite, elems, n);
    std::memcpy(out8, d.w, 32);
    API_CATCH
}
const char* hfb200_hash_pair(int suite, const uint32_t* a8, const uint32_t* b8, uint32_t* out8) {
    API_TRY
    suite_arg(suite, "hfb200_hash_pair");
    if (!a8 || !b8 || !out8) throw Err("hfb200_hash_pair: NULL argument");
    Digest8 a, b;
    std::memcpy(a.w, a8, 32); std::memcpy(b.w, b8, 32);
    const Digest8 d = suite_hash_pair(suite, a, b);
    std::memcpy(out8, d.w, 32);
    API_CATCH
}
const char* hfb200_rng_script(int suite, const uint32_t* ops, size_t n_ops, const uint32_t* digests, size_t n_digests, uint32_t* out, size_t cap,
                              size_t* n_out) {
    API_TRY
    suite_arg(suite, "hfb200_rng_script");
    if ((!ops && n_ops) || (!digests && n_digests) || (!out && cap) || !n_out) throw Err("hfb200_rng_script: NULL argument");
    HostRng rng(suite);
    size_t d = 0, o = 0;
    for (size_t i = 0; i < n_ops; i++) {
        const uint32_t op = ops[2 * i], arg = ops[2 * i + 1];
        if (op > 2) throw Err("hfb200_rng_script: op must be 0 (mix), 1 (random_elem) or 2 (random_bits)");
        if (op == 2 && (arg < 1 || arg > 31)) throw Err("hfb200_rng_script: random_bits takes 1..31 bits");
        if (op == 0) {
            if (d >= n_digests) throw Err("hfb200_rng_script: more mix ops than digests");
            rng.mix(digests + 8 * d++);
            continue;
        }
        if (o >= cap) throw Err("hfb200_rng_script: out buffer too small");
        out[o++] = op == 1 ? rng.random_elem() : rng.random_bits(arg);
    }
    *n_out = o;
    API_CATCH
}

const char* hfb200_control_root(hfb200_ctx* ctx, uint32_t po2, const uint32_t* code, uint32_t* root_out) {
    return control_root_impl(ctx, po2, code, root_out, 0);
}
const char* hfb200_bench_modmul(hfb200_ctx* ctx, int kind, uint32_t iters, double* products_per_s) {
    API_TRY
    if (!ctx || !products_per_s) throw Err("bench_modmul: NULL argument");
    if (kind < 0 || kind > 2) throw Err("bench_modmul: kind must be 0 (Montgomery), 1 (Shoup) or 2 (S-box chain)");
    Prover& p = ctx->p;
    p.bind();
    const unsigned blocks = (unsigned)p.dev.sm_count * 4, threads = 256;  // 8 warps per SM sub-partition
    uint32_t* out = (uint32_t*)p.dev.alloc((size_t)blocks * threads * 4);
    Timer t; t.init(p.dev.stream);
    p.dev.launch<ModmulProbeKernel, 256, 1>(blocks, 1, threads, 0, out, 12345u, iters, kind);  // warm-up (clocks)
    t.start();
    p.dev.launch<ModmulProbeKernel, 256, 1>(blocks, 1, threads, 0, out, 12345u, iters, kind);
    t.stop();
    const float ms = t.ms();
    t.destroy();
    p.dev.free(out);
    const double products = (double)blocks * threads * ModmulProbeKernel::ILP * (double)iters * (kind == 2 ? 4.0 : 1.0);
    *products_per_s = ms > 0 ? products / (ms * 1e-3) : 0.0;
    API_CATCH
}
const char* hfb200_mark(hfb200_ctx* ctx, int slot) {
    API_TRY
    if (!ctx || slot < 0 || slot > 3) throw Err("hfb200_mark: bad argument");
#ifndef HFB200_EMU
    ctx->p.bind();
    if (!ctx->marks[slot]) CUDA_CHECK(cudaEventCreate(&ctx->marks[slot]));
    CUDA_CHECK(cudaEventRecord(ctx->marks[slot], ctx->p.dev.stream));
#endif
    API_CATCH
}
const char* hfb200_mark_elapsed(hfb200_ctx* a, int slot_a, hfb200_ctx* b, int slot_b, float* ms) {
    API_TRY
    if (!a || !b || !ms || slot_a < 0 || slot_a > 3 || slot_b < 0 || slot_b > 3) throw Err("hfb200_mark_elapsed: bad argument");
    *ms = 0.f;
#ifndef HFB200_EMU
    if (!a->marks[slot_a] || !b->marks[slot_b]) throw Err("hfb200_mark_elapsed: mark not recorded");
    a->p.bind();
    CUDA_CHECK(cudaEventSynchronize(a->marks[slot_a]));
    CUDA_CHECK(cudaEventSynchronize(b->marks[slot_b]));
    CUDA_CHECK(cudaEventElapsedTime(ms, a->marks[slot_a], b->marks[slot_b]));
#endif
    API_CATCH
}

}  // extern "C"

static const char* control_root_impl(hfb200_ctx* ctx, uint32_t po2, const uint32_t* code, uint32_t* root_out, uint64_t gen) {
    API_TRY
    if (!ctx || !code || !root_out) throw Err("hfb200_control_root: NULL argument");
    Prover& p = ctx->p;
    if (p.begun) throw Err("hfb200_control_root: a segment is in flight (call hfb200_segment_finish first)");
    p.bind();
    p.layout(po2);
    p.control_cached = false; p.control_gen = 0;
    const size_t N = (size_t)1 << po2, D = 4 * N;
    const uint32_t w = p.cir.group_width(GROUP_CODE);
    p.dev.h2d(p.tr[GROUP_CODE], code, (size_t)w * N * 4);
    p.ntt.lde(p.tr[GROUP_CODE], N, p.ev[GROUP_CODE], D, p.scratch, w, (int)po2);
    p.merkle.build(p.ev[GROUP_CODE], D, (uint32_t)D, w, p.nodes[GROUP_CODE]);
    // keep the committed control group for the segments that follow with code == NULL
    p.commit_tree(Tree{p.ev[GROUP_CODE], D, (uint32_t)D, w, p.nodes[GROUP_CODE]}, "code_root", &p.control_top);
    p.proof.clear(); p.cps.clear(); p.rng = HostRng(p.hash_suite);  // commit_tree wrote into the transcript of no segment
    std::memcpy(root_out, &p.control_top[8], 32);       // heap layout: node 1 is the root
    p.control_cached = true;
    p.control_gen = gen;
    p.have_trace = false;  // the resident trace (if any) lost its code group
    API_CATCH
}
