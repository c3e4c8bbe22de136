// The segment prover: orchestration of the kernels + host-side Fiat-Shamir transcript.
// Replaces risc0-circuit-rv32im 4.0.4 `SegmentProver::prove(&Segment) -> Seal` and the risc0-zkp 3.0.4
// `Prover::{commit_group, finalize}` / `fri_prove` flow it drives (/root/reference/Cargo.lock:3087-3223,
// not vendored; entered from /root/reference/host/src/main.rs:423; SURVEY.md section 3.3 / Appendix A.7).
// Everything heavy stays on the device; the host only runs the (tiny, strictly sequential) transcript.
#pragma once
#include <chrono>
#include <map>
#include "ntt.cuh"
#include "poseidon2.cuh"
#include "circuit.cuh"
#include "deep.cuh"
#include "jit.cuh"
#include "transcript.cuh"
#ifndef HFB200_EMU
#include <nvtx3/nvToolsExt.h>  // header-only; ranges are no-ops unless a tool (nsys) injects the NVTX library
#endif

namespace hf {

// NVTX range per prover stage on the host thread that enqueues it (SURVEY.md section 5: tracing).  Stage names match hfb200_stats.
struct StageRange {
#ifndef HFB200_EMU
    explicit StageRange(const char* name) { nvtxRangePushA(name); }
    ~StageRange() { nvtxRangePop(); }
#else
    explicit StageRange(const char*) {}
#endif
};

static constexpr uint32_t QUERIES = 50, INV_RATE = 4, FRI_FOLD = 16, FRI_MIN_DEGREE = 256, CHECK_SIZE = 16;
static constexpr uint32_t MIN_PO2 = 12, MAX_PO2 = 22;  // segment sizes a context can be created for (max_po2) and can prove

struct MerkleShape {
    uint32_t rows, layers, top_layer, top_size;
    explicit MerkleShape(uint32_t r) : rows(r) {
        layers = (uint32_t)ilog2(r);
        top_layer = 0;
        for (uint32_t i = 1; i < layers; i++) { if ((1u << i) > QUERIES) break; top_layer = i; }
        top_size = 1u << top_layer;
    }
    uint32_t path_words() const { return 8 * (layers - top_layer); }
};

struct Arena {
    uint8_t* base = nullptr;
    size_t cap = 0, off = 0;
    template <typename T> T* take(size_t count) {
        size_t bytes = (count * sizeof(T) + 255) & ~(size_t)255;
        if (off + bytes > cap) throw Err("device arena exhausted (raise max_po2 at hfb200_init)");
        T* p = reinterpret_cast<T*>(base + off);
        off += bytes;
        return p;
    }
};

struct Stats {
    float ms_total = 0, ms_device = 0, ms_h2d = 0, ms_ntt_main = 0, ms_hash_main = 0, ms_accum = 0, ms_check = 0, ms_deep = 0, ms_fri = 0;
    uint64_t launches = 0, ntt_main_bytes = 0, host_syncs = 0;
};

struct Tree { uint32_t* matrix; uint64_t col_stride; uint32_t rows, cols; uint32_t* nodes; };

#ifndef HFB200_EMU
// Trace uploads of the contexts that share a device are CHAINED: a context's data copies start when the previous context's have
// landed (a stream-order wait on that context's last chunk event, no host involvement).  Copies queued together from several
// streams share the copy engine and the host's memory bandwidth, so k contexts starting together all get their trace after k
// uploads' worth of time; in FIFO order the first one has it after one and its NTTs start while the others still copy.  Matters
// where the host side is the narrow part (8 GPUs pulling from one host: ~15 GB/s per GPU).  HFB200_UPLOAD_CHAIN=0 disables it.
struct UploadChain {
    std::mutex mu;
    cudaEvent_t last = nullptr;  // last chunk event of the most recent upload queued on this device (owned by its context)
    static UploadChain& of(int device) {
        static UploadChain chains[Dev::MAX_DEVICES];
        return chains[device >= 0 && device < Dev::MAX_DEVICES ? device : 0];
    }
    static bool enabled() { static const bool on = [] { const char* e = std::getenv("HFB200_UPLOAD_CHAIN"); return !e || std::atoi(e) != 0; }(); return on; }
};
#endif

struct Prover {
    Dev dev;
    Ntt ntt;
    Merkle merkle;
    CircuitHost cir;
    GenericCircuitHost gen;  // active for data-defined circuits (hfb200_init_ir)
    JitEvalCheck jit;        // their eval_check, specialised at registration (NVRTC, sm_100a)
    uint32_t max_po2 = 0;
    char circuit_info[17] = {0};  // upstream CircuitImpl::CIRCUIT_INFO: second commit of every transcript (poseidon2.cuh)
    // HASH_POSEIDON2 or HASH_SHA256 (upstream's `hashfn`): the Merkle trees (merkle.suite) and the host transcript hash with it
    int hash_suite = HASH_POSEIDON2;
    int device_id = 0;
    Arena arena;
    bool debug_checkpoints = false;

    // ---- per-segment state ----
    uint32_t po2 = 0;
    bool have_trace = false, begun = false;
    // Control-group commitment kept across segments (opt-in: hfb200_control_root loads it, code == NULL uses it).  The
    // control columns depend on (circuit, po2) only -- upstream's verifier checks their root against a per-po2 table --
    // so their LDE and Merkle tree need not be rebuilt per segment.  Valid while the context stays at this po2 and hash suite.
    bool control_cached = false;
    uint64_t control_gen = 0;           // which hfb200_pool_load_control call the cached group came from (0: not from a pool)
    std::vector<uint32_t> control_top;  // the tree's top layers as commit_tree reads them
    uint32_t* tr[3] = {nullptr, nullptr, nullptr};  // resident traces: accum, code, data
    uint32_t* ev[3] = {nullptr, nullptr, nullptr};
    uint32_t* nodes[3] = {nullptr, nullptr, nullptr};
    uint32_t *scratch = nullptr, *check = nullptr, *ev_check = nullptr, *nodes_check = nullptr;
    uint32_t* d_mix = nullptr;
    size_t seg_mark = 0;  // arena offset after the per-po2 fixed buffers
    uint32_t globals[N_GLOBAL];
    std::vector<uint32_t> mix;
    // zero-knowledge blinding (blind.cuh): OS entropy per segment unless the caller opted into the deterministic test mode
    int blind_mode = BLIND_OS_ENTROPY;
    BlindKey blind_key{};
    BlindKey make_blind_key(uint64_t seed) const { return blind_mode == BLIND_DETERMINISTIC ? blind_key_from_seed(seed) : blind_key_from_os(seed); }
    std::vector<uint32_t> proof;
    HostRng rng;
    std::vector<std::pair<std::string, std::vector<uint32_t>>> cps;
    Stats stats;
    uint64_t launches_at_begin = 0;
    std::chrono::steady_clock::time_point t_begin;
#ifndef HFB200_EMU
    static constexpr int N_EV = 16;
    cudaEvent_t evs[N_EV] = {};
    // host->device staging of the data columns runs on its own stream in H2D_CHUNKS column slices; the LDE of a slice
    // starts as soon as its copy has landed, so the PCIe transfer hides behind the code commit and the data NTTs
#ifndef HFB200_H2D_CHUNKS
#define HFB200_H2D_CHUNKS 4
#endif
    static constexpr int H2D_CHUNKS = HFB200_H2D_CHUNKS;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t chunk_ev[H2D_CHUNKS] = {};
    cudaEvent_t copy_gate = nullptr;
#endif
    float stage_ms[8] = {0};
    // small host->device parameter uploads (mix powers, weights, descriptors) go through a pinned staging area so that the
    // copy is truly asynchronous and the source needs no stream synchronisation to stay alive
    uint8_t* stage_h = nullptr;
    size_t stage_cap = 0, stage_off = 0;
    std::string metrics_path;     // HFB200_METRICS=<file|stderr>: one JSON line per proved segment
    double metrics_peak_gbs = 0;  // HFB200_HBM_PEAK_GBS: denominator for the NTT/LDE roofline fraction in that line
    uint64_t host_syncs = 0, host_syncs_at_begin = 0;

    void init(int device, uint32_t max_po2_, uint32_t wc, uint32_t wd, uint32_t wa, const IrTap* taps = nullptr, size_t n_taps = 0,
              const IrStep* steps = nullptr, size_t n_steps = 0, uint32_t ret = 0, uint32_t n_mix_ir = 0, const uint8_t* info16 = nullptr) {
        if (max_po2_ < MIN_PO2 || max_po2_ > MAX_PO2) throw Err("max_po2 must be in [12, 22]");
        max_po2 = max_po2_;
        set_circuit_info(circuit_info, taps != nullptr, info16);
#ifndef HFB200_EMU
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0) throw Err(std::string("no CUDA device available (libhfb200 has no CPU fallback): ") + cudaGetErrorString(e));
        if (device < 0 || device >= count) throw Err("device index out of range");
        CUDA_CHECK(cudaSetDevice(device));
        device_id = device;
        dev.device = device;
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10) throw Err(std::string("libhfb200 is built for sm_100a only; found ") + prop.name);
        dev.sm_count = prop.multiProcessorCount;
        CUDA_CHECK(cudaStreamCreateWithFlags(&dev.stream, cudaStreamNonBlocking));
        for (auto& ev_ : evs) CUDA_CHECK(cudaEventCreate(&ev_));
        CUDA_CHECK(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
        for (auto& ev_ : chunk_ev) CUDA_CHECK(cudaEventCreateWithFlags(&ev_, cudaEventDisableTiming));
        CUDA_CHECK(cudaEventCreateWithFlags(&copy_gate, cudaEventDisableTiming));
#else
        (void)device;
#endif
        ntt.init(&dev);
        merkle.init(&dev);
        if (taps) {
            gen.init(&dev, wc, wd, wa, n_mix_ir, taps, n_taps, steps, n_steps, ret);
            jit.init(gen, max_po2);  // specialised for the context's largest segment size now, for other sizes on first use
            cir.init_widths(wc, wd, wa, (uint32_t)gen.taps.size(), n_mix_ir);
        } else {
            cir.init(&dev, wc, wd, wa);
        }
        arena.cap = arena_bytes(max_po2);
        arena.base = (uint8_t*)dev.alloc(arena.cap);
        if (const char* env = std::getenv("HFB200_DEBUG_CHECKPOINTS")) debug_checkpoints = std::atoi(env) != 0;
        if (const char* env = std::getenv("HFB200_METRICS")) metrics_path = env;
        if (const char* env = std::getenv("HFB200_HBM_PEAK_GBS")) metrics_peak_gbs = std::atof(env);
        stage_cap = (size_t)4 << 20;
        if (gen.active) stage_cap += (size_t)gen.n_mixpow * sizeof(E4);
        // the device transcript's landing area, sized once for the largest segment (seal_words grows with po2): a CUDA graph of
        // transcript mode 2 records its device->host copies into this buffer, so it must stay put until destroy()
        out_cap = (seal_words(max_po2) + CP_WORDS) * 4;
#ifndef HFB200_EMU
        CUDA_CHECK(cudaHostAlloc((void**)&stage_h, stage_cap, cudaHostAllocDefault));
        CUDA_CHECK(cudaHostAlloc((void**)&out_h, out_cap, cudaHostAllocDefault));
#else
        stage_h = (uint8_t*)std::malloc(stage_cap);
        out_h = (uint8_t*)std::malloc(out_cap);
        if (!stage_h || !out_h) throw Err("emu: out of memory");
#endif
    }
    // asynchronous upload of a small host array: staged in pinned memory when it fits (no sync needed), else copy + sync
    void h2d_small(void* d, const void* h, size_t bytes) {
        const size_t need = (bytes + 63) & ~(size_t)63;
        if (stage_h && stage_off + need <= stage_cap) {
            std::memcpy(stage_h + stage_off, h, bytes);
            dev.h2d(d, stage_h + stage_off, bytes);
            stage_off += need;
        } else {
            if (marks_off) throw Err("internal: parameter staging area exhausted while a CUDA graph is captured or replayed");
            dev.h2d(d, h, bytes);
            sync();
        }
    }
    void sync() { dev.sync(); host_syncs++; }
    // error path of an API entry: wait for everything queued on both streams (best effort, never throws) so that no copy from
    // or to caller memory is still in flight when the error is returned; the half-proved segment is abandoned
    void quiesce() noexcept {
#ifndef HFB200_EMU
        cudaSetDevice(device_id);
        if (copy_stream) cudaStreamSynchronize(copy_stream);
        if (dev.stream) cudaStreamSynchronize(dev.stream);
#endif
        begun = false;
        witness_open = false;
    }
    void destroy() {
        dev.free(arena.base);
        dev.free(wit_scratch);
        wit_scratch = nullptr; wit_scratch_cap = 0;
#ifndef HFB200_EMU
        drop_graphs();
        if (stage_h) cudaFreeHost(stage_h);
        if (out_h) cudaFreeHost(out_h);
#else
        std::free(stage_h);
        std::free(out_h);
#endif
        out_h = nullptr; out_cap = 0;
        stage_h = nullptr;
        jit.destroy();
        gen.destroy(&dev);
        cir.destroy(&dev);
        ntt.destroy();
#ifndef HFB200_EMU
        for (auto& ev_ : evs) if (ev_) cudaEventDestroy(ev_);
        {
            UploadChain& chain = UploadChain::of(device_id);
            std::lock_guard<std::mutex> lock(chain.mu);
            if (chain.last == chunk_ev[H2D_CHUNKS - 1]) chain.last = nullptr;  // nobody may wait on an event that is about to go
        }
        for (auto& ev_ : chunk_ev) if (ev_) cudaEventDestroy(ev_);
        if (copy_gate) cudaEventDestroy(copy_gate);
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (dev.stream) cudaStreamDestroy(dev.stream);
#endif
    }

    size_t arena_bytes(uint32_t p) const {
        const size_t N = (size_t)1 << p, W = cir.n_regs();
        // traces W*N, LDE (W+16)*4N, trees 4 * 2*4N*8, scratch wd*N, check 16N, E4 side arrays, FRI (< 40N), slack
        size_t words = W * N + (W + 16) * 4 * N + 4 * 64 * N + (size_t)cir.cd.w_data * N + 16 * N + 8 * 4 * N + 48 * N;
        words += (W + 16) * ((N + 511) / 512) * 16 + (1u << 20);  // dot-product partials (>= 512 rows per block)
        return words * 4 + (64u << 20);
    }

    // every API entry binds the calling host thread to this context's device (contexts may be driven from any thread)
    void bind() {
#ifndef HFB200_EMU
        CUDA_CHECK(cudaSetDevice(device_id));
#endif
    }
    bool marks_off = false;  // graph capture / replay: stage events cannot be recorded inside the graph
    void mark(int i) {
#ifndef HFB200_EMU
        if (marks_off) return;
        CUDA_CHECK(cudaEventRecord(evs[i], dev.stream));
#else
        (void)i;
#endif
    }
    float between(int i, int j) {
#ifndef HFB200_EMU
        if (marks_off) return 0.f;
        float m = 0; CUDA_CHECK(cudaEventElapsedTime(&m, evs[i], evs[j])); return m;
#else
        (void)i; (void)j; return 0.f;
#endif
    }

    static void nvtx_push(const char* name) {
#ifndef HFB200_EMU
        nvtxRangePushA(name);
#else
        (void)name;
#endif
    }
    static void nvtx_pop() {
#ifndef HFB200_EMU
        nvtxRangePop();
#endif
    }
    // one JSON line per segment (SURVEY.md section 5): po2, stage milliseconds, algorithmic bytes and GB/s of the NTT/LDE
    // pipeline, its fraction of the HBM peak when HFB200_HBM_PEAK_GBS is given, launches and host synchronisations
    void emit_metrics() const {
        if (metrics_path.empty()) return;
        char buf[1024];
        const double gbs = stats.ms_ntt_main > 0 ? (double)stats.ntt_main_bytes / (stats.ms_ntt_main * 1e-3) / 1e9 : 0.0;
        int n = std::snprintf(buf, sizeof buf,
            "{\"po2\": %u, \"columns\": %u, \"device\": %d, \"ms_total\": %.3f, \"ms_device\": %.3f, \"ms_h2d\": %.3f, \"ms_ntt_main\": %.3f, \"ms_hash_main\": %.3f, "
            "\"ms_accum\": %.3f, \"ms_check\": %.3f, \"ms_deep\": %.3f, \"ms_fri\": %.3f, \"launches\": %llu, \"host_syncs\": %llu, \"ntt_main_bytes\": %llu, \"ntt_main_gbs\": %.1f",
            po2, cir.n_regs(), device_id, stats.ms_total, stats.ms_device, stats.ms_h2d, stats.ms_ntt_main, stats.ms_hash_main, stats.ms_accum, stats.ms_check, stats.ms_deep,
            stats.ms_fri, (unsigned long long)stats.launches, (unsigned long long)stats.host_syncs, (unsigned long long)stats.ntt_main_bytes, gbs);
        if (metrics_peak_gbs > 0 && n > 0 && (size_t)n < sizeof buf) n += std::snprintf(buf + n, sizeof buf - n, ", \"hbm_peak_gbs\": %.1f, \"ntt_main_frac\": %.4f", metrics_peak_gbs, gbs / metrics_peak_gbs);
        if (n <= 0 || (size_t)n >= sizeof buf - 3) return;
        buf[n++] = '}'; buf[n++] = '\n'; buf[n] = 0;
        static std::mutex mu;  // contexts on several threads share the sink
        std::lock_guard<std::mutex> lock(mu);
        if (metrics_path == "stderr") { std::fputs(buf, stderr); return; }
        if (FILE* f = std::fopen(metrics_path.c_str(), "a")) { std::fputs(buf, f); std::fclose(f); }
    }

    void cp_add(const std::string& name, const uint32_t* w, size_t n) { cps.emplace_back(name, std::vector<uint32_t>(w, w + n)); }
    void cp_add(const std::string& name, const E4& e) { cp_add(name, e.c, 4); }

    // ---- buffers that depend on po2 only (resident trace lives here) ----
    void layout(uint32_t p) {
        if (p < 12 || p > max_po2) throw Err("po2 out of range for this context");
        if (p == po2 && tr[0]) return;
        po2 = p; have_trace = false; control_cached = false;
        const size_t N = (size_t)1 << p, D = 4 * N;
        arena.off = 0;
        const uint32_t w[3] = {cir.cd.w_accum, cir.cd.w_code, cir.cd.w_data};
        for (int g = 0; g < 3; g++) tr[g] = arena.take<uint32_t>((size_t)w[g] * N);
        for (int g = 0; g < 3; g++) ev[g] = arena.take<uint32_t>((size_t)w[g] * D);
        for (int g = 0; g < 3; g++) nodes[g] = arena.take<uint32_t>(2 * D * 8);
        ev_check = arena.take<uint32_t>(CHECK_SIZE * D);
        nodes_check = arena.take<uint32_t>(2 * D * 8);
        check = arena.take<uint32_t>(4 * D);
        scratch = arena.take<uint32_t>((size_t)cir.cd.w_data * N);
        d_mix = arena.take<uint32_t>(cir.n_mix());
        seg_mark = arena.off;
    }

    // ---- commit helpers ----
    void commit_tree(const Tree& t, const char* cp_name, std::vector<uint32_t>* keep = nullptr, const std::vector<uint32_t>* cached = nullptr) {
        const MerkleShape ms(t.rows);
        std::vector<uint32_t> top((size_t)2 * ms.top_size * 8);
        if (cached) {
            if (cached->size() != top.size()) throw Err("internal: cached control tree has the wrong shape");
            top = *cached;
        } else {
            dev.d2h(top.data(), t.nodes, top.size() * 4);
            sync();  // the root feeds the transcript: a true dependency
        }
        if (keep) *keep = top;
        proof.insert(proof.end(), top.begin() + (size_t)ms.top_size * 8, top.end());
        rng.mix(&top[8]);
        cp_add(cp_name, &top[8], 8);
    }
    void commit_group(int g, const char* cp_name, int ev_ntt0, int ev_ntt1, int ev_hash1) {
        const size_t N = (size_t)1 << po2, D = 4 * N;
        const uint32_t w = cir.group_width(g);
        mark(ev_ntt0);
        ntt.lde(tr[g], N, ev[g], D, scratch, w, (int)po2);
        mark(ev_ntt1);
        merkle.build(ev[g], D, (uint32_t)D, w, nodes[g]);
        mark(ev_hash1);
        commit_tree(Tree{ev[g], D, (uint32_t)D, w, nodes[g]}, cp_name);
    }

    // checks the arguments, resets the per-segment state and queues the host->device copies of the trace (data columns in
    // H2D_CHUNKS slices on the copy stream).  Returns whether the data copy is chunked / the cached control group is used.
    struct Staged { bool chunked, use_control; };
    // HFB200_DEV_INPUTS: the caller's columns must be device memory of this context's device (a host pointer would make the
    // device-to-device copy fault or read another GPU's memory).  The emulator has no device memory to tell apart.
    void check_device_ptr(const void* ptr, const char* what) const {
#ifndef HFB200_EMU
        cudaPointerAttributes a{};
        const cudaError_t e = cudaPointerGetAttributes(&a, ptr);
        if (e != cudaSuccess) cudaGetLastError();  // not a pointer the driver knows: clear the error, refuse below
        if (e != cudaSuccess || a.type != cudaMemoryTypeDevice || a.device != device_id)
            throw Err(std::string("HFB200_DEV_INPUTS: ") + what + " is not device memory of device " + std::to_string(device_id));
#else
        (void)ptr; (void)what;
#endif
    }
    Staged stage_inputs(uint32_t p, const uint32_t* globals_h, const uint32_t* code_h, const uint32_t* data_h, uint64_t blind, bool dev_inputs = false) {
        t_begin = std::chrono::steady_clock::now();
        // data == NULL after hfb200_segment_witness_dev: the DATA columns are the caller's, already in place, blinded with the key
        // derived there (one segment, one key)
        const bool witness = !data_h && witness_open;
        if (witness && p != po2)
            throw Err("po2 " + std::to_string(p) + " differs from the one of hfb200_segment_witness_dev (" + std::to_string(po2) + ")");
        if (witness && blind != witness_seed)
            throw Err("blind_seed " + std::to_string(blind) + " differs from the one of hfb200_segment_witness_dev (" + std::to_string(witness_seed) + ")");
        bind();
        layout(p);
        const size_t N = (size_t)1 << po2;
        arena.off = seg_mark;
        proof.clear(); cps.clear(); rng = HostRng(hash_suite); stats = Stats();
        for (auto& s : stage_ms) s = 0;
        launches_at_begin = dev.launches;
        host_syncs_at_begin = host_syncs;
        stage_off = 0;
        // every argument check comes BEFORE the first copy is queued: an error return must not leave DMA from caller memory in flight
        for (uint32_t i = 0; i < N_GLOBAL; i++) if (globals_h[i] >= P) throw Err("globals: non-canonical field element");
        if ((data_h || witness) && !code_h && !control_cached) throw Err("code is NULL and no control group is resident for this po2 (hfb200_control_root)");
        if (!data_h && !witness && !have_trace) throw Err("no trace: pass code/data (code may be NULL after hfb200_control_root) or call hfb200_witgen_synth first");
        if (!witness) blind_key = make_blind_key(blind);
        witness_open = false;  // any begin consumes (or, with data, abandons) the open witness
        if (dev_inputs && code_h) check_device_ptr(code_h, "code");
        if (dev_inputs && data_h) check_device_ptr(data_h, "data");
        std::memcpy(globals, globals_h, sizeof globals);
        mark(0);
        bool chunked = false;
        if (code_h) {
            if (dev_inputs) dev.d2d(tr[GROUP_CODE], code_h, (size_t)cir.cd.w_code * N * 4);
            else dev.h2d(tr[GROUP_CODE], code_h, (size_t)cir.cd.w_code * N * 4);
        }
        if (dev_inputs && data_h) dev.d2d(tr[GROUP_DATA], data_h, (size_t)cir.cd.w_data * N * 4);  // in stream order: no chunking needed
#ifndef HFB200_EMU
        else if (data_h && cir.cd.w_data >= (uint32_t)H2D_CHUNKS) {
            // the copy stream may not overwrite the data columns before everything already queued on the main
            // stream (a previous segment's readers) has finished
            CUDA_CHECK(cudaEventRecord(copy_gate, dev.stream));
            CUDA_CHECK(cudaStreamWaitEvent(copy_stream, copy_gate, 0));
            UploadChain& chain = UploadChain::of(device_id);
            std::unique_lock<std::mutex> chain_lock(chain.mu, std::defer_lock);
            if (UploadChain::enabled()) {
                chain_lock.lock();  // held while this upload is queued: the chain order is the queueing order
                if (chain.last && chain.last != chunk_ev[H2D_CHUNKS - 1]) CUDA_CHECK(cudaStreamWaitEvent(copy_stream, chain.last, 0));
            }
            for (int k = 0; k < H2D_CHUNKS; k++) {
                const uint32_t c0 = cir.cd.w_data * k / H2D_CHUNKS, c1 = cir.cd.w_data * (k + 1) / H2D_CHUNKS;
                CUDA_CHECK(cudaMemcpyAsync(tr[GROUP_DATA] + (size_t)c0 * N, data_h + (size_t)c0 * N, (size_t)(c1 - c0) * N * 4, cudaMemcpyHostToDevice, copy_stream));
                CUDA_CHECK(cudaEventRecord(chunk_ev[k], copy_stream));
            }
            if (chain_lock.owns_lock()) chain.last = chunk_ev[H2D_CHUNKS - 1];
            chunked = true;
        } else
#endif
        if (data_h && !dev_inputs) { dev.h2d(tr[GROUP_DATA], data_h, (size_t)cir.cd.w_data * N * 4); }
        const bool use_control = !code_h && (data_h || witness) && control_cached;
        if (code_h) { control_cached = false; control_gen = 0; }  // the resident control columns change
        if (data_h) have_trace = true;
        return Staged{chunked, use_control};
    }
    // LDE of the data group, slice by slice as the chunked copies land (or in one piece)
    void lde_data(bool chunked) {
        const size_t N = (size_t)1 << po2, D = 4 * N;
#ifndef HFB200_EMU
        if (chunked) {
            for (int k = 0; k < H2D_CHUNKS; k++) {
                const uint32_t c0 = cir.cd.w_data * k / H2D_CHUNKS, c1 = cir.cd.w_data * (k + 1) / H2D_CHUNKS;
                CUDA_CHECK(cudaStreamWaitEvent(dev.stream, chunk_ev[k], 0));
                ntt.lde(tr[GROUP_DATA] + (size_t)c0 * N, N, ev[GROUP_DATA] + (size_t)c0 * D, D, scratch, c1 - c0, (int)po2);
            }
            return;
        }
#endif
        (void)chunked;
        ntt.lde(tr[GROUP_DATA], N, ev[GROUP_DATA], D, scratch, cir.cd.w_data, (int)po2);
    }

    // ---- SegmentProver::prove, phase 1: header + CODE + DATA commits, returns the accum mix ----
    void begin(uint32_t p, const uint32_t* globals_h, const uint32_t* code_h, const uint32_t* data_h, uint64_t blind, bool dev_inputs = false) {
        const Staged sg = stage_inputs(p, globals_h, code_h, data_h, blind, dev_inputs);
        const bool chunked = sg.chunked, use_control = sg.use_control;
        const size_t N = (size_t)1 << po2;
        mark(1);
        const Digest8 gh = transcript_header(rng, circuit_info, globals, N_GLOBAL, po2);
        proof.insert(proof.end(), globals, globals + N_GLOBAL);
        proof.push_back(po2);
        cp_add("globals_hash", gh.w, 8);
        if (use_control) {
            mark(2); mark(3);
            const size_t D = 4 * N;
            commit_tree(Tree{ev[GROUP_CODE], D, (uint32_t)D, cir.cd.w_code, nodes[GROUP_CODE]}, "code_root", nullptr, &control_top);
        } else {
            StageRange r("hfb200:commit_code");
            commit_group(GROUP_CODE, "code_root", 1, 2, 3);
        }
        StageRange r_data("hfb200:commit_data");
        {
            const size_t D = 4 * N;
            mark(3);
            lde_data(chunked);
            mark(4);
            merkle.build(ev[GROUP_DATA], D, (uint32_t)D, cir.cd.w_data, nodes[GROUP_DATA]);
            mark(5);
            commit_tree(Tree{ev[GROUP_DATA], D, (uint32_t)D, cir.cd.w_data, nodes[GROUP_DATA]}, "data_root");
        }
        stage_ms[0] = between(0, 1);
        stage_ms[1] = between(1, 2) + between(3, 4);
        stage_ms[2] = between(2, 3) + between(4, 5);
        mix.resize(cir.n_mix());
        for (auto& m : mix) m = rng.random_elem();
        cp_add("accum_mix", mix.data(), mix.size());
        begun = true;
    }

    // ---- the device seam of the two-phase form (hfb200_segment_begin_dev .. _finish_dev) ----
    uint32_t* d_globals = nullptr;  // per segment, from the arena: valid until the segment is finished
    // begin, then the mix and the globals in device memory for the caller's step_accum
    void begin_dev(uint32_t p, const uint32_t* globals_h, const uint32_t* code_h, const uint32_t* data_h, uint64_t blind, bool dev_inputs) {
        begin(p, globals_h, code_h, data_h, blind, dev_inputs);
        d_globals = arena.take<uint32_t>(N_GLOBAL);
        h2d_small(d_globals, globals, N_GLOBAL * 4);
        h2d_small(d_mix, mix.data(), mix.size() * 4);
    }
    // in-place inclusive scan (product or sum) of the Fp4 chains in accum columns 4c..4c+3, rows [0, rows)
    void accum_scan(int kind, uint32_t first_chain, uint32_t n_chains, uint64_t rows) {
        if (!begun) throw Err("hfb200_segment_accum_scan: no segment in flight");
        if (kind != SCAN_PRODUCT && kind != SCAN_SUM) throw Err("hfb200_segment_accum_scan: kind must be HFB200_SCAN_PRODUCT (0) or HFB200_SCAN_SUM (1)");
        const uint32_t chains = cir.cd.w_accum / 4;
        if ((uint64_t)first_chain + n_chains > chains)
            throw Err("hfb200_segment_accum_scan: chains [" + std::to_string(first_chain) + ", " + std::to_string((uint64_t)first_chain + n_chains) +
                      ") beyond w_accum / 4 = " + std::to_string(chains));
        const uint64_t N = 1ull << po2;
        if (rows > N) throw Err("hfb200_segment_accum_scan: rows " + std::to_string(rows) + " > N = " + std::to_string(N));
        if (n_chains == 0 || rows == 0) return;
        bind();
        const uint32_t nblk = (uint32_t)((rows + ACC_RPB - 1) / ACC_RPB);
        const size_t save = arena.off;
        E4* partial = arena.take<E4>((size_t)n_chains * nblk);
        const size_t sm = (SCAN_TILE + 2 * ACC_ITEMS) * sizeof(E4);
        dev.launch<AccumScanKernel, 256, 1>(nblk, n_chains, 256, sm, tr[GROUP_ACCUM], N, rows, first_chain, kind, partial, 0);
        dev.launch<AccumOffsetsKernel, 256, 1>(1, n_chains, 256, 2 * (size_t)nblk * sizeof(E4), partial, nblk, kind);
        dev.launch<AccumScanKernel, 256, 1>(nblk, n_chains, 256, sm, tr[GROUP_ACCUM], N, rows, first_chain, kind, partial, 1);
        arena.off = save;  // stream order makes reuse by later kernels safe
    }
    // the ZK_CYCLES blinding rows of every column of group g, from this segment's key
    void blind_rows(int g) {
        bind();
        const uint32_t w = cir.group_width(g);
        const uint64_t total = (uint64_t)w * ZK_CYCLES;
        dev.launch<BlindRowsKernel, 256, 1>((unsigned)((total + 255) / 256), 1, 256, 0, tr[g], w, po2, ZK_CYCLES, (uint32_t)g, blind_key);
    }
    void accum_blind() {
        if (!begun) throw Err("hfb200_segment_accum_blind: no segment in flight");
        blind_rows(GROUP_ACCUM);
    }

    // ---- the device witness seam (hfb200_segment_witness_dev .. the begin that commits the columns) ----
    // witness_dev lays the context out for po2 and derives the segment's blinding key once; the caller's witness generator then
    // writes the resident DATA columns, and the next begin with data == NULL commits them as they stand, under that same key.
    bool witness_open = false;
    uint64_t witness_seed = 0;
    void* wit_scratch = nullptr;  // hfb200_segment_scratch: grows on demand, freed in destroy()
    size_t wit_scratch_cap = 0;
    void witness_dev(uint32_t p, uint64_t blind) {
        if (p < MIN_PO2 || p > max_po2)
            throw Err("hfb200_segment_witness_dev: po2 " + std::to_string(p) + " outside [12, " + std::to_string(max_po2) + "]");
        bind();
        if (begun) quiesce();  // a segment still in flight is abandoned; its chunked upload must not land over the caller's columns
        layout(p);             // the same po2 again keeps the resident control group
        have_trace = false;    // the data columns are the caller's from here on
        blind_key = make_blind_key(blind);
        witness_seed = blind;
        witness_open = true;
    }
    void data_blind() {
        if (!witness_open) throw Err("hfb200_segment_data_blind: no witness open (call hfb200_segment_witness_dev)");
        blind_rows(GROUP_DATA);
    }
    void* segment_scratch(size_t bytes) {
        if (!witness_open) throw Err("hfb200_segment_scratch: no witness open (call hfb200_segment_witness_dev)");
        if (bytes > wit_scratch_cap) {
            bind();
            if (wit_scratch) { dev.sync(); dev.free(wit_scratch); wit_scratch = nullptr; wit_scratch_cap = 0; }  // earlier users are done
            wit_scratch = dev.alloc(bytes);
            wit_scratch_cap = bytes;
        }
        return wit_scratch;
    }

    // key_dev != NULL: the blinding key is read from device memory (graph replay); the by-value copy is then a placeholder
    void step_accum(const BlindKey* key_dev = nullptr) {
        const size_t N = (size_t)1 << po2;
        const uint32_t nblk = (uint32_t)((N + ACC_RPB - 1) / ACC_RPB);
        E4* partial = arena.take<E4>((size_t)cir.cd.n_chains * nblk);
        const size_t sm1 = 2 * ACC_ITEMS * sizeof(E4);
        const BlindKey by_value = key_dev ? BlindKey{} : blind_key;
        dev.launch<AccumKernel, 256, 1>(nblk, cir.cd.n_chains, 256, sm1, tr[GROUP_ACCUM], (const uint32_t*)tr[GROUP_DATA], (const uint32_t*)d_mix, partial, cir.cd, po2, by_value, 0, key_dev);
        dev.launch<AccumOffsetsKernel, 256, 1>(1, cir.cd.n_chains, 256, 2 * (size_t)nblk * sizeof(E4), partial, nblk);
        dev.launch<AccumKernel, 256, 1>(nblk, cir.cd.n_chains, 256, sm1, tr[GROUP_ACCUM], (const uint32_t*)tr[GROUP_DATA], (const uint32_t*)d_mix, partial, cir.cd, po2, by_value, 1, key_dev);
    }

    static uint32_t rou_fwd(int k) { uint32_t g = to_mont(137); for (int i = k; i < 27; i++) g = fmul(g, g); return g; }

    // evaluates `w` columns against weight vector Wt (and its shift by one for the first n_back1 columns)
    void dot_group(const uint32_t* cols, uint32_t w, uint32_t n_back1, const E4* Wt, E4* out_dev) {
        const size_t N = (size_t)1 << po2;
        const uint32_t rpb = dot_rows_per_block(po2);
        const uint32_t nblk = (uint32_t)(N / rpb);
        const size_t save = arena.off;
        E4* partial = arena.take<E4>((size_t)w * nblk * 2);
        dev.launch<DotKernel, 256, 2>(nblk, (w + DT_CG - 1) / DT_CG, DT_T, DT_SMEM, cols, (uint64_t)N, w, n_back1, Wt, po2, partial, rpb);
        dev.launch<DotReduceKernel, 128, 1>((2 * w + 127) / 128, 1, 128, 0, (const E4*)partial, w, nblk, out_dev);
        arena.off = save;  // stream order makes reuse by later kernels safe
    }

    void dot_group_g(const uint32_t* cols, uint32_t w, const uint8_t* colmask, const Backs4& bk, const E4* Wt, E4* out_dev) {
        const size_t N = (size_t)1 << po2;
        const uint32_t nblk = (uint32_t)((N + DOT_RPB - 1) / DOT_RPB);
        const size_t save = arena.off;
        E4* partial = arena.take<E4>((size_t)w * nblk * GEN_MAX_BACKS);
        dev.launch<DotKernelG, 128, 3>(nblk, (w + DOTG_CPB - 1) / DOTG_CPB, DOTG_T, (size_t)DOTG_T * DOTG_CPB * GEN_MAX_BACKS * sizeof(E4), cols, (uint64_t)N, w, colmask, bk, Wt, po2, partial);
        dev.launch<DotReduceKernelG, 128, 1>((GEN_MAX_BACKS * w + 127) / 128, 1, 128, 0, (const E4*)partial, w, nblk, out_dev);
        arena.off = save;
    }
    // coefficients (low to high) of the polynomial of degree < n through (xs[i], ys[i]), n <= 4
    static void lagrange_e4(E4* out, const E4* xs, const E4* ys, uint32_t n) {
        for (uint32_t i = 0; i < n; i++) out[i] = e4_zero();
        for (uint32_t i = 0; i < n; i++) {
            E4 b[5]; uint32_t nb = 1; b[0] = e4_one();
            E4 den = e4_one();
            for (uint32_t j = 0; j < n; j++) {
                if (j == i) continue;
                E4 nbuf[5];
                for (uint32_t k = 0; k <= nb; k++) nbuf[k] = e4_zero();
                for (uint32_t k = 0; k < nb; k++) { nbuf[k + 1] = e4_add(nbuf[k + 1], b[k]); nbuf[k] = e4_sub(nbuf[k], e4_mul(b[k], xs[j])); }
                nb++;
                for (uint32_t k = 0; k < nb; k++) b[k] = nbuf[k];
                den = e4_mul(den, e4_sub(xs[i], xs[j]));
            }
            const E4 sc = e4_mul(ys[i], e4_inv(den));
            for (uint32_t k = 0; k < nb; k++) out[k] = e4_add(out[k], e4_mul(b[k], sc));
        }
    }

    // ---- phase 2: ACCUM commit, check polynomial, DEEP, FRI, queries ----
    // dev_accum: hfb200_segment_finish_dev -- the accum columns are already in device memory (the caller's step_accum); ms_accum
    // is then the stream time from the end of the DATA commit (begin's event 5) to this call
    void finish(const uint32_t* accum_h, std::vector<uint32_t>& seal_out, bool dev_accum = false) {
        if (!begun) throw Err(dev_accum ? "hfb200_segment_finish_dev: no segment in flight" : "segment_finish without segment_begin");
        begun = false;
        bind();
        const size_t N = (size_t)1 << po2, D = 4 * N;
        const CircuitDev& cd = cir.cd;
        const uint32_t W = cir.n_regs(), T = cir.n_taps;

        if (dev_accum) {
            mark(6);
            h2d_small(d_mix, mix.data(), mix.size() * 4);  // after begin (host) the mix is not on the device yet
        } else {
            mark(5);
            h2d_small(d_mix, mix.data(), mix.size() * 4);
            if (accum_h) dev.h2d(tr[GROUP_ACCUM], accum_h, (size_t)cd.w_accum * N * 4);
            else if (gen.active) throw Err("data-defined circuit: step_accum is the caller's (pass the accum columns to hfb200_segment_finish)");
            else step_accum();
            mark(6);
        }
        { StageRange r("hfb200:commit_accum"); commit_group(GROUP_ACCUM, "accum_root", 6, 7, 8); }  // ends with a stream sync: events 5..8 are complete
        stage_ms[3] = between(5, 6);
        stage_ms[1] += between(6, 7);
        stage_ms[2] += between(7, 8);

        // ---- check polynomial ----
        nvtx_push("hfb200:check");
        const E4 poly_mix = rng.random_ext();
        cp_add("poly_mix", poly_mix);
        uint32_t yinv4[4];
        {
            const uint32_t three_n = fpow(THREE, N), w4 = rou_fwd(2);
            uint32_t y = three_n;
            for (int s = 0; s < 4; s++) { yinv4[s] = finv(fsub(y, ONE)); y = fmul(y, w4); }
        }
        if (gen.active) {
            std::vector<E4> mp(gen.n_mixpow);
            E4 cur = e4_one();
            for (auto& m : mp) { m = cur; cur = e4_mul(cur, poly_mix); }
            E4* d_mp = arena.take<E4>(mp.size());
            h2d_small(d_mp, mp.data(), mp.size() * sizeof(E4));
            uint32_t* d_gl = arena.take<uint32_t>(N_GLOBAL);
            h2d_small(d_gl, globals, N_GLOBAL * 4);
            if (jit.ensure(po2)) {  // per size: the interpreter runs a size whose kernels are neither cached nor compilable
                JitEvalArgs ja{};
                ja.ev[0] = ev[GROUP_ACCUM]; ja.ev[1] = ev[GROUP_CODE]; ja.ev[2] = ev[GROUP_DATA];
                ja.check = check; ja.mixpow = d_mp; ja.mix = d_mix; ja.globals = d_gl; ja.po2 = po2;
                for (int s_ = 0; s_ < 4; s_++) ja.yinv[s_] = yinv4[s_];
                jit.launch(dev, ja, D);
            } else {
            // interpreter kernel, one launch per chunk (same chunks as the JIT: small slot files, more rows per block)
            bool first = true;
            for (const GenericCircuitHost::Chunk& ck : gen.chunks) {
                GenEvalArgs a{};
                a.ev[0] = ev[GROUP_ACCUM]; a.ev[1] = ev[GROUP_CODE]; a.ev[2] = ev[GROUP_DATA];
                a.check = check; a.prog = ck.d_prog; a.n_ins = (uint32_t)ck.prog.size(); a.mixpow = d_mp; a.mix = d_mix; a.globals = d_gl;
                a.n_mix = gen.n_mix; a.po2 = po2; a.n_fp_slots = ck.n_fp_slots; a.n_mix_slots = ck.n_mix_slots; a.ret_slot = ck.ret_slot;
                a.accumulate = first ? 0u : 1u;
                first = false;
                for (int s_ = 0; s_ < 4; s_++) a.yinv[s_] = yinv4[s_];
                // rows per block: as many as fit the slot files in shared memory
                const size_t per_row = (size_t)ck.n_mix_slots * sizeof(E4) + (size_t)ck.n_fp_slots * 4;
                uint32_t R = 128;
                while (R > 32 && per_row * R + (N_GLOBAL + gen.n_mix) * 4 > 160 * 1024) R >>= 1;
                if (per_row * R + (N_GLOBAL + gen.n_mix) * 4 > 220 * 1024) throw Err("data-defined circuit: too many live values for the interpreter's shared-memory slot file");
                a.rows_per_block = R;
                dev.launch<GenEvalCheckKernel, 128, 1>((unsigned)((D + R - 1) / R), 1, (int)R, per_row * R + (N_GLOBAL + gen.n_mix) * 4 + 16, a);
            }
            }
        } else {
            const uint32_t nc = cd.n_constraints();
            std::vector<E4> mp(nc);
            E4 cur = e4_one();
            for (auto& m : mp) { m = cur; cur = e4_mul(cur, poly_mix); }
            E4* d_mp = arena.take<E4>(nc);
            h2d_small(d_mp, mp.data(), nc * sizeof(E4));
            EvalCheckArgs a{};
            a.ev_accum = ev[GROUP_ACCUM]; a.ev_code = ev[GROUP_CODE]; a.ev_data = ev[GROUP_DATA];
            a.check = check; a.mixpow = d_mp; a.mix = d_mix; a.global0 = globals[0];
            for (int s_ = 0; s_ < 4; s_++) a.yinv[s_] = yinv4[s_];
            a.po2 = po2; a.cd = cd;
            a.rows_per_block = 128;
            dev.launch<EvalCheckKernel, 128, 1>((unsigned)((D + 127) / 128), 1, 128, (size_t)nc * sizeof(E4) + (size_t)6 * cd.n_free * 2 + 16, a);
        }
        // 4 polys of 4N evaluations -> coefficients (no zk_shift); bit-reversed order makes them 16 polys of N
        ntt.interpolate(check, D, check, D, 4, (int)po2 + 2, false);
        ntt.expand_evaluate(check, N, ev_check, D, CHECK_SIZE, (int)po2, 2);
        merkle.build(ev_check, D, (uint32_t)D, CHECK_SIZE, nodes_check);
        mark(9);
        commit_tree(Tree{ev_check, D, (uint32_t)D, CHECK_SIZE, nodes_check}, "check_root");
        stage_ms[4] = between(8, 9);
        nvtx_pop();
        nvtx_push("hfb200:deep");

        // ---- DEEP: evaluations at z ----
        const E4 z = rng.random_ext();
        cp_add("z", z);
        const uint32_t omega = rou_fwd((int)po2), back_one = finv(omega);
        const E4 z3 = e4_scale(z, THREE), z4 = e4_pow(z, 4);
        E4 A = e4_pow(z3, N); A.c[0] = fsub(A.c[0], ONE);
        A = e4_scale(A, finv(to_mont((uint32_t)(N % P))));
        E4* INV = arena.take<E4>(N); E4* Lw = arena.take<E4>(N); E4* INV4 = arena.take<E4>(N); E4* W4 = arena.take<E4>(N);
        dev.launch<DeepWeightsKernel, 256, 1>((unsigned)((N + 255) / 256), 1, 256, 0, INV, Lw, INV4, z3, z4, A, po2, ntt.rt);
        {
            std::vector<E4> xs(po2);
            E4 cur = z4;
            for (uint32_t k = 0; k < po2; k++) { xs[k] = cur; cur = e4_mul(cur, cur); }
            E4* d_xs = arena.take<E4>(po2);
            h2d_small(d_xs, xs.data(), po2 * sizeof(E4));
            dev.launch<PowBitrevKernel, 256, 1>((unsigned)((N + 255) / 256), 1, 256, 0, W4, (const E4*)d_xs, po2);
        }
        std::vector<E4> coeff_u(T + CHECK_SIZE);
        std::vector<uint32_t> reg_tap(W);
        std::vector<uint8_t> reg_two(W);
        if (gen.active) {
            // data-defined circuit: arbitrary tap sets.  Evaluations for every (column, back slot), then per register
            // the Lagrange interpolant through its tap points.
            Backs4 bk{};
            bk.nb = (uint32_t)gen.backs.size();
            for (uint32_t s_ = 0; s_ < bk.nb; s_++) bk.back[s_] = gen.backs[s_];
            E4* d_ev = arena.take<E4>((size_t)GEN_MAX_BACKS * W);
            E4* d_evc = arena.take<E4>((size_t)2 * CHECK_SIZE);
            const uint32_t goff4[3] = {0, GEN_MAX_BACKS * cd.w_accum, GEN_MAX_BACKS * (cd.w_accum + cd.w_code)};
            for (int g = 0; g < 3; g++) dot_group_g(tr[g], cir.group_width(g), gen.d_colmask[g], bk, Lw, d_ev + goff4[g]);
            dot_group(check, CHECK_SIZE, 0, W4, d_evc);
            std::vector<E4> h_ev((size_t)GEN_MAX_BACKS * W), h_evc((size_t)2 * CHECK_SIZE);
            dev.d2h(h_ev.data(), d_ev, h_ev.size() * sizeof(E4));
            dev.d2h(h_evc.data(), d_evc, h_evc.size() * sizeof(E4));
            sync();
            for (const GenReg& r : gen.regs) {
                E4 xs[4], ys[4];
                for (uint32_t k = 0; k < r.size; k++) {
                    const uint32_t back = gen.taps[r.tap_begin + k].back;
                    xs[k] = e4_scale(z, fpow(back_one, back));
                    ys[k] = h_ev[goff4[r.group] + GEN_MAX_BACKS * r.offset + gen.back_slot(back)];
                }
                lagrange_e4(&coeff_u[r.tap_begin], xs, ys, r.size);
            }
            for (uint32_t c = 0; c < CHECK_SIZE; c++) coeff_u[T + c] = h_evc[2 * c];
        } else {
        E4* d_evals = arena.take<E4>((size_t)2 * (W + CHECK_SIZE));
        uint32_t goff[4] = {0, 2 * cd.w_accum, 2 * (cd.w_accum + cd.w_code), 2 * W};
        for (int g = 0; g < 3; g++) dot_group(tr[g], cir.group_width(g), cir.group_back1(g), Lw, d_evals + goff[g]);
        dot_group(check, CHECK_SIZE, 0, W4, d_evals + goff[3]);
        std::vector<E4> h_evals((size_t)2 * (W + CHECK_SIZE));
        dev.d2h(h_evals.data(), d_evals, h_evals.size() * sizeof(E4));
        sync();  // the tap evaluations feed the transcript: a true dependency
        // taps order: (group, column, back).  coeff_u: per register, interpolant through its tap points.
        {
            const E4 x0 = z, x1 = e4_scale(z, back_one);
            const E4 dinv = e4_inv(e4_sub(x0, x1));
            uint32_t t = 0, reg = 0;
            for (int g = 0; g < 3; g++)
                for (uint32_t c = 0; c < cir.group_width(g); c++, reg++) {
                    const E4 u0 = h_evals[goff[g] + 2 * c], u1 = h_evals[goff[g] + 2 * c + 1];
                    reg_tap[reg] = t;
                    if (c < cir.group_back1(g)) {
                        const E4 c1 = e4_mul(e4_sub(u0, u1), dinv);
                        coeff_u[t] = e4_sub(u0, e4_mul(c1, x0));
                        coeff_u[t + 1] = c1;
                        reg_two[reg] = 1; t += 2;
                    } else { coeff_u[t] = u0; reg_two[reg] = 0; t += 1; }
                }
            if (t != T) throw Err("internal: tap count mismatch");
            for (uint32_t c = 0; c < CHECK_SIZE; c++) coeff_u[T + c] = h_evals[goff[3] + 2 * c];
        }
        }
        proof.insert(proof.end(), reinterpret_cast<uint32_t*>(coeff_u.data()), reinterpret_cast<uint32_t*>(coeff_u.data()) + 4 * coeff_u.size());
        const Digest8 hash_u = suite_hash_elems(hash_suite, reinterpret_cast<uint32_t*>(coeff_u.data()), 4 * coeff_u.size());
        rng.mix(hash_u.w);
        cp_add("hash_u", hash_u.w, 8);

        // ---- DEEP: quotient, point-wise on the trace domain ----
        const E4 dmix = rng.random_ext();
        cp_add("deep_mix", dmix);
        const uint32_t n_regs = gen.active ? (uint32_t)gen.regs.size() : W;
        std::vector<E4> reg_mix(n_regs + CHECK_SIZE);
        { E4 cur = e4_one(); for (auto& m : reg_mix) { m = cur; cur = e4_mul(cur, dmix); } }
        E4 Vc = e4_zero();
        for (uint32_t c = 0; c < CHECK_SIZE; c++) Vc = e4_add(Vc, e4_mul(reg_mix[n_regs + c], coeff_u[T + c]));
        E4* d_regmix = arena.take<E4>(n_regs + CHECK_SIZE);
        h2d_small(d_regmix, reg_mix.data(), reg_mix.size() * sizeof(E4));
        uint32_t* S0 = arena.take<uint32_t>(4 * N);
        uint32_t* S1 = arena.take<uint32_t>(4 * N);
        uint32_t* fin = arena.take<uint32_t>(4 * N);
        dev.launch<CheckMixKernel, 256, 1>((unsigned)((N + 255) / 256), 1, 256, 0, (const uint32_t*)check, (const E4*)(d_regmix + n_regs), S0, po2, ntt.rt);
        ntt.expand_evaluate(S0, N, S1, N, 4, (int)po2, 0);
        if (gen.active) {
            DeepMixGArgs ga{};
            const uint32_t C = (uint32_t)gen.combos.size();
            ga.n_combos = C; ga.Vc = Vc;
            // registers grouped by combo (the sum is exact, its order is free), mix powers permuted alongside
            std::vector<uint32_t> rc_sorted; std::vector<E4> rm_sorted;
            for (uint32_t c = 0; c < C; c++) {
                ga.combo_start[c] = (uint32_t)rc_sorted.size();
                ga.combo_nb[c] = (uint32_t)gen.combos[c].size();
                for (uint32_t k = 0; k < ga.combo_nb[c]; k++) {
                    ga.combo_back[c][k] = gen.combos[c][k];
                    ga.combo_fb[c][k] = fmul(fneg(THREE), fpow(omega, gen.combos[c][k]));
                    ga.U[c][k] = e4_zero();
                }
                for (size_t ri = 0; ri < gen.regs.size(); ri++) {
                    const GenReg& r = gen.regs[ri];
                    if (r.combo != c) continue;
                    rc_sorted.push_back((r.group << 28) | r.offset);
                    rm_sorted.push_back(reg_mix[ri]);
                    for (uint32_t k = 0; k < r.size; k++) ga.U[c][k] = e4_add(ga.U[c][k], e4_mul(reg_mix[ri], coeff_u[r.tap_begin + k]));
                }
            }
            ga.combo_start[C] = (uint32_t)rc_sorted.size();
            uint32_t* d_rc = arena.take<uint32_t>(rc_sorted.size());
            E4* d_rm = arena.take<E4>(rm_sorted.size());
            h2d_small(d_rc, rc_sorted.data(), rc_sorted.size() * 4);
            h2d_small(d_rm, rm_sorted.data(), rm_sorted.size() * sizeof(E4));
            for (int g = 0; g < 3; g++) ga.tr[g] = tr[g];
            ga.regcol = d_rc; ga.regmix = d_rm; ga.S = S1; ga.INV = INV; ga.INV4 = INV4; ga.out = fin; ga.po2 = po2; ga.rt = ntt.rt;
            dev.launch<DeepMixKernelG, 256, 1>((unsigned)((N + 255) / 256), 1, 256, 0, ga);
        } else {
            DeepMixArgs da{};
            da.U0 = da.U1a = da.U1b = e4_zero();
            da.Vc = Vc;
            for (uint32_t reg = 0; reg < W; reg++) {
                if (reg_two[reg]) { da.U1a = e4_add(da.U1a, e4_mul(reg_mix[reg], coeff_u[reg_tap[reg]])); da.U1b = e4_add(da.U1b, e4_mul(reg_mix[reg], coeff_u[reg_tap[reg] + 1])); }
                else da.U0 = e4_add(da.U0, e4_mul(reg_mix[reg], coeff_u[reg_tap[reg]]));
            }
            for (int g = 0; g < 3; g++) { da.tr[g] = tr[g]; da.w[g] = cir.group_width(g); da.n_back1[g] = cir.group_back1(g); }
            da.mixpow = d_regmix; da.S = S1; da.INV = INV; da.INV4 = INV4; da.out = fin; da.omega = omega; da.po2 = po2; da.rt = ntt.rt;
            dev.launch<DeepMixKernel, 256, 1>((unsigned)((N + 255) / 256), 1, 256, 0, da);
        }
        ntt.interpolate(fin, N, fin, N, 4, (int)po2, true);  // bit-reversed coefficients of the FRI polynomial
        mark(10);
        nvtx_pop();
        nvtx_push("hfb200:fri");
        if (debug_checkpoints) {
            std::vector<uint32_t> fc(4 * N);
            dev.d2h(fc.data(), fin, fc.size() * 4); sync();
            const Digest8 d = suite_hash_elems(hash_suite, fc.data(), fc.size());
            cp_add("final_poly_hash", d.w, 8);
        }

        // ---- FRI ----
        struct Round { Tree tree; };
        std::vector<Round> rounds;
        uint32_t* coeffs = fin;
        size_t n = N;
        while (n > FRI_MIN_DEGREE) {
            const size_t dom = n * INV_RATE, rows = dom / FRI_FOLD;
            uint32_t* evr = arena.take<uint32_t>(4 * dom);
            uint32_t* ndr = arena.take<uint32_t>(2 * rows * 8);
            ntt.expand_evaluate(coeffs, n, evr, dom, 4, ilog2(n), 2);
            merkle.build(evr, rows, (uint32_t)rows, FRI_FOLD * 4, ndr);
            Tree t{evr, rows, (uint32_t)rows, FRI_FOLD * 4, ndr};
            const std::string rn = std::to_string(rounds.size());
            commit_tree(t, ("fri_root_" + rn).c_str());
            const E4 fm = rng.random_ext();
            cp_add("fri_mix_" + rn, fm);
            FriFoldArgs fa{};
            fa.in = coeffs; fa.n = (uint32_t)n;
            fa.out = arena.take<uint32_t>(4 * n / FRI_FOLD);
            { E4 cur = e4_one(); for (int i = 0; i < 16; i++) { fa.mixpow[i] = cur; cur = e4_mul(cur, fm); } }
            dev.launch<FriFoldKernel, 256, 1>((unsigned)((n / 16 + 255) / 256), 1, 256, 0, fa);
            coeffs = fa.out;
            n /= FRI_FOLD;
            rounds.push_back(Round{t});
        }
        {
            uint32_t* nat = arena.take<uint32_t>(4 * n);
            dev.launch<BitRevKernel, 256, 1>((unsigned)((4 * n + 255) / 256), 1, 256, 0, (const uint32_t*)coeffs, nat, 4u, (uint32_t)ilog2(n));
            std::vector<uint32_t> fc(4 * n);
            dev.d2h(fc.data(), nat, fc.size() * 4); sync();  // the final coefficients feed the transcript
            proof.insert(proof.end(), fc.begin(), fc.end());
            const Digest8 d = suite_hash_elems(hash_suite, fc.data(), fc.size());
            rng.mix(d.w);
            cp_add("fri_final_hash", d.w, 8);
        }
        // ---- queries: every opening of every tree in one gather launch ----
        {
            const Tree main_trees[4] = {Tree{ev[0], D, (uint32_t)D, cd.w_accum, nodes[0]}, Tree{ev[1], D, (uint32_t)D, cd.w_code, nodes[1]},
                                        Tree{ev[2], D, (uint32_t)D, cd.w_data, nodes[2]}, Tree{ev_check, D, (uint32_t)D, CHECK_SIZE, nodes_check}};
            std::vector<OpenDesc> descs;
            std::vector<uint32_t> positions;
            uint32_t off = 0;
            auto add = [&](const Tree& t, uint32_t idx) {
                const MerkleShape ms(t.rows);
                descs.push_back(OpenDesc{t.matrix, t.nodes, t.col_stride, t.rows, t.cols, idx, ms.top_size, off});
                off += t.cols + ms.path_words();
            };
            for (uint32_t q = 0; q < QUERIES; q++) {
                uint32_t pos = rng.random_bits((unsigned)ilog2(D)) % (uint32_t)D;
                positions.push_back(pos);
                for (const Tree& t : main_trees) add(t, pos);
                for (const Round& r : rounds) { pos %= r.tree.rows; add(r.tree, pos); }
            }
            cp_add("query_positions", positions.data(), positions.size());
            OpenDesc* d_descs = arena.take<OpenDesc>(descs.size());
            uint32_t* d_out = arena.take<uint32_t>(off);
            h2d_small(d_descs, descs.data(), descs.size() * sizeof(OpenDesc));
            dev.launch<OpenKernel, 128, 1>((unsigned)descs.size(), 1, 128, 0, (const OpenDesc*)d_descs, d_out);
            const size_t at = proof.size();
            proof.resize(at + off);
            mark(11);
            dev.d2h(proof.data() + at, d_out, (size_t)off * 4);
            sync();
        }
        nvtx_pop();
        stage_ms[5] = between(9, 10);
        stage_ms[6] = between(10, 11);
        stats.ms_h2d = stage_ms[0]; stats.ms_ntt_main = stage_ms[1]; stats.ms_hash_main = stage_ms[2]; stats.ms_accum = stage_ms[3];
        stats.ms_check = stage_ms[4]; stats.ms_deep = stage_ms[5]; stats.ms_fri = stage_ms[6];
        stats.ms_device = between(0, 11);
        stats.ms_total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        stats.launches = dev.launches - launches_at_begin;
        stats.ntt_main_bytes = 28ull * W * N;
        stats.host_syncs = host_syncs - host_syncs_at_begin;
        emit_metrics();
        seal_out = proof;
    }

    // ---- SegmentProver::prove with the transcript on the device (built-in circuit, one-shot entries) -------------------------
    // Same kernels and the same seal as begin() + finish(); what differs is WHO runs the transcript: every Fiat-Shamir step is a
    // one-warp kernel on the stream (transcript.cuh), the parameters it derives stay in device memory, the seal is assembled in
    // a device buffer.  The host enqueues the whole segment and synchronises ONCE, for the seal (10 times on the host path).
    // OPT-IN (HFB200_DEVICE_TRANSCRIPT=1 or hfb200_set_transcript): measured on B200 it is ~1 % SLOWER than the host transcript
    // at 1, 2 and 4 contexts in flight (18.74 / 19.47 / 19.81 against 18.95 / 19.54 / 19.86 segments/s at po2 = 20; 6.19 against
    // 5.54 ms for one po2 = 16 segment): a segment's transcript is ~170 SEQUENTIAL Poseidon2 permutations (92 for hash_u, 64 for the
    // final coefficients, 13 for the query draws), a warp-cooperative permutation takes ~3.3 us on the GPU against ~1 us on a host
    // core, and the stream synchronisations it removes cost less than that.  It pays where host threads are the scarce resource.
    // Mode 2 adds CUDA-GRAPH REPLAY on top: a device-transcript segment is a fixed, stream-ordered sequence of ~170 launches and a
    // handful of small copies whose arguments depend on (circuit, po2) only -- every per-segment value (globals, RNG header,
    // blinding key, tree descriptors) reaches the kernels through pinned staging memory or device memory, never by value.  The
    // first segment of a (po2, control-reuse) shape runs plainly (module loading, attribute set-up), the second is captured
    // (cudaStreamBeginCapture .. EndCapture, instantiated once), every later one refills the staging area and issues ONE
    // cudaGraphLaunch.  Trace uploads from caller memory stay outside the graph (their source pointers change per call).
    int transcript_mode = -1;  // -1: environment, 0: host, 1: device, 2: device + CUDA-graph replay
    static int env_transcript() { static const int v = [] { const char* e = std::getenv("HFB200_DEVICE_TRANSCRIPT"); return e ? std::atoi(e) : 0; }(); return v; }
    int transcript_setting() const { return transcript_mode < 0 ? env_transcript() : transcript_mode; }
    // the device transcript runs Poseidon2Rng only: SHA-256 contexts always take the host transcript
    bool device_transcript() const { return transcript_setting() >= 1 && !gen.active && hash_suite == HASH_POSEIDON2; }
    bool graph_replay() const { return device_transcript() && transcript_setting() >= 2 && !debug_checkpoints; }
    uint64_t graph_launches = 0;  // segments issued as one cudaGraphLaunch
    uint8_t* out_h = nullptr;     // pinned landing area of the seal and the checkpoint words (device-transcript path), allocated in init
    size_t out_cap = 0;
#ifndef HFB200_EMU
    struct GraphEntry { int state = 0; cudaGraphExec_t exec = nullptr; };  // 0: never run, 1: warmed up, 2: instantiated
    std::map<uint64_t, GraphEntry> graphs;                                // key = po2 * 2 + use_control
    void drop_graphs() {
        for (auto& g : graphs) if (g.second.exec) cudaGraphExecDestroy(g.second.exec);
        graphs.clear();
    }
#endif
    void prove_device(uint32_t p, const uint32_t* globals_h, const uint32_t* code_h, const uint32_t* data_h, uint64_t blind, std::vector<uint32_t>& seal_out) {
        const Staged sg = stage_inputs(p, globals_h, code_h, data_h, blind);
        begun = false;
        const size_t N = (size_t)1 << po2, D = 4 * N;
        const CircuitDev& cd = cir.cd;
        const uint32_t W = cir.n_regs(), T = cir.n_taps, n_mix = cir.n_mix();
        const size_t words = seal_words(po2);
        if (n_mix > 4096) throw Err("internal: accum mix larger than the checkpoint buffer");
        const size_t cp_words = CP_ACCUM_MIX + n_mix;
        if ((words + cp_words) * 4 > out_cap) throw Err("internal: seal larger than the landing buffer sized for max_po2");
        uint32_t* seal_pin = reinterpret_cast<uint32_t*>(out_h);
        uint32_t* cp_pin = seal_pin + words;
        HostRng r0;
        const Digest8 gh = transcript_header(r0, circuit_info, globals, N_GLOBAL, po2);  // host-computed in every transcript mode
        bool chunked = sg.chunked;
        uint32_t round = 0;
        uint32_t* fin = nullptr;
        // Everything that is queued on the stream for this segment.  Runs once per call: plainly, under stream capture, or -- graph
        // replay -- with launches and copies suppressed (dev.replay) so that only the pinned staging area is refilled.
        auto enqueue = [&]() {
        uint32_t* d_seal = arena.take<uint32_t>(words);
        uint32_t* d_cp = arena.take<uint32_t>(CP_WORDS);
        TxState* d_tx = arena.take<TxState>(1);
        TxParams* d_tp = arena.take<TxParams>(1);
        BlindKey* d_key = arena.take<BlindKey>(1);
        h2d_small(d_key, &blind_key, sizeof blind_key);
        // header: the globals are the caller's, so their hash and the RNG state after mixing it are computed here and uploaded
        {
            TxState h{};
            std::memcpy(h.cells, r0.cells, sizeof h.cells);
            h2d_small(d_tx, &h, sizeof h);
            uint32_t head[N_GLOBAL + 1];
            std::memcpy(head, globals, sizeof globals); head[N_GLOBAL] = po2;
            h2d_small(d_seal, head, sizeof head);
        }
        size_t off = N_GLOBAL + 1;
        const MerkleShape ms0((uint32_t)D);
        auto commit = [&](const uint32_t* nd, const MerkleShape& ms, uint32_t cp_off) {
            dev.launch<TxCommitKernel, 32, 1>(1, 1, 32, 0, d_tx, nd, ms.top_size, d_seal + off, d_cp + cp_off);
            off += (size_t)8 * ms.top_size;
        };
        mark(1);
        // CODE
        if (sg.use_control) { mark(2); mark(3); }
        else {
            StageRange r("hfb200:commit_code");
            ntt.lde(tr[GROUP_CODE], N, ev[GROUP_CODE], D, scratch, cd.w_code, (int)po2);
            mark(2);
            merkle.build(ev[GROUP_CODE], D, (uint32_t)D, cd.w_code, nodes[GROUP_CODE]);
            mark(3);
        }
        commit(nodes[GROUP_CODE], ms0, CP_CODE_ROOT);
        // DATA
        {
            StageRange r("hfb200:commit_data");
            lde_data(chunked);
            mark(4);
            merkle.build(ev[GROUP_DATA], D, (uint32_t)D, cd.w_data, nodes[GROUP_DATA]);
            mark(5);
            commit(nodes[GROUP_DATA], ms0, CP_DATA_ROOT);
            dev.launch<TxDrawElemsKernel, 32, 1>(1, 1, 32, 0, d_tx, d_mix, n_mix, d_cp + CP_ACCUM_MIX);
        }
        // ACCUM
        {
            StageRange r("hfb200:commit_accum");
            step_accum(d_key);
            mark(6);
            ntt.lde(tr[GROUP_ACCUM], N, ev[GROUP_ACCUM], D, scratch, cd.w_accum, (int)po2);
            mark(7);
            merkle.build(ev[GROUP_ACCUM], D, (uint32_t)D, cd.w_accum, nodes[GROUP_ACCUM]);
            mark(8);
            commit(nodes[GROUP_ACCUM], ms0, CP_ACCUM_ROOT);
        }
        // check polynomial
        nvtx_push("hfb200:check");
        uint32_t yinv4[4];
        {
            const uint32_t three_n = fpow(THREE, N), w4 = rou_fwd(2);
            uint32_t y = three_n;
            for (int s = 0; s < 4; s++) { yinv4[s] = finv(fsub(y, ONE)); y = fmul(y, w4); }
        }
        {
            const uint32_t nc = cd.n_constraints();
            E4* d_mp = arena.take<E4>(nc);
            dev.launch<TxPolyMixKernel, 32, 1>(1, 1, 32, 0, d_tx, d_tp, d_mp, nc, d_cp + CP_POLY_MIX);
            EvalCheckArgs a{};
            a.ev_accum = ev[GROUP_ACCUM]; a.ev_code = ev[GROUP_CODE]; a.ev_data = ev[GROUP_DATA];
            a.check = check; a.mixpow = d_mp; a.mix = d_mix; a.global0 = 0; a.global0_dev = d_seal;  // seal word 0 = globals[0]
            for (int s_ = 0; s_ < 4; s_++) a.yinv[s_] = yinv4[s_];
            a.po2 = po2; a.cd = cd;
            a.rows_per_block = 128;
            dev.launch<EvalCheckKernel, 128, 1>((unsigned)((D + 127) / 128), 1, 128, (size_t)nc * sizeof(E4) + (size_t)6 * cd.n_free * 2 + 16, a);
        }
        ntt.interpolate(check, D, check, D, 4, (int)po2 + 2, false);
        ntt.expand_evaluate(check, N, ev_check, D, CHECK_SIZE, (int)po2, 2);
        merkle.build(ev_check, D, (uint32_t)D, CHECK_SIZE, nodes_check);
        mark(9);
        commit(nodes_check, ms0, CP_CHECK_ROOT);
        nvtx_pop();
        // DEEP
        nvtx_push("hfb200:deep");
        const uint32_t omega = rou_fwd((int)po2), back_one = finv(omega);
        dev.launch<TxDeepPointKernel, 32, 1>(1, 1, 32, 0, d_tx, d_tp, po2, finv(to_mont((uint32_t)(N % P))), d_cp + CP_Z);
        E4* INV = arena.take<E4>(N); E4* Lw = arena.take<E4>(N); E4* INV4 = arena.take<E4>(N); E4* W4 = arena.take<E4>(N);
        dev.launch<DeepWeightsKernelD, 256, 1>((unsigned)((N + 255) / 256), 1, 256, 0, INV, Lw, INV4, (const TxParams*)d_tp, po2, ntt.rt);
        dev.launch<PowBitrevKernel, 256, 1>((unsigned)((N + 255) / 256), 1, 256, 0, W4, (const E4*)d_tp->xs, po2);
        E4* d_evals = arena.take<E4>((size_t)2 * (W + CHECK_SIZE));
        const uint32_t goff[4] = {0, 2 * cd.w_accum, 2 * (cd.w_accum + cd.w_code), 2 * W};
        for (int g = 0; g < 3; g++) dot_group(tr[g], cir.group_width(g), cir.group_back1(g), Lw, d_evals + goff[g]);
        dot_group(check, CHECK_SIZE, 0, W4, d_evals + goff[3]);
        E4* d_coeff_u = arena.take<E4>(T + CHECK_SIZE);
        E4* d_regmix = arena.take<E4>(W + CHECK_SIZE);
        {
            TxCoeffUArgs a{};
            a.t = d_tx; a.p = d_tp; a.evals = d_evals;
            for (int g = 0; g < 4; g++) a.goff[g] = goff[g];
            for (int g = 0; g < 3; g++) { a.w[g] = cir.group_width(g); a.back1[g] = cir.group_back1(g); }
            a.n_taps = T; a.back_one = back_one; a.coeff_u = d_coeff_u; a.seal_dst = d_seal + off; a.regmix = d_regmix; a.cp = d_cp;
            dev.launch<TxCoeffUKernel, 32, 1>(1, 1, 32, (32 + 32 * 16) * 4, a);
            off += (size_t)4 * (T + CHECK_SIZE);
        }
        uint32_t* S0 = arena.take<uint32_t>(4 * N);
        uint32_t* S1 = arena.take<uint32_t>(4 * N);
        fin = arena.take<uint32_t>(4 * N);
        dev.launch<CheckMixKernel, 256, 1>((unsigned)((N + 255) / 256), 1, 256, 0, (const uint32_t*)check, (const E4*)(d_regmix + W), S0, po2, ntt.rt);
        ntt.expand_evaluate(S0, N, S1, N, 4, (int)po2, 0);
        {
            DeepMixArgs da{};
            da.U0 = da.U1a = da.U1b = da.Vc = e4_zero();
            da.uvec = d_tp->uvec;
            for (int g = 0; g < 3; g++) { da.tr[g] = tr[g]; da.w[g] = cir.group_width(g); da.n_back1[g] = cir.group_back1(g); }
            da.mixpow = d_regmix; da.S = S1; da.INV = INV; da.INV4 = INV4; da.out = fin; da.omega = omega; da.po2 = po2; da.rt = ntt.rt;
            dev.launch<DeepMixKernel, 256, 1>((unsigned)((N + 255) / 256), 1, 256, 0, da);
        }
        ntt.interpolate(fin, N, fin, N, 4, (int)po2, true);
        mark(10);
        nvtx_pop();
        // FRI
        nvtx_push("hfb200:fri");
        std::vector<TxTreeInfo> trees;
        trees.push_back(TxTreeInfo{ev[0], nodes[0], D, (uint32_t)D, cd.w_accum, ms0.top_size, 0});
        trees.push_back(TxTreeInfo{ev[1], nodes[1], D, (uint32_t)D, cd.w_code, ms0.top_size, 0});
        trees.push_back(TxTreeInfo{ev[2], nodes[2], D, (uint32_t)D, cd.w_data, ms0.top_size, 0});
        trees.push_back(TxTreeInfo{ev_check, nodes_check, D, (uint32_t)D, CHECK_SIZE, ms0.top_size, 0});
        uint32_t* coeffs = fin;
        size_t n = N;
        round = 0;
        uint32_t query_words = W + CHECK_SIZE + 4 * ms0.path_words();
        while (n > FRI_MIN_DEGREE) {
            if (round >= TX_MAX_FRI_ROUNDS) throw Err("internal: more FRI rounds than TxParams holds");
            const size_t dom = n * INV_RATE, rows = dom / FRI_FOLD;
            uint32_t* evr = arena.take<uint32_t>(4 * dom);
            uint32_t* ndr = arena.take<uint32_t>(2 * rows * 8);
            ntt.expand_evaluate(coeffs, n, evr, dom, 4, ilog2(n), 2);
            merkle.build(evr, rows, (uint32_t)rows, FRI_FOLD * 4, ndr);
            const MerkleShape mr((uint32_t)rows);
            dev.launch<TxFriCommitKernel, 32, 1>(1, 1, 32, 0, d_tx, d_tp, (const uint32_t*)ndr, mr.top_size, d_seal + off, round, d_cp);
            off += (size_t)8 * mr.top_size;
            uint32_t* out = arena.take<uint32_t>(4 * n / FRI_FOLD);
            dev.launch<FriFoldKernelD, 256, 1>((unsigned)((n / 16 + 255) / 256), 1, 256, 0, (const uint32_t*)coeffs, out, (uint32_t)n, (const E4*)d_tp->fri_mixpow[round]);
            trees.push_back(TxTreeInfo{evr, ndr, rows, (uint32_t)rows, FRI_FOLD * 4, mr.top_size, 0});
            query_words += FRI_FOLD * 4 + mr.path_words();
            coeffs = out;
            n /= FRI_FOLD;
            round++;
        }
        uint32_t* nat = arena.take<uint32_t>(4 * n);
        dev.launch<BitRevKernel, 256, 1>((unsigned)((4 * n + 255) / 256), 1, 256, 0, (const uint32_t*)coeffs, nat, 4u, (uint32_t)ilog2(n));
        {
            TxTreeInfo* d_trees = arena.take<TxTreeInfo>(trees.size());
            h2d_small(d_trees, trees.data(), trees.size() * sizeof(TxTreeInfo));
            const size_t n_desc = (size_t)QUERIES * trees.size();
            OpenDesc* d_descs = arena.take<OpenDesc>(n_desc);
            TxQueriesArgs a{};
            a.t = d_tx; a.p = d_tp; a.final_nat = nat; a.final_words = (uint32_t)(4 * n); a.seal_final = d_seal + off;
            a.trees = d_trees; a.n_main = 4; a.n_rounds = round; a.domain_bits = (uint32_t)ilog2(D); a.descs = d_descs; a.query_words = query_words; a.cp = d_cp;
            dev.launch<TxQueriesKernel, 32, 1>(1, 1, 32, 32 * 4, a);
            off += 4 * n;
            dev.launch<OpenKernel, 128, 1>((unsigned)n_desc, 1, 128, 0, (const OpenDesc*)d_descs, d_seal + off);
            off += (size_t)QUERIES * query_words;
        }
        if (off != words) throw Err("internal: seal layout mismatch");
        mark(11);
        dev.d2h(seal_pin, d_seal, words * 4);
        dev.d2h(cp_pin, d_cp, cp_words * 4);
        nvtx_pop();
        };  // enqueue

        bool as_graph = false;
#ifndef HFB200_EMU
        if (graph_replay()) {
            GraphEntry& ge = graphs[(uint64_t)po2 * 2 + (sg.use_control ? 1 : 0)];
            if (ge.state == 0) ge.state = 1;  // first segment of this shape: plain run below (module loading, attribute set-up)
            else {
                as_graph = true;
                // trace uploads stay outside the graph: the graph's first node follows the last slice in stream order
                if (chunked) { CUDA_CHECK(cudaStreamWaitEvent(dev.stream, chunk_ev[H2D_CHUNKS - 1], 0)); chunked = false; }
                marks_off = true;
                try {
                    if (ge.state == 1) {
                        CUDA_CHECK(cudaStreamBeginCapture(dev.stream, cudaStreamCaptureModeThreadLocal));
                        cudaGraph_t g = nullptr;
                        try { enqueue(); }
                        catch (...) { cudaStreamEndCapture(dev.stream, &g); if (g) cudaGraphDestroy(g); throw; }
                        CUDA_CHECK(cudaStreamEndCapture(dev.stream, &g));
                        const cudaError_t e = cudaGraphInstantiate(&ge.exec, g, 0);
                        cudaGraphDestroy(g);
                        CUDA_CHECK(e);
                        ge.state = 2;
                    } else {
                        dev.replay = true;
                        try { enqueue(); } catch (...) { dev.replay = false; throw; }
                        dev.replay = false;
                    }
                } catch (...) { marks_off = false; throw; }
                marks_off = false;
                mark(1);
                CUDA_CHECK(cudaGraphLaunch(ge.exec, dev.stream));
                mark(11);
                graph_launches++;
            }
        }
#endif
        if (!as_graph) enqueue();
        std::vector<uint32_t> fc;
        if (debug_checkpoints) { fc.resize(4 * N); dev.d2h(fc.data(), fin, fc.size() * 4); }
        sync();  // the only synchronisation of the segment
        seal_out.assign(seal_pin, seal_pin + words);
        std::vector<uint32_t> cp(cp_pin, cp_pin + cp_words);
        // checkpoints, under the names of the host-transcript path
        cp_add("globals_hash", gh.w, 8);
        cp_add("code_root", &cp[CP_CODE_ROOT], 8); cp_add("data_root", &cp[CP_DATA_ROOT], 8);
        cp_add("accum_mix", &cp[CP_ACCUM_MIX], n_mix);
        cp_add("accum_root", &cp[CP_ACCUM_ROOT], 8); cp_add("poly_mix", &cp[CP_POLY_MIX], 4); cp_add("check_root", &cp[CP_CHECK_ROOT], 8);
        cp_add("z", &cp[CP_Z], 4); cp_add("hash_u", &cp[CP_HASH_U], 8); cp_add("deep_mix", &cp[CP_DEEP_MIX], 4);
        if (debug_checkpoints) { const Digest8 d = host_hash_elems(fc.data(), fc.size()); cp_add("final_poly_hash", d.w, 8); }
        for (uint32_t r = 0; r < round; r++) { cp_add("fri_root_" + std::to_string(r), &cp[CP_FRI_ROOT0 + 8 * r], 8); cp_add("fri_mix_" + std::to_string(r), &cp[CP_FRI_MIX0 + 4 * r], 4); }
        cp_add("fri_final_hash", &cp[CP_FRI_FINAL_HASH], 8);
        cp_add("query_positions", &cp[CP_POSITIONS], QUERIES);
        mix.assign(cp.begin() + CP_ACCUM_MIX, cp.begin() + CP_ACCUM_MIX + n_mix);
        stage_ms[0] = between(0, 1);
        if (!as_graph) {  // a replayed graph has no stage events inside it: only the upload and the whole-segment time are known
            stage_ms[1] = between(1, 2) + between(3, 4) + between(6, 7);
            stage_ms[2] = between(2, 3) + between(4, 5) + between(7, 8);
            stage_ms[3] = between(5, 6);
            stage_ms[4] = between(8, 9); stage_ms[5] = between(9, 10); stage_ms[6] = between(10, 11);
        }
        stats.ms_h2d = stage_ms[0]; stats.ms_ntt_main = stage_ms[1]; stats.ms_hash_main = stage_ms[2]; stats.ms_accum = stage_ms[3];
        stats.ms_check = stage_ms[4]; stats.ms_deep = stage_ms[5]; stats.ms_fri = stage_ms[6];
        stats.ms_device = between(0, 11);
        stats.ms_total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        stats.launches = dev.launches - launches_at_begin;
        stats.ntt_main_bytes = 28ull * W * N;
        stats.host_syncs = host_syncs - host_syncs_at_begin;
        emit_metrics();
    }

    // between segments: a different suite commits the control columns to a different root, so the resident group is dropped
    void set_hash_suite(int s) {
        if (!hash_suite_valid(s)) throw Err("hash suite must be HFB200_HASH_POSEIDON2 (0) or HFB200_HASH_SHA256 (1)");
        if (begun) throw Err("a segment is in flight");
        if (s == HASH_SHA256 && transcript_mode >= 1)
            throw Err("the SHA-256 suite runs the host transcript only (this context is in device transcript mode " + std::to_string(transcript_mode) + ")");
        if (s != hash_suite) { control_cached = false; control_gen = 0; }
        hash_suite = s;
        merkle.suite = s;
    }

    void witgen(uint32_t p, uint64_t trace_seed, uint64_t blind, uint32_t* globals_out) {
        if (gen.active) throw Err("hfb200_witgen_synth: only for the built-in synthetic circuit");
        bind();
        layout(p);
        control_cached = false; control_gen = 0;  // the resident control columns are overwritten below
        const size_t N = (size_t)1 << po2;
        for (uint32_t i = 0; i < N_GLOBAL; i++) globals_out[i] = synth_value(trace_seed ^ 0x676C6F62ull, 0xFFFFu, i);
        std::memcpy(globals, globals_out, sizeof globals);
        const CircuitDev& cd = cir.cd;
        dev.launch<GenCodeKernel, 256, 1>((unsigned)(((size_t)cd.w_code * N + 255) / 256), 1, 256, 0, tr[GROUP_CODE], cd.w_code, po2);
        dev.launch<GenFreeKernel, 256, 1>((unsigned)(((size_t)cd.w_data * N + 255) / 256), 1, 256, 0, tr[GROUP_DATA], cd, po2, trace_seed, make_blind_key(blind), globals_out[0]);
        dev.launch<GenDerivedKernel, 256, 1>((unsigned)(((size_t)cd.n_free * N + 255) / 256), 1, 256, 0, tr[GROUP_DATA], (const uint32_t*)tr[GROUP_CODE], cd, po2);
        dev.sync();
        have_trace = true;
    }

    size_t seal_words(uint32_t p) const {
        const size_t W = cir.n_regs(), T = cir.n_taps;
        size_t n = (size_t)1 << p;
        const MerkleShape m0((uint32_t)(4 * n));
        size_t words = N_GLOBAL + 1 + 4 * 8 * m0.top_size + 4 * (T + CHECK_SIZE);
        size_t per_query = W + CHECK_SIZE + 4 * m0.path_words();
        while (n > FRI_MIN_DEGREE) {
            const MerkleShape mr((uint32_t)(4 * n / FRI_FOLD));
            words += 8 * mr.top_size;
            per_query += 64 + mr.path_words();
            n /= FRI_FOLD;
        }
        return words + 4 * n + QUERIES * per_query;
    }
};

}  // namespace hf
