// eval_check of a DATA-DEFINED circuit as a run-time specialised sm_100a kernel.
//
// Upstream turns the constraint IR (`risc0_zkp::adapter::PolyExtStepDef`) into generated C++/CUDA at crate build time
// (risc0-circuit-rv32im-sys `eval_check.cu`; /root/reference/Cargo.lock:3121-3132, not vendored).  Here the circuit
// arrives as data (`hfb200_init_ir`), so the same specialisation happens when the circuit is registered: the
// slot-allocated bytecode of `GenericCircuitHost` is printed as straight-line CUDA (one thread per LDE row, every value a
// register, constraint sums in the lazy 64-bit accumulators of field.cuh), compiled for sm_100a with NVRTC and loaded
// through the runtime's library API.  Each specialisation is compiled once per process (JitCache below), or not at all on a
// host that loads a prebuilt bundle (hfb200_ir_compile / hfb200_ir_load_kernels, the counterpart of upstream's build-time
// compile).  The interpreter kernel (`GenEvalCheckKernel`) stays as the path for a size that is neither cached nor compilable
// (no libnvrtc) and as the cross-check in the tests (HFB200_IR_JIT=0 selects it for every size).
#pragma once
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <string>
#include <thread>
#include "circuit.cuh"
#include "poseidon2.cuh"

#ifndef HFB200_EMU
#include <dlfcn.h>
#include <nvrtc.h>
#endif

namespace hf {

struct JitEvalArgs {
    const uint32_t* ev[3];   // accum, code, data LDEs [w][domain]
    uint32_t* check;         // [4][domain]
    const E4* mixpow;        // poly_mix^k (device)
    const uint32_t* mix;     // accum mix (device)
    const uint32_t* globals; // device copy of the 32 globals
    uint32_t yinv[4];
    uint32_t po2;
};

static const char* const JIT_PRELUDE = R"JIT(
typedef unsigned int uint32_t;
typedef unsigned long long uint64_t;
#define FI __device__ __forceinline__
static constexpr uint32_t P = 2013265921u, P_INV = 0x88000001u, ONE = 268435454u, NBETA = 1073741848u;
FI uint32_t umin32(uint32_t a, uint32_t b) { return a < b ? a : b; }
FI uint32_t fadd(uint32_t a, uint32_t b) { uint32_t x = a + b; return umin32(x, x - P); }
FI uint32_t fsub(uint32_t a, uint32_t b) { uint32_t x = a - b; return umin32(x, x + P); }
FI uint32_t fmul(uint32_t a, uint32_t b) {
    uint64_t o = (uint64_t)a * b; uint32_t m = (uint32_t)o * P_INV; uint32_t r = (uint32_t)(o >> 32) - __umulhi(m, P); return umin32(r, r + P);
}
struct __align__(16) E4 { uint32_t c[4]; };
FI E4 e4_scale(const E4& a, uint32_t s) { E4 r; r.c[0] = fmul(a.c[0], s); r.c[1] = fmul(a.c[1], s); r.c[2] = fmul(a.c[2], s); r.c[3] = fmul(a.c[3], s); return r; }
FI E4 e4_mul(const E4& a, const E4& b) {
    uint32_t a0 = a.c[0], a1 = a.c[1], a2 = a.c[2], a3 = a.c[3], b0 = b.c[0], b1 = b.c[1], b2 = b.c[2], b3 = b.c[3];
    uint32_t t0 = fadd(fadd(fmul(a1, b3), fmul(a2, b2)), fmul(a3, b1));
    uint32_t t1 = fadd(fmul(a2, b3), fmul(a3, b2));
    uint32_t t2 = fmul(a3, b3);
    E4 r;
    r.c[0] = fadd(fmul(a0, b0), fmul(NBETA, t0));
    r.c[1] = fadd(fadd(fmul(a0, b1), fmul(a1, b0)), fmul(NBETA, t1));
    r.c[2] = fadd(fadd(fadd(fmul(a0, b2), fmul(a1, b1)), fmul(a2, b0)), fmul(NBETA, t2));
    r.c[3] = fadd(fadd(fmul(a0, b3), fmul(a1, b2)), fadd(fmul(a2, b1), fmul(a3, b0)));
    return r;
}
struct A64 { uint32_t lo, hi; };
FI void mac(A64& a, uint32_t x, uint32_t y) {
    const uint64_t t = (uint64_t)x * y + (((uint64_t)a.hi << 32) | a.lo);
    const uint32_t h = (uint32_t)(t >> 32); a.lo = (uint32_t)t; a.hi = umin32(h, h - P);
}
FI uint32_t redc(const A64& a) { const uint32_t m = a.lo * P_INV; const uint32_t r = a.hi - __umulhi(m, P); return umin32(r, r + P); }
struct E4A { A64 c[4]; };
FI E4A e4a_zero() { E4A a; for (int k = 0; k < 4; k++) { a.c[k].lo = 0; a.c[k].hi = 0; } return a; }
FI void e4a_mac(E4A& a, const E4& w, uint32_t t) { mac(a.c[0], w.c[0], t); mac(a.c[1], w.c[1], t); mac(a.c[2], w.c[2], t); mac(a.c[3], w.c[3], t); }
FI void e4a_add(E4A& a, const E4& t) { mac(a.c[0], t.c[0], ONE); mac(a.c[1], t.c[1], ONE); mac(a.c[2], t.c[2], ONE); mac(a.c[3], t.c[3], ONE); }
FI E4 e4a_redc(const E4A& a) { E4 r; r.c[0] = redc(a.c[0]); r.c[1] = redc(a.c[1]); r.c[2] = redc(a.c[2]); r.c[3] = redc(a.c[3]); return r; }
struct JitEvalArgs { const uint32_t* ev[3]; uint32_t* check; const E4* mixpow; const uint32_t* mix; const uint32_t* globals; uint32_t yinv[4]; uint32_t po2; };
)JIT";

#ifndef JIT_FENCE_EVERY
#define JIT_FENCE_EVERY 2u
#endif
// straight-line CUDA for the bytecode of chunk `k` of one circuit (kernel hfb200_eval_check_jit_<k>); chunk 0 stores its partial
// sum (times 1 / Z), the others add theirs
// The kernel is specialised for the segment size as well: with `domain` a literal, a tap read is `ev[<column * domain> + row_b]` -- a
// constant offset from four row indices.  With `domain` a run-time value ptxas treats every `column * domain` product as a common
// subexpression worth keeping (hundreds of 64-bit values per chunk): 3 KB of spills per thread and ~50 s of compile time per chunk.
static inline std::string jit_kernel_source(const GenericCircuitHost& g, size_t k, uint32_t po2) {
    const GenericCircuitHost::Chunk& c = g.chunks[k];
    const uint64_t domain = 4ull << po2;
    std::string s;
    // tuning knobs of the generated code (experiments: profiles/r2_ir_scale.txt)
    static const int minb = [] { const char* e = std::getenv("HFB200_IR_JIT_MINB"); const int v = e ? std::atoi(e) : 4; return v >= 1 && v <= 8 ? v : 4; }();
    static const uint32_t fence_every = [] { const char* e = std::getenv("HFB200_IR_JIT_FENCE"); const int v = e ? std::atoi(e) : (int)JIT_FENCE_EVERY; return (uint32_t)(v >= 0 ? v : 2); }();
    s += "extern \"C\" __global__ void __launch_bounds__(128, " + std::to_string(minb) + ") hfb200_eval_check_jit_" + std::to_string(k) + "(JitEvalArgs p) {\n";
    s += "  const uint64_t domain = " + std::to_string(domain) + "ull, dmask = domain - 1ull;\n";
    s += "  if (p.po2 != " + std::to_string(po2) + "u) return;\n";
    s += "  const uint32_t* __restrict__ ev0 = p.ev[0]; const uint32_t* __restrict__ ev1 = p.ev[1]; const uint32_t* __restrict__ ev2 = p.ev[2];\n";
    // grid-stride loop over the rows: the straight-line body is executed many times by every warp, so its instructions come from the
    // instruction cache instead of being streamed from L2 once per warp (what bounds a one-row-per-thread kernel of this size)
    s += "  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < domain; i += (uint64_t)gridDim.x * blockDim.x) {\n";
    for (uint32_t b : g.backs) s += "  const uint64_t r" + std::to_string(b) + " = (i + domain - " + std::to_string(4ull * b) + "ull) & dmask;\n";
    // q<b>: the row indices the loads actually use; made opaque again at every fence so that ptxas cannot keep the ADDRESS of a tap
    // read in a register pair until the same tap is read again hundreds of steps later (that alone was ~450 live values per chunk)
    std::string reopaque;
    for (uint32_t b : g.backs) { s += "  uint64_t q" + std::to_string(b) + " = r" + std::to_string(b) + ";\n"; reopaque += "  q" + std::to_string(b) + " = r" + std::to_string(b) + "; asm volatile(\"\" : \"+l\"(q" + std::to_string(b) + "));\n"; }
    for (uint32_t q = 0; q < c.n_fp_slots; q++) s += "  uint32_t f" + std::to_string(q) + " = 0;\n";
    for (uint32_t q = 0; q < c.n_mix_slots; q++) s += "  E4A m" + std::to_string(q) + " = e4a_zero();\n";
    auto F = [](uint32_t q) { return "f" + std::to_string(q); };
    auto M = [](uint32_t q) { return "m" + std::to_string(q); };
    uint32_t since_fence = 0;
    for (const BcIns& ins : c.prog) {
        const std::string d = std::to_string(ins.dst);
        // a compiler-level memory fence after every few constraints: without it ptxas hoists the (independent) loads of a whole
        // chunk -- hundreds of tap reads and mix powers -- to the top of the kernel and spills them (3 KB of stack per thread,
        // 50 s of compile time per chunk); latency is hidden by the other warps of the SM, not by this thread's own loads
        if (fence_every && (ins.op == BC_MEQZ || ins.op == BC_MCOND) && ++since_fence >= fence_every) { s += "  asm volatile(\"\" ::: \"memory\");\n" + reopaque; since_fence = 0; }
        switch (ins.op) {
            case BC_CONST: s += "  f" + d + " = " + std::to_string(ins.a) + "u;\n"; break;
            case BC_GET:
                s += "  f" + d + " = ev" + std::to_string(ins.a) + "[" + std::to_string((uint64_t)ins.b * domain) + "ull + q" + std::to_string(ins.c) + "];\n";
                break;
            case BC_GETG: s += "  f" + d + " = " + (ins.a == 0 ? "p.globals[" : "p.mix[") + std::to_string(ins.b) + "];\n"; break;
            case BC_ADD: s += "  f" + d + " = fadd(" + F(ins.a) + ", " + F(ins.b) + ");\n"; break;
            case BC_SUB: s += "  f" + d + " = fsub(" + F(ins.a) + ", " + F(ins.b) + ");\n"; break;
            case BC_MUL: s += "  f" + d + " = fmul(" + F(ins.a) + ", " + F(ins.b) + ");\n"; break;
            case BC_MTRUE: s += "  m" + d + " = e4a_zero();\n"; break;
            case BC_MEQZ:
                if (ins.dst != ins.a) s += "  m" + d + " = " + M(ins.a) + ";\n";
                s += "  e4a_mac(m" + d + ", p.mixpow[" + std::to_string(ins.c) + "], " + F(ins.b) + ");\n";
                break;
            default:  // BC_MCOND: tot = x.tot + cond * inner.tot * mix^k
                s += "  { const E4 t_ = e4_scale(e4_mul(e4a_redc(" + M(ins.b >> 16) + "), p.mixpow[" + std::to_string(ins.c) + "]), " + F(ins.b & 0xFFFFu) + "); E4A x_ = " + M(ins.a) +
                     "; e4a_add(x_, t_); m" + d + " = x_; }\n";
                break;
        }
    }
    s += "  const E4 tot = e4a_redc(m" + std::to_string(c.ret_slot) + ");\n  const uint32_t yi = p.yinv[i & 3];\n";
    if (k == 0) s += "  for (int k = 0; k < 4; k++) p.check[(uint64_t)k * domain + i] = fmul(tot.c[k], yi);\n  }\n}\n";
    else s += "  for (int k = 0; k < 4; k++) p.check[(uint64_t)k * domain + i] = fadd(p.check[(uint64_t)k * domain + i], fmul(tot.c[k], yi));\n  }\n}\n";
    return s;
}
// every chunk kernel in one translation unit (hfb200_ir_source; the library itself compiles one unit per chunk, in parallel)
static inline std::string jit_source(const GenericCircuitHost& g, uint32_t po2 = 20) {
    std::string s = JIT_PRELUDE;
    for (size_t k = 0; k < g.chunks.size(); k++) s += jit_kernel_source(g, k, po2);
    return s;
}

#ifndef HFB200_EMU
struct NvrtcApi {
    void* h = nullptr;
    std::string why;  // why the last load() failed
    nvrtcResult (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    nvrtcResult (*CompileProgram)(nvrtcProgram, int, const char* const*) = nullptr;
    nvrtcResult (*GetCUBINSize)(nvrtcProgram, size_t*) = nullptr;
    nvrtcResult (*GetCUBIN)(nvrtcProgram, char*) = nullptr;
    nvrtcResult (*GetProgramLogSize)(nvrtcProgram, size_t*) = nullptr;
    nvrtcResult (*GetProgramLog)(nvrtcProgram, char*) = nullptr;
    nvrtcResult (*DestroyProgram)(nvrtcProgram*) = nullptr;
    bool load() {
        if (h) return true;
        // HFB200_NVRTC_LIB=<path>: that library only (a toolkit installed elsewhere), in place of the search list
        const char* given = std::getenv("HFB200_NVRTC_LIB");
        std::vector<std::string> names;
        if (given) names.push_back(given);
        else names = {"libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so"};
        for (const std::string& n : names) { h = dlopen(n.c_str(), RTLD_NOW | RTLD_LOCAL); if (h) break; }
        if (!h) { why = given ? std::string(given) + " (HFB200_NVRTC_LIB) not found" : "libnvrtc.so.12 not found"; return false; }
        bool ok = true;
        auto sym = [&](auto& fn, const char* name) { fn = reinterpret_cast<std::decay_t<decltype(fn)>>(dlsym(h, name)); ok = ok && fn != nullptr; };
        sym(CreateProgram, "nvrtcCreateProgram"); sym(CompileProgram, "nvrtcCompileProgram"); sym(GetCUBINSize, "nvrtcGetCUBINSize");
        sym(GetCUBIN, "nvrtcGetCUBIN"); sym(GetProgramLogSize, "nvrtcGetProgramLogSize"); sym(GetProgramLog, "nvrtcGetProgramLog");
        sym(DestroyProgram, "nvrtcDestroyProgram");
        if (!ok) { dlclose(h); h = nullptr; why = "the NVRTC library lacks the entry points used here"; }
        return ok;
    }
};

// ---- process-wide cache of the specialised cubins ---------------------------------------------------------------------------
// A chunk program is keyed by the Poseidon2 byte digest (host_digest_bytes, as hfb200_digest_bytes) of its whole NVRTC input:
// the options, the prelude and the kernel source.  The source spells out everything that shapes the code -- the circuit's
// bytecode, the po2, the chunking (HFB200_IR_CHUNK), HFB200_IR_JIT_MINB and HFB200_IR_JIT_FENCE -- so a key never matches code
// generated differently.  The cache holds cubin bytes: every context still loads its own cudaLibrary_t's from them, so library
// lifetime and fault handling stay per context.  It is filled by contexts (JitEvalCheck::ensure), ahead of time by
// hfb200_ir_compile, and from a serialised bundle by hfb200_ir_load_kernels.
static const char* const JIT_OPTIONS[] = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo"};
static constexpr int JIT_N_OPTIONS = 3;
static constexpr char JIT_ARCH[] = "sm_100a";

struct JitKey {
    uint32_t w[8];
    bool operator<(const JitKey& o) const { return std::memcmp(w, o.w, sizeof w) < 0; }
};
using JitCubin = std::shared_ptr<const std::vector<char>>;

// one specialisation: the NVRTC input of every chunk of one (circuit, po2), and its keys
struct JitSpec {
    uint32_t po2 = 0;
    std::vector<std::string> text;  // prelude + kernel source of chunk k
    std::vector<JitKey> keys;
};

// threads = 0: up to 8 (and no more than there is work)
static inline unsigned jit_threads(unsigned requested, size_t work) {
    unsigned n = requested;
    if (n == 0) { n = std::thread::hardware_concurrency(); n = std::min(std::max(n, 1u), 8u); }
    return (unsigned)std::max<size_t>(1, std::min<size_t>(n, work));
}
// f(0) .. f(n - 1) on `threads` host threads, this one included; f must not throw
template <class F> static void jit_parallel(size_t n, unsigned threads, F&& f) {
    std::atomic<size_t> next{0};
    auto work = [&] { for (size_t i = next.fetch_add(1); i < n; i = next.fetch_add(1)) f(i); };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < threads; t++) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
}
static inline JitKey jit_key(const std::string& text) {
    std::string in;
    for (const char* o : JIT_OPTIONS) { in += o; in += '\n'; }
    in += '\0';
    in += text;
    const Digest8 d = host_digest_bytes(reinterpret_cast<const uint8_t*>(in.data()), in.size());
    JitKey k;
    std::memcpy(k.w, d.w, sizeof k.w);
    return k;
}
static inline JitSpec jit_spec(const GenericCircuitHost& g, uint32_t po2, unsigned threads) {
    JitSpec s;
    s.po2 = po2;
    const size_t K = g.chunks.size();
    s.text.resize(K);
    s.keys.resize(K);
    jit_parallel(K, jit_threads(threads, K), [&](size_t k) {
        s.text[k] = std::string(JIT_PRELUDE) + jit_kernel_source(g, k, po2);
        s.keys[k] = jit_key(s.text[k]);
    });
    return s;
}

struct JitCache {
    std::mutex mu;
    std::condition_variable cv;
    std::map<JitKey, JitCubin> cubins;
    std::set<JitKey> compiling;        // keys some thread is compiling now: the others wait for it (single flight)
    std::atomic<uint64_t> programs{0};  // NVRTC programs compiled by this process (hfb200_ir_nvrtc_programs)
    NvrtcApi api;

    static JitCache& get() { static JitCache c; return c; }
    // loads NVRTC on first use; only a compile needs it
    bool nvrtc(std::string* why = nullptr) {
        std::lock_guard<std::mutex> lock(mu);
        if (api.load()) return true;
        if (why) *why = api.why;
        return false;
    }
    // one NVRTC program; returns "" or the error
    std::string compile(const std::string& text, size_t k, std::vector<char>& cubin) {
        nvrtcProgram prog = nullptr;
        if (api.CreateProgram(&prog, text.c_str(), "hfb200_eval_check_jit.cu", 0, nullptr, nullptr) != NVRTC_SUCCESS) return "nvrtcCreateProgram failed";
        programs++;
        if (api.CompileProgram(prog, JIT_N_OPTIONS, JIT_OPTIONS) != NVRTC_SUCCESS) {
            size_t n = 0; api.GetProgramLogSize(prog, &n);
            std::string log(n, '\0'); if (n) api.GetProgramLog(prog, &log[0]);
            api.DestroyProgram(&prog);
            return "NVRTC compilation of eval_check chunk " + std::to_string(k) + " failed: " + log.substr(0, 2000);
        }
        size_t nb = 0; api.GetCUBINSize(prog, &nb);
        cubin.resize(nb);
        api.GetCUBIN(prog, cubin.data());
        api.DestroyProgram(&prog);
        return "";
    }
    // The cubins of s's chunks: cached ones as they are, the others compiled here on `threads` threads.  A key that another
    // thread is compiling is waited for, not compiled twice.  A failed compile is not cached: it throws here, and the next
    // caller of that key compiles it again.  Without NVRTC the chunks that are not cached come back empty.
    std::vector<JitCubin> fetch(const JitSpec& s, unsigned threads) {
        const size_t K = s.keys.size();
        std::vector<JitCubin> out(K);
        std::vector<size_t> todo(K);
        for (size_t k = 0; k < K; k++) todo[k] = k;
        while (!todo.empty()) {
            std::vector<size_t> mine, theirs;
            {
                std::lock_guard<std::mutex> lock(mu);
                for (size_t k : todo) {
                    const auto it = cubins.find(s.keys[k]);
                    if (it != cubins.end()) out[k] = it->second;
                    else if (compiling.count(s.keys[k])) theirs.push_back(k);
                    else { compiling.insert(s.keys[k]); mine.push_back(k); }
                }
            }
            todo.clear();
            if (!mine.empty()) {
                const bool have = nvrtc();
                std::vector<std::string> errors(mine.size());
                jit_parallel(mine.size(), have ? jit_threads(threads, mine.size()) : 1, [&](size_t i) {
                    const size_t k = mine[i];
                    std::shared_ptr<std::vector<char>> bin;
                    if (have) {
                        try { bin = std::make_shared<std::vector<char>>(); errors[i] = compile(s.text[k], k, *bin); }
                        catch (const std::exception& e) { errors[i] = e.what(); }
                        if (!errors[i].empty()) bin.reset();
                    }
                    std::lock_guard<std::mutex> lock(mu);
                    if (bin) cubins.emplace(s.keys[k], bin);
                    compiling.erase(s.keys[k]);
                    out[k] = bin;
                    cv.notify_all();
                });
                for (const std::string& e : errors) if (!e.empty()) throw Err("data-defined circuit: " + e);
            }
            if (!theirs.empty()) {
                std::unique_lock<std::mutex> lock(mu);
                for (size_t k : theirs) {
                    cv.wait(lock, [&] { return compiling.count(s.keys[k]) == 0; });
                    const auto it = cubins.find(s.keys[k]);
                    if (it != cubins.end()) out[k] = it->second;
                    else todo.push_back(k);  // that compile failed (or found no NVRTC): try it here
                }
            }
        }
        return out;
    }
    // adds records (never replaces one: a key names its code); returns how many were new
    size_t add(const std::vector<std::pair<JitKey, JitCubin>>& recs) {
        std::lock_guard<std::mutex> lock(mu);
        size_t n = 0;
        for (const auto& r : recs) n += cubins.emplace(r.first, r.second).second ? 1 : 0;
        return n;
    }
};

// ---- kernel bundles (hfb200_ir_compile -> caller's storage -> hfb200_ir_load_kernels) -------------------------------------
// Little-endian:  magic "HFB200KB" | u32 version | u32 arch length | arch ("sm_100a") | u32 specialisations |
//                 per specialisation: u32 po2 | u32 chunks | per chunk: key (32 bytes) | u64 cubin bytes | cubin |
//                 digest (32 bytes)
// The digest is host_digest_bytes of everything before it with every cubin replaced by its own host_digest_bytes (so the
// cubins, most of the bytes, are hashed in parallel).  A bundle is refused whole unless every check passes.
static constexpr char JIT_BUNDLE_MAGIC[8] = {'H', 'F', 'B', '2', '0', '0', 'K', 'B'};
static constexpr uint32_t JIT_BUNDLE_VERSION = 1;

struct JitBundleWriter {
    std::string out, meta;  // the bundle, and the digest's input
    void put(const void* p, size_t n) { out.append((const char*)p, n); meta.append((const char*)p, n); }
    void u32(uint32_t v) { put(&v, 4); }
    void u64(uint64_t v) { put(&v, 8); }
};
static inline std::vector<Digest8> jit_cubin_digests(const std::vector<const std::vector<char>*>& bins, unsigned threads) {
    std::vector<Digest8> d(bins.size());
    jit_parallel(bins.size(), jit_threads(threads, bins.size()),
                 [&](size_t i) { d[i] = host_digest_bytes(reinterpret_cast<const uint8_t*>(bins[i]->data()), bins[i]->size()); });
    return d;
}
static inline std::string jit_bundle(const std::vector<JitSpec>& specs, const std::vector<std::vector<JitCubin>>& bins, unsigned threads) {
    std::vector<const std::vector<char>*> flat;
    for (const auto& v : bins) for (const JitCubin& b : v) flat.push_back(b.get());
    const std::vector<Digest8> dig = jit_cubin_digests(flat, threads);
    JitBundleWriter w;
    w.put(JIT_BUNDLE_MAGIC, 8);
    w.u32(JIT_BUNDLE_VERSION);
    w.u32((uint32_t)std::strlen(JIT_ARCH));
    w.put(JIT_ARCH, std::strlen(JIT_ARCH));
    w.u32((uint32_t)specs.size());
    size_t f = 0;
    for (size_t i = 0; i < specs.size(); i++) {
        w.u32(specs[i].po2);
        w.u32((uint32_t)specs[i].keys.size());
        for (size_t k = 0; k < specs[i].keys.size(); k++, f++) {
            w.put(specs[i].keys[k].w, 32);
            w.u64(flat[f]->size());
            w.out.append(flat[f]->data(), flat[f]->size());
            w.meta.append((const char*)dig[f].w, 32);
        }
    }
    const Digest8 d = host_digest_bytes(reinterpret_cast<const uint8_t*>(w.meta.data()), w.meta.size());
    w.out.append((const char*)d.w, 32);
    return w.out;
}
// parses and checks a bundle; returns its records and (via *specs) the number of specialisations.  Throws on any defect.
static inline std::vector<std::pair<JitKey, JitCubin>> jit_parse_bundle(const uint8_t* b, size_t n, size_t* specs) {
    const char* fn = "hfb200_ir_load_kernels: ";
    size_t at = 0;
    auto take = [&](void* dst, size_t len) {
        if (len > n - at) throw Err(std::string(fn) + "bundle truncated");
        std::memcpy(dst, b + at, len);
        at += len;
    };
    auto u32 = [&] { uint32_t v; take(&v, 4); return v; };
    char magic[8];
    take(magic, 8);
    if (std::memcmp(magic, JIT_BUNDLE_MAGIC, 8) != 0) throw Err(std::string(fn) + "not an eval_check kernel bundle (bad magic)");
    const uint32_t version = u32();
    if (version != JIT_BUNDLE_VERSION) throw Err(std::string(fn) + "bundle format version " + std::to_string(version) + ", this library reads " + std::to_string(JIT_BUNDLE_VERSION));
    const uint32_t arch_len = u32();
    if (arch_len > 64) throw Err(std::string(fn) + "bundle header is malformed");
    std::string arch(arch_len, '\0');
    take(&arch[0], arch_len);
    if (arch != JIT_ARCH) throw Err(std::string(fn) + "bundle holds kernels for " + arch + ", this library runs " + JIT_ARCH);
    const uint32_t n_specs = u32();
    std::vector<std::pair<JitKey, JitCubin>> recs;
    std::vector<std::pair<size_t, size_t>> spans;  // cubin offset, length
    std::vector<size_t> slots;                     // where each cubin's digest goes in `meta`
    std::string meta(reinterpret_cast<const char*>(b), at);
    for (uint32_t i = 0; i < n_specs; i++) {
        const size_t s0 = at;
        const uint32_t po2 = u32(), chunks = u32();
        if (po2 < 12 || po2 > 22 || chunks == 0) throw Err(std::string(fn) + "bundle record is malformed");
        meta.append(reinterpret_cast<const char*>(b + s0), at - s0);
        for (uint32_t k = 0; k < chunks; k++) {
            const size_t r0 = at;
            JitKey key;
            take(key.w, 32);
            uint64_t len;
            take(&len, 8);
            if (len > n - at) throw Err(std::string(fn) + "bundle truncated");
            meta.append(reinterpret_cast<const char*>(b + r0), at - r0);
            recs.emplace_back(key, nullptr);
            spans.emplace_back(at, (size_t)len);
            at += (size_t)len;
            slots.push_back(meta.size());
            meta.append(32, '\0');  // the cubin's digest, filled in below
        }
    }
    if (n - at != 32) throw Err(std::string(fn) + (n - at < 32 ? "bundle truncated" : "bundle has trailing bytes"));
    std::vector<std::vector<char>> bins(spans.size());
    std::vector<const std::vector<char>*> ptrs(spans.size());
    for (size_t i = 0; i < spans.size(); i++) {
        bins[i].assign(b + spans[i].first, b + spans[i].first + spans[i].second);
        ptrs[i] = &bins[i];
    }
    const std::vector<Digest8> dig = jit_cubin_digests(ptrs, 0);
    for (size_t i = 0; i < slots.size(); i++) std::memcpy(&meta[slots[i]], dig[i].w, 32);
    const Digest8 d = host_digest_bytes(reinterpret_cast<const uint8_t*>(meta.data()), meta.size());
    if (std::memcmp(d.w, b + at, 32) != 0) throw Err(std::string(fn) + "bundle digest does not match its contents (corrupted)");
    for (size_t i = 0; i < recs.size(); i++) recs[i].second = std::make_shared<const std::vector<char>>(std::move(bins[i]));
    if (specs) *specs = n_specs;
    return recs;
}

struct JitEvalCheck {
    struct Compiled { std::vector<cudaLibrary_t> libs; std::vector<cudaKernel_t> kernels; };  // one kernel per chunk, launched in order
    std::map<uint32_t, Compiled> by_po2;  // sizes whose specialised kernels this context has loaded (max_po2 at init, others on first use)
    std::set<uint32_t> interp_po2;        // sizes that run the interpreter kernel: not in the cache, and NVRTC unavailable
    const GenericCircuitHost* g = nullptr;
    bool enabled = false;  // HFB200_IR_JIT is not 0
    bool ready = false;    // specialised kernels for the context's max_po2 (hfb200_ir_jit_active)
    std::string note;      // why they are not (empty when ready)
    float compile_ms = 0;  // the most recent specialisation: sources + cache lookup + NVRTC for the misses + load

    void init(const GenericCircuitHost& gen, uint32_t first_po2) {
        if (const char* env = std::getenv("HFB200_IR_JIT")) if (std::atoi(env) == 0) { note = "disabled by HFB200_IR_JIT=0"; return; }
        g = &gen;
        enabled = true;
        ready = ensure(first_po2);
        if (!ready) {
            std::string why;
            JitCache::get().nvrtc(&why);
            note = "eval_check kernels for po2 " + std::to_string(first_po2) + " are not cached and NVRTC is unavailable: " + why;
        }
    }
    // true: po2 runs the specialised kernels (loaded now if this is the first segment of that size); false: the interpreter
    bool ensure(uint32_t po2) {
        if (!enabled) return false;
        if (by_po2.count(po2)) return true;
        if (interp_po2.count(po2)) return false;
        const auto t0 = std::chrono::steady_clock::now();
        unsigned threads = 0;
        if (const char* env = std::getenv("HFB200_IR_JIT_THREADS")) { const int v = std::atoi(env); if (v >= 1) threads = (unsigned)v; }
        const JitSpec s = jit_spec(*g, po2, threads);
        const std::vector<JitCubin> bins = JitCache::get().fetch(s, threads);
        for (const JitCubin& b : bins) if (!b) { interp_po2.insert(po2); return false; }
        Compiled c;
        try {
            for (size_t k = 0; k < bins.size(); k++) {
                cudaLibrary_t lib = nullptr;
                CUDA_CHECK(cudaLibraryLoadData(&lib, bins[k]->data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
                c.libs.push_back(lib);
                cudaKernel_t kern = nullptr;
                const std::string name = "hfb200_eval_check_jit_" + std::to_string(k);
                CUDA_CHECK(cudaLibraryGetKernel(&kern, lib, name.c_str()));
                c.kernels.push_back(kern);
            }
        } catch (...) {
            for (cudaLibrary_t l : c.libs) cudaLibraryUnload(l);  // the libraries loaded before the failure
            throw;
        }
        by_po2[po2] = std::move(c);
        compile_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        return true;
    }
    void destroy() { for (auto& kv : by_po2) for (auto& l : kv.second.libs) if (l) cudaLibraryUnload(l); by_po2.clear(); interp_po2.clear(); ready = enabled = false; }
    // after ensure(a.po2) returned true
    void launch(Dev& dev, const JitEvalArgs& a, uint64_t domain) {
        JitEvalArgs args = a;
        void* params[] = {&args};
        static const unsigned per_sm = [] { const char* e = std::getenv("HFB200_IR_JIT_BLOCKS_PER_SM"); const int v = e ? std::atoi(e) : 8; return (unsigned)(v >= 1 ? v : 8); }();
        const unsigned block = 128;
        const unsigned grid = (unsigned)std::min<uint64_t>((domain + block - 1) / block, (uint64_t)dev.sm_count * per_sm);
        for (cudaKernel_t k : by_po2.at(a.po2).kernels) {
            CUDA_CHECK(cudaLaunchKernel((const void*)k, dim3(grid), dim3(block), params, 0, dev.stream));
            dev.launches++;
        }
    }
};
#else
struct JitEvalCheck {
    bool ready = false;
    std::string note = "host emulator build";
    float compile_ms = 0;
    void init(const GenericCircuitHost&, uint32_t) {}
    bool ensure(uint32_t) { return false; }
    void destroy() {}
    void launch(Dev&, const JitEvalArgs&, uint64_t) {}
};
#endif

}  // namespace hf
