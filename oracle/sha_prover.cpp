// ORACLE (test infrastructure only).  The oracle's prover, verifier and control ids with upstream's SHA-256 hash suite
// (`segment_prover("sha-256")`), built into its own library (oracle/_build/liboracle_sha.so, oracle/sha_suite.py).
//
// The suite decides the Merkle hash and the transcript RNG, nothing else of the protocol.  So this file does not restate the
// protocol a second time: it compiles the oracle's own prover.cpp (and the headers it includes) again, in namespace orc_sha, with
// the Poseidon2 names of poseidon2.h -- the leaf / element hash, hash_pair and Poseidon2Rng -- bound to the SHA-256 ones of
// sha256.h.  poseidon2.h itself is read first, with its names intact, so only the code that USES those names (merkle_iop.h,
// prover.cpp) switches suite.  The claim digests are not part of this code.
#define orc orc_sha
#include "poseidon2.h"
#include "sha256.h"
#define unpadded_hash_stride sha_hash_stride
#define hash_elems sha_hash_elems
#define hash_ext_elems sha_hash_ext_elems
#define hash_pair sha_hash_pair
#define Poseidon2Rng ShaRng
#include "prover.cpp"
#undef unpadded_hash_stride
#undef hash_elems
#undef hash_ext_elems
#undef hash_pair
#undef Poseidon2Rng
#include <cstring>

using namespace orc_sha;

static thread_local std::string g_err;
#define ORC_TRY try {
#define ORC_CATCH } catch (const std::exception& e) { g_err = e.what(); return -1; } return 0;

struct ShaProofHandle { SegmentProof proof; OracleTimes times; };

extern "C" {

const char* orc_sha_last_error() { return g_err.c_str(); }

// ---- primitives ----
void orc_sha_sha256(const uint8_t* msg, size_t n, uint32_t* out8) { Digest d = sha256_padded(msg, n); std::memcpy(out8, d.w, 32); }
void orc_sha_hash_elems(const uint32_t* in, size_t n, uint32_t* out8) {
    Digest d = sha_hash_elems(reinterpret_cast<const Fp*>(in), n);
    std::memcpy(out8, d.w, 32);
}
void orc_sha_hash_pair(const uint32_t* a, const uint32_t* b, uint32_t* out8) {
    Digest d = sha_hash_pair(*reinterpret_cast<const Digest*>(a), *reinterpret_cast<const Digest*>(b));
    std::memcpy(out8, d.w, 32);
}
// A script over one ShaRng: ops[2i] = 0 mix(the next digest of `digests`), 1 random_elem (raw Montgomery word to out),
// 2 random_bits(ops[2i + 1]) to out.  Returns the number of words written.
size_t orc_sha_rng_script(const uint32_t* ops, size_t n_ops, const uint32_t* digests, uint32_t* out) {
    ShaRng r;
    size_t d = 0, o = 0;
    for (size_t i = 0; i < n_ops; i++) {
        const uint32_t op = ops[2 * i], arg = ops[2 * i + 1];
        if (op == 0) r.mix(*reinterpret_cast<const Digest*>(digests + 8 * d++));
        else if (op == 1) out[o++] = r.random_elem().v;
        else out[o++] = r.random_bits(arg);
    }
    return o;
}
// nodes_out (optional): 2*rows digests in heap layout.
int orc_sha_merkle(const uint32_t* matrix, size_t rows, size_t cols, uint32_t* root_out, uint32_t* nodes_out) {
    ORC_TRY
    MerkleTreeProver t(reinterpret_cast<const Fp*>(matrix), rows, cols);
    std::memcpy(root_out, t.root().w, 32);
    if (nodes_out) std::memcpy(nodes_out, t.nodes.data(), 2 * rows * 32);
    ORC_CATCH
}

// ---- circuits (the handle API of capi.cpp) ----
void* orc_sha_circuit_new(uint32_t wc, uint32_t wd, uint32_t wa, uint32_t variant) {
    try { return new Circuit(wc, wd, wa, variant); } catch (const std::exception& e) { g_err = e.what(); return nullptr; }
}
void orc_sha_circuit_free(void* h) { delete static_cast<Circuit*>(h); }
int orc_sha_circuit_set_ir(void* h, const uint32_t* taps, size_t n_taps, const uint32_t* steps, size_t n_steps, uint32_t ret, const uint8_t* info16) {
    ORC_TRY
    Circuit* c = static_cast<Circuit*>(h);
    if (taps) {
        std::vector<Tap> t(n_taps);
        for (size_t i = 0; i < n_taps; i++) t[i] = Tap{taps[3 * i], taps[3 * i + 1], taps[3 * i + 2], 0};
        c->set_taps(t);
    }
    std::vector<PolyStep> st(n_steps);
    for (size_t i = 0; i < n_steps; i++) st[i] = PolyStep{steps[4 * i], steps[4 * i + 1], steps[4 * i + 2], steps[4 * i + 3]};
    c->set_ir(st, ret, info16);
    ORC_CATCH
}
int orc_sha_control_id(void* h, unsigned po2, uint32_t* root_out) {
    ORC_TRY Digest d = control_id(*static_cast<Circuit*>(h), po2); std::memcpy(root_out, d.w, 32); ORC_CATCH
}
int orc_sha_prove_segment(void* h, unsigned po2, const uint32_t* globals, const uint32_t* code, const uint32_t* data, uint64_t blind_seed, void** handle_out) {
    ORC_TRY
    ShaProofHandle* ph = new ShaProofHandle();
    try {
        ph->proof = prove_segment(*static_cast<Circuit*>(h), po2, reinterpret_cast<const Fp*>(globals), reinterpret_cast<const Fp*>(code),
                                  reinterpret_cast<const Fp*>(data), blind_seed, &ph->times);
    } catch (...) { delete ph; throw; }
    *handle_out = ph;
    ORC_CATCH
}
int orc_sha_verify_segment(void* h, const uint32_t* seal, size_t seal_words, const uint32_t* code_root, unsigned* po2_out) {
    ORC_TRY
    verify_segment(*static_cast<Circuit*>(h), seal, seal_words, *reinterpret_cast<const Digest*>(code_root), po2_out);
    ORC_CATCH
}
size_t orc_sha_proof_seal_words(void* h) { return static_cast<ShaProofHandle*>(h)->proof.seal.size(); }
void orc_sha_proof_seal(void* h, uint32_t* out) { auto& s = static_cast<ShaProofHandle*>(h)->proof.seal; std::memcpy(out, s.data(), s.size() * 4); }
size_t orc_sha_proof_n_checkpoints(void* h) { return static_cast<ShaProofHandle*>(h)->proof.cp.items.size(); }
size_t orc_sha_proof_checkpoint(void* h, size_t i, char* name, size_t name_cap, uint32_t* words, size_t cap) {
    auto& it = static_cast<ShaProofHandle*>(h)->proof.cp.items[i];
    std::snprintf(name, name_cap, "%s", it.first.c_str());
    size_t n = it.second.size() < cap ? it.second.size() : cap;
    std::memcpy(words, it.second.data(), n * 4);
    return it.second.size();
}
void orc_sha_proof_free(void* h) { delete static_cast<ShaProofHandle*>(h); }

}  // extern "C"
