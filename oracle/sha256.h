// ORACLE (test infrastructure only).  SHA-256 hash suite, written from FIPS 180-4 over BYTE strings (a different shape from
// the product's word-window kernels in hyperfridge-r0_b200/csrc/sha256.cuh, so agreement is a cross-check).
// Suite convention recalled from risc0-zkp 3.0.4 `core/hash/sha/{mod,cpu,rng}.rs` (not vendored): a digest is the 32 output
// bytes read as 8 little-endian u32 words; elements hash as their raw Montgomery words' little-endian bytes, 64 bytes per
// compression from the IV, the last block zero-filled, no length block; hash_pair is one compression of a || b; ShaRng below.
#pragma once
#include <cstring>
#include <vector>
#include "fp.h"
#include "poseidon2.h"

namespace orc {

struct Sha256 {
    uint32_t h[8];
    Sha256() { reset(); }
    void reset() {
        static const uint32_t iv[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
        std::memcpy(h, iv, sizeof h);
    }
    static uint32_t rotr(uint32_t x, unsigned n) { return (x >> n) | (x << (32 - n)); }
    // FIPS 180-4 section 6.2.2 on one 64-byte block
    void compress(const uint8_t* block) {
        static const uint32_t k[64] = {
            0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98, 0x12835b01, 0x243185be,
            0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc, 0x2de92c6f, 0x4a7484aa,
            0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967, 0x27b70a85,
            0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85, 0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3,
            0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f,
            0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};
        uint32_t w[64];
        for (int t = 0; t < 16; t++)
            w[t] = (uint32_t)block[4 * t] << 24 | (uint32_t)block[4 * t + 1] << 16 | (uint32_t)block[4 * t + 2] << 8 | (uint32_t)block[4 * t + 3];
        for (int t = 16; t < 64; t++) {
            const uint32_t s0 = rotr(w[t - 15], 7) ^ rotr(w[t - 15], 18) ^ (w[t - 15] >> 3);
            const uint32_t s1 = rotr(w[t - 2], 17) ^ rotr(w[t - 2], 19) ^ (w[t - 2] >> 10);
            w[t] = w[t - 16] + s0 + w[t - 7] + s1;
        }
        uint32_t v[8];
        std::memcpy(v, h, sizeof v);
        for (int t = 0; t < 64; t++) {
            const uint32_t S1 = rotr(v[4], 6) ^ rotr(v[4], 11) ^ rotr(v[4], 25);
            const uint32_t ch = (v[4] & v[5]) ^ (~v[4] & v[6]);
            const uint32_t T1 = v[7] + S1 + ch + k[t] + w[t];
            const uint32_t S0 = rotr(v[0], 2) ^ rotr(v[0], 13) ^ rotr(v[0], 22);
            const uint32_t maj = (v[0] & v[1]) ^ (v[0] & v[2]) ^ (v[1] & v[2]);
            const uint32_t T2 = S0 + maj;
            for (int i = 7; i > 0; i--) v[i] = v[i - 1];
            v[4] += T1;
            v[0] = T1 + T2;
        }
        for (int i = 0; i < 8; i++) h[i] += v[i];
    }
    // the 32 output bytes (big-endian state words) as 8 little-endian digest words
    Digest digest() const {
        uint8_t out[32];
        for (int i = 0; i < 8; i++) { out[4 * i] = (uint8_t)(h[i] >> 24); out[4 * i + 1] = (uint8_t)(h[i] >> 16); out[4 * i + 2] = (uint8_t)(h[i] >> 8); out[4 * i + 3] = (uint8_t)h[i]; }
        Digest d;
        for (int i = 0; i < 8; i++) d.w[i] = (uint32_t)out[4 * i] | (uint32_t)out[4 * i + 1] << 8 | (uint32_t)out[4 * i + 2] << 16 | (uint32_t)out[4 * i + 3] << 24;
        return d;
    }
};

// standard SHA-256 (FIPS 180-4 padding) of a byte string
static inline Digest sha256_padded(const uint8_t* msg, size_t n) {
    std::vector<uint8_t> m(msg, msg + n);
    m.push_back(0x80);
    while (m.size() % 64 != 56) m.push_back(0);
    for (int i = 7; i >= 0; i--) m.push_back((uint8_t)(((uint64_t)n * 8) >> (8 * i)));
    Sha256 s;
    for (size_t off = 0; off < m.size(); off += 64) s.compress(&m[off]);
    return s.digest();
}
// The suite's hashes over field elements (hash_raw_data_slice: the raw Montgomery words as little-endian bytes, 64 bytes per
// compression from the IV, the last block zero-filled, no length block) and of two digests (one compression of a || b).
static inline Digest sha_hash_stride(const Fp* in, size_t count, size_t stride) {
    Sha256 s;
    uint8_t block[64];
    size_t used = 0;
    for (size_t i = 0; i < count; i++) {
        const uint32_t v = in[i * stride].v;
        for (int b = 0; b < 4; b++) block[used++] = (uint8_t)(v >> (8 * b));
        if (used == 64) { s.compress(block); used = 0; }
    }
    if (used) { std::memset(block + used, 0, 64 - used); s.compress(block); }
    return s.digest();
}
static inline Digest sha_hash_elems(const Fp* in, size_t count) { return sha_hash_stride(in, count, 1); }
static inline Digest sha_hash_ext_elems(const Fp4* in, size_t count) { return sha_hash_elems(reinterpret_cast<const Fp*>(in), count * 4); }
static inline Digest sha_hash_pair(const Digest& a, const Digest& b) {
    uint8_t block[64];
    for (int i = 0; i < 8; i++)
        for (int k = 0; k < 4; k++) { block[4 * i + k] = (uint8_t)(a.w[i] >> (8 * k)); block[32 + 4 * i + k] = (uint8_t)(b.w[i] >> (8 * k)); }
    Sha256 s;
    s.compress(block);
    return s.digest();
}

// risc0-zkp `ShaRng`: the transcript RNG of the suite (the interface of Poseidon2Rng)
struct ShaRng {
    Digest pool0, pool1;
    size_t pool_used = 0;
    ShaRng() {
        pool0 = sha256_padded(reinterpret_cast<const uint8_t*>("Hello"), 5);
        pool1 = sha256_padded(reinterpret_cast<const uint8_t*>("World"), 5);
    }
    void step() {
        pool0 = sha_hash_pair(pool0, pool1);
        pool1 = sha_hash_pair(pool0, pool1);
        pool_used = 0;
    }
    void mix(const Digest& d) {
        for (int i = 0; i < 8; i++) pool0.w[i] ^= d.w[i];
        step();
    }
    uint32_t next_u32() {
        if (pool_used == 8) step();
        return pool0.w[pool_used++];
    }
    Fp random_elem() {
        uint64_t v = 0;
        for (int i = 0; i < 6; i++) v = ((v << 32) + next_u32()) % P;
        return Fp::from_u32((uint32_t)v);
    }
    Fp4 random_ext_elem() { Fp a = random_elem(), b = random_elem(), c = random_elem(), d = random_elem(); return Fp4(a, b, c, d); }
    uint32_t random_bits(unsigned bits) { return next_u32() & (uint32_t)(((uint64_t)1 << bits) - 1); }
};

}  // namespace orc
