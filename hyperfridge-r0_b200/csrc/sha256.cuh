// SHA-256 hash suite: the FIPS 180-4 compression, the Merkle leaf / fold kernels over it and the host pieces of the transcript.
// Replaces risc0-zkp 3.0.4 `core::hash::sha::{cpu, rng}` (`Sha256HashSuite`) + `Hal::hash_rows` / `Hal::hash_fold` with that
// suite (upstream GPU: risc0-sys `sha_rows` / `sha_fold`).  Pure 32-bit ALU work: one thread owns one 8-word state and a
// 16-word message window in registers; rotates are funnel shifts, byte swaps are PRMT, Ch / Maj fold into LOP3.
//
// Convention (recalled from risc0-zkp 3.0.4 `core/hash/sha/{mod,cpu,rng}.rs` and risc0-sys `sha_rows` / `sha_fold`; only the
// compression function itself is fixed by FIPS 180-4):
//   * digest: 8 u32 words whose little-endian bytes are the standard SHA-256 output bytes, i.e. each word is the byte-swapped
//     state word;
//   * hash of n field elements (`hash_raw_data_slice`): the elements' raw Montgomery words as little-endian bytes, 16 words per
//     compression from the standard IV, the last block zero-filled, no length block (n = 0: the IV itself).  Merkle leaves,
//     H(PROOF_SYSTEM_INFO), H(CIRCUIT_INFO), H(globals ++ po2), the FRI final coefficients and hash_u;
//   * hash_pair(a, b): one compression of the 64-byte block a.bytes || b.bytes from the IV, no padding;
//   * ShaRng: pool0 = sha256("Hello"), pool1 = sha256("World") (standard, padded); step: pool0 = hash_pair(pool0, pool1), then
//     pool1 = hash_pair(pool0, pool1); mix(d): pool0 ^= d, step; next_u32: step when all 8 words are used, then the next word
//     of pool0; random_elem: six times v = (v << 32 + next_u32) mod p, in Montgomery form; random_bits(b): next_u32 & (2^b - 1).
#pragma once
#include "dev.cuh"

namespace hf {

enum : int { HASH_POSEIDON2 = 0, HASH_SHA256 = 1 };  // include/hfb200.h HFB200_HASH_*
static inline bool hash_suite_valid(int s) { return s == HASH_POSEIDON2 || s == HASH_SHA256; }

HD uint32_t sha_rotr(uint32_t x, int n) {
#ifdef __CUDA_ARCH__
    return __funnelshift_r(x, x, n);
#else
    return (x >> n) | (x << (32 - n));
#endif
}
HD uint32_t sha_bswap(uint32_t x) {
#ifdef __CUDA_ARCH__
    return __byte_perm(x, 0, 0x0123);
#else
    return __builtin_bswap32(x);
#endif
}

HD void sha256_iv(uint32_t st[8]) {
    st[0] = 0x6a09e667u; st[1] = 0xbb67ae85u; st[2] = 0x3c6ef372u; st[3] = 0xa54ff53au;
    st[4] = 0x510e527fu; st[5] = 0x9b05688cu; st[6] = 0x1f83d9abu; st[7] = 0x5be0cd19u;
}

// One compression of the 16 big-endian message words w (clobbered: it is the schedule window) into st.
HD void sha256_compress(uint32_t st[8], uint32_t w[16]) {
    const uint32_t K[64] = {
        0x428a2f98u, 0x71374491u, 0xb5c0fbcfu, 0xe9b5dba5u, 0x3956c25bu, 0x59f111f1u, 0x923f82a4u, 0xab1c5ed5u,
        0xd807aa98u, 0x12835b01u, 0x243185beu, 0x550c7dc3u, 0x72be5d74u, 0x80deb1feu, 0x9bdc06a7u, 0xc19bf174u,
        0xe49b69c1u, 0xefbe4786u, 0x0fc19dc6u, 0x240ca1ccu, 0x2de92c6fu, 0x4a7484aau, 0x5cb0a9dcu, 0x76f988dau,
        0x983e5152u, 0xa831c66du, 0xb00327c8u, 0xbf597fc7u, 0xc6e00bf3u, 0xd5a79147u, 0x06ca6351u, 0x14292967u,
        0x27b70a85u, 0x2e1b2138u, 0x4d2c6dfcu, 0x53380d13u, 0x650a7354u, 0x766a0abbu, 0x81c2c92eu, 0x92722c85u,
        0xa2bfe8a1u, 0xa81a664bu, 0xc24b8b70u, 0xc76c51a3u, 0xd192e819u, 0xd6990624u, 0xf40e3585u, 0x106aa070u,
        0x19a4c116u, 0x1e376c08u, 0x2748774cu, 0x34b0bcb5u, 0x391c0cb3u, 0x4ed8aa4au, 0x5b9cca4fu, 0x682e6ff3u,
        0x748f82eeu, 0x78a5636fu, 0x84c87814u, 0x8cc70208u, 0x90befffau, 0xa4506cebu, 0xbef9a3f7u, 0xc67178f2u};
    uint32_t a = st[0], b = st[1], c = st[2], d = st[3], e = st[4], f = st[5], g = st[6], h = st[7];
#pragma unroll
    for (int i = 0; i < 64; i++) {
        if (i >= 16) {
            const uint32_t x = w[(i - 15) & 15], y = w[(i - 2) & 15];
            const uint32_t s0 = sha_rotr(x, 7) ^ sha_rotr(x, 18) ^ (x >> 3);
            const uint32_t s1 = sha_rotr(y, 17) ^ sha_rotr(y, 19) ^ (y >> 10);
            w[i & 15] += s0 + w[(i - 7) & 15] + s1;
        }
        const uint32_t t1 = h + (sha_rotr(e, 6) ^ sha_rotr(e, 11) ^ sha_rotr(e, 25)) + ((e & f) ^ (~e & g)) + K[i] + w[i & 15];
        const uint32_t t2 = (sha_rotr(a, 2) ^ sha_rotr(a, 13) ^ sha_rotr(a, 22)) + ((a & b) | (c & (a | b)));
        h = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
    }
    st[0] += a; st[1] += b; st[2] += c; st[3] += d; st[4] += e; st[5] += f; st[6] += g; st[7] += h;
}

// hash_pair: digests a, b (8 words each, suite byte order) -> out
HD void sha_hash_pair(const uint32_t* a, const uint32_t* b, uint32_t* out) {
    uint32_t w[16], st[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { w[i] = sha_bswap(a[i]); w[8 + i] = sha_bswap(b[i]); }
    sha256_iv(st);
    sha256_compress(st, w);
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = sha_bswap(st[i]);
}

// ---- kernels ------------------------------------------------------------------------------------
// Hal::hash_rows: leaf r = raw hash of row r, matrix element (r, c) at matrix[c * col_stride + r]; one thread per row, so a
// warp reads 32 consecutive words of a column (one 128-byte line) per load.  Digest -> leaves[8 r ..].
struct ShaRowsKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, const uint32_t* matrix, uint64_t col_stride, uint32_t rows, uint32_t cols, uint32_t* leaves) {
        const uint64_t r = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (r >= rows) return;
        const uint32_t* src = matrix + r;
        uint32_t st[8], w[16];
        sha256_iv(st);
        uint32_t c = 0;
        for (; c + 16 <= cols; c += 16) {
#pragma unroll
            for (int i = 0; i < 16; i++) w[i] = sha_bswap(src[(uint64_t)(c + i) * col_stride]);
            sha256_compress(st, w);
        }
        if (c < cols) {
#pragma unroll
            for (int i = 0; i < 16; i++) w[i] = c + i < cols ? sha_bswap(src[(uint64_t)(c + i) * col_stride]) : 0u;
            sha256_compress(st, w);
        }
#ifdef __CUDA_ARCH__
        uint4* dst = reinterpret_cast<uint4*>(leaves + r * 8);
        dst[0] = make_uint4(sha_bswap(st[0]), sha_bswap(st[1]), sha_bswap(st[2]), sha_bswap(st[3]));
        dst[1] = make_uint4(sha_bswap(st[4]), sha_bswap(st[5]), sha_bswap(st[6]), sha_bswap(st[7]));
#else
        for (int i = 0; i < 8; i++) leaves[r * 8 + i] = sha_bswap(st[i]);
#endif
    }
};

// Hal::hash_fold for one level: nodes[i] = hash_pair(nodes[2i], nodes[2i+1]) for i in [level_size, 2 level_size); one thread per node.
struct ShaFoldKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* nodes, uint32_t level_size) {
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (t >= level_size) return;
        const uint64_t i = level_size + t;
        uint32_t w[16], st[8];
#ifdef __CUDA_ARCH__
        const uint4* in = reinterpret_cast<const uint4*>(nodes + 2 * i * 8);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint4 v = in[k];
            w[4 * k] = sha_bswap(v.x); w[4 * k + 1] = sha_bswap(v.y); w[4 * k + 2] = sha_bswap(v.z); w[4 * k + 3] = sha_bswap(v.w);
        }
#else
        for (int k = 0; k < 16; k++) w[k] = sha_bswap(nodes[2 * i * 8 + k]);
#endif
        sha256_iv(st);
        sha256_compress(st, w);
#ifdef __CUDA_ARCH__
        uint4* dst = reinterpret_cast<uint4*>(nodes + i * 8);
        dst[0] = make_uint4(sha_bswap(st[0]), sha_bswap(st[1]), sha_bswap(st[2]), sha_bswap(st[3]));
        dst[1] = make_uint4(sha_bswap(st[4]), sha_bswap(st[5]), sha_bswap(st[6]), sha_bswap(st[7]));
#else
        for (int k = 0; k < 8; k++) nodes[i * 8 + k] = sha_bswap(st[k]);
#endif
    }
};

// The last levels of the tree in one block: levels of size top, top/2, ..., 1 (top <= block threads).
struct ShaFoldTailKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* nodes, uint32_t top) {
        for (uint32_t level = top; level >= 1; level >>= 1) {
            for (uint32_t t = cx.tid; t < level; t += cx.nt) {
                const uint64_t i = level + t;
                sha_hash_pair(nodes + 2 * i * 8, nodes + (2 * i + 1) * 8, nodes + i * 8);
            }
#ifdef __CUDA_ARCH__
            __threadfence_block();
#endif
            cx.sync();
        }
    }
};

// ---- host side -----------------------------------------------------------------------------------
// hash_raw_data_slice over n words (field elements in Montgomery form, or raw words such as the po2 of the header)
static inline void sha_hash_words(const uint32_t* in, size_t n, uint32_t* out8) {
    uint32_t st[8], w[16];
    sha256_iv(st);
    size_t used = 0;
    for (size_t i = 0; i < n; i++) {
        w[used++] = sha_bswap(in[i]);
        if (used == 16) { sha256_compress(st, w); used = 0; }
    }
    if (used != 0) { for (size_t k = used; k < 16; k++) w[k] = 0; sha256_compress(st, w); }
    for (int i = 0; i < 8; i++) out8[i] = sha_bswap(st[i]);
}
// standard SHA-256 of a byte string (FIPS 180-4 padding), as digest words
static inline void sha256_bytes(const uint8_t* bytes, size_t n, uint32_t* out8) {
    std::vector<uint8_t> m(bytes, bytes + n);
    m.push_back(0x80);
    while (m.size() % 64 != 56) m.push_back(0);
    const uint64_t bits = (uint64_t)n * 8;
    for (int b = 0; b < 8; b++) m.push_back((uint8_t)(bits >> (56 - 8 * b)));
    uint32_t st[8], w[16];
    sha256_iv(st);
    for (size_t off = 0; off < m.size(); off += 64) {
        for (int i = 0; i < 16; i++) {
            const uint8_t* q = &m[off + 4 * i];
            w[i] = (uint32_t)q[0] << 24 | (uint32_t)q[1] << 16 | (uint32_t)q[2] << 8 | q[3];
        }
        sha256_compress(st, w);
    }
    for (int i = 0; i < 8; i++) out8[i] = sha_bswap(st[i]);
}

// risc0-zkp `ShaRng` (the Fiat-Shamir RNG of the SHA-256 suite)
struct ShaRng {
    uint32_t pool0[8], pool1[8];
    int pool_used = 0;
    ShaRng() {
        // the initial pools are constants: hashed once per process (every transcript and verifier starts from them)
        static const struct Init {
            uint32_t p0[8], p1[8];
            Init() {
                sha256_bytes(reinterpret_cast<const uint8_t*>("Hello"), 5, p0);
                sha256_bytes(reinterpret_cast<const uint8_t*>("World"), 5, p1);
            }
        } init;
        std::memcpy(pool0, init.p0, sizeof pool0);
        std::memcpy(pool1, init.p1, sizeof pool1);
    }
    void step() {
        sha_hash_pair(pool0, pool1, pool0);
        sha_hash_pair(pool0, pool1, pool1);
        pool_used = 0;
    }
    void mix(const uint32_t* d8) {
        for (int i = 0; i < 8; i++) pool0[i] ^= d8[i];
        step();
    }
    uint32_t next_u32() {
        if (pool_used == 8) step();
        return pool0[pool_used++];
    }
    uint32_t random_elem() {
        uint64_t v = 0;
        for (int i = 0; i < 6; i++) v = ((v << 32) + next_u32()) % P;
        return to_mont((uint32_t)v);
    }
    uint32_t random_bits(unsigned bits) { return next_u32() & (uint32_t)((1ull << bits) - 1); }
};

}  // namespace hf
