// Poseidon2 (BabyBear, t = 24, x^7, 4+21+4 rounds) permutation, sponge and Merkle kernels.
// Replaces risc0-zkp 3.0.4 `core::hash::poseidon2` + `Hal::hash_rows` / `Hal::hash_fold` (upstream GPU:
// sppark poseidon2_rows/fold in risc0-sys 1.5.0; /root/reference/Cargo.lock:3174-3223, not vendored;
// SURVEY.md Appendix A.3/A.4).  Integer-pipe bound: one thread owns one 24-word sponge state in
// registers; a warp owns 32 consecutive rows so every column read is one coalesced 128-byte line.
#pragma once
#include "dev.cuh"

namespace hf {

#include "poseidon2_consts.inc"

struct P2Consts {
    uint32_t rc_first[96], rc_partial[21], rc_last[96], diag[24];  // Montgomery form
    uint32_t diag_std[24], diag_shoup[24];  // canonical d_i and floor(d_i * 2^32 / p): constant multiplier in Shoup form
    int32_t tri_c[21];  // partial rounds in tensor form: c_k = (M_I^k)[0][0] * 2^32 mod p, balanced in (-p/2, p/2], k = 1..20 (only k < P2TC_BS are read)
};

// ---- the 21 partial rounds as two linear maps ----------------------------------------------------------------------------
// Partial round r (r = 0..20) on state v_r: cell 0 becomes sbox(v_r[0] + rc_r), then v_{r+1} = M_I (v_r + delta_r e0) with
// M_I = 1 1^T + diag(d) and delta_r = sbox(v_r[0] + rc_r) - v_r[0].  Unrolled from the state v = v_0 entering the section:
//   v_r[0] = a_r . v + sum_{j<r} c_{r-j} delta_j         a_r = e0^T M_I^r,  c_k = (M_I^k)[0][0]
//   v_21   = M_I^21 v + sum_j delta_j M_I^(21-j) e0      (one 24 x 45 map of [v | delta])
// so everything but the S-boxes and the 210-term triangular sum is two dense maps over the states of a CTA: GEMM 1 yields
// a_1..a_20 . v (20 outputs), GEMM 2 yields v_21 (24 outputs).  Both run exactly on the int8 tensor cores: the 32-bit input
// words are split into their 4 bytes (K = 4 per input), the byte weight 2^(8b) and the Montgomery factor 2^32 are folded
// into the constant, C'_((i,b),o) = 2^(8b) * m_oi * 2^32 mod p, whose 4 bytes j form 4 output planes (N = 4 per output).
// Plane j accumulates Q_j = sum bytes * bytes <= 180 * 255^2 < 2^24 in int32; V = sum_j 2^(8j) Q_j < 2^49 < p 2^32, so one
// Montgomery REDC of V is the Montgomery residue of the output.  The state words need no conversion: a little-endian u32 is
// already its 4 byte inputs.
//
// Blocked chain: the 21 rounds are cut into P2TC_BLOCKS blocks of P2TC_BS rounds.  Once the deltas of block b - 1 are known,
// one small GEMM (K = the bytes of that block's deltas) adds sum_{j in block b-1} c_{r-j} delta_j to the planes of every
// later round r, accumulating into the TMEM columns where GEMM 1 left a_r . v.  SIMT then sums only the terms inside a block
// (3 x 21 = 63 instead of 210 for 3 blocks of 7).  A plane accumulates at most 96 + 4 * 21 bytes * bytes, so Q_j < 2^24 holds.
// 1 block is the plain two-GEMM form (-DP2TC_BLOCKS=1 through tools/build_variant.sh, for A/B).
#ifndef P2TC_BLOCKS
#define P2TC_BLOCKS 3
#endif
static_assert(P2TC_BLOCKS >= 1 && P2TC_BLOCKS <= 4, "P2TC_BLOCKS: 1..4");
static constexpr uint32_t P2TC_NB = P2TC_BLOCKS;
static constexpr uint32_t P2TC_BS = (21 + P2TC_NB - 1) / P2TC_NB;  // rounds per block (the last may be shorter)
static constexpr uint32_t P2TC_BW = (P2TC_BS + 7) / 8 * 8;          // A words per block: each block starts on a 32-byte K step
static constexpr uint32_t P2TC_AW = 24 + P2TC_NB * P2TC_BW;         // A row: [v | delta block 0 | ... | block NB-1], zero-padded
static constexpr uint32_t P2TC_K1 = 96, P2TC_N1 = 80;    // GEMM 1: bytes of v -> 4 planes of a_1..a_20 . v (round r: columns 4(r-1)..)
static constexpr uint32_t P2TC_K2 = 4 * P2TC_AW, P2TC_N2 = 96;  // GEMM 2: bytes of the whole A row -> 4 planes of v_21
static constexpr uint32_t P2TC_B1_BYTES = P2TC_K1 * P2TC_N1;
// block GEMM b = 1..NB-1 (A = delta block b-1, K = 4 BW) writes TMEM columns [c0, 80): c0 is the 16-aligned column at or below
// the first plane of round b BS, and the B rows in front of that plane are zero.
HD constexpr uint32_t p2tc_blk_c0(uint32_t b) { return (4 * (b * P2TC_BS - 1)) & ~15u; }
HD constexpr uint32_t p2tc_blk_n(uint32_t b) { return P2TC_N1 - p2tc_blk_c0(b); }
HD constexpr uint32_t p2tc_blk_boff(uint32_t b) { return b <= 1 ? P2TC_B1_BYTES : p2tc_blk_boff(b - 1) + 4 * P2TC_BW * p2tc_blk_n(b - 1); }
static constexpr uint32_t P2TC_B2_OFF = p2tc_blk_boff(P2TC_NB);  // GEMM 2's B rows follow the block GEMMs'
static constexpr uint32_t P2TC_B_BYTES = P2TC_B2_OFF + P2TC_K2 * P2TC_N2;
// Operand layout of all GEMMs (tcgen05 shared-memory descriptor, K-major, no swizzle): core matrices of 8 rows x 16 bytes,
// 128 contiguous bytes each; the next 16 bytes along K are 128 bytes further (LBO), the next 8 rows 8 K bytes further (SBO).
HD uint32_t p2tc_off(uint32_t row, uint32_t k, uint32_t K) { return (row >> 3) * (K * 8) + (k >> 4) * 128 + (row & 7) * 16 + (k & 15); }
struct P2TcTables {
    uint8_t b[P2TC_B_BYTES];  // B operands (rows = the N output planes) in the layout above: GEMM 1, the block GEMMs, GEMM 2
};

static inline uint32_t p2_mod_mul(uint32_t a, uint32_t b) { return (uint32_t)((uint64_t)a * b % P); }
// M_I^k for k = 0..21, canonical entries, exact
static inline std::vector<std::vector<uint32_t>> p2_m_int_powers() {
    std::vector<std::vector<uint32_t>> pw(22, std::vector<uint32_t>(24 * 24, 0));
    for (int i = 0; i < 24; i++) pw[0][i * 24 + i] = 1;
    for (int k = 1; k < 22; k++)
        for (int o = 0; o < 24; o++)
            for (int i = 0; i < 24; i++) {  // (M_I X)[o][i] = sum_l X[l][i] + d_o X[o][i]
                uint64_t acc = p2_mod_mul(P2_M_INT_DIAG[o], pw[k - 1][o * 24 + i]);
                for (int l = 0; l < 24; l++) acc += pw[k - 1][l * 24 + i];
                pw[k][o * 24 + i] = (uint32_t)(acc % P);
            }
    return pw;
}
// one linear output o = sum_i m_i x_i of a GEMM with K input bytes, written as byte planes n = 4 o + j
static inline void p2tc_put_output(uint8_t* b, uint32_t K, uint32_t o, const uint32_t* m, int n_in) {
    for (int i = 0; i < n_in; i++)
        for (uint32_t bb = 0; bb < 4; bb++) {
            const uint32_t c = to_mont(p2_mod_mul(m[i], 1u << (8 * bb)));  // 2^(8b) m_i 2^32 mod p
            for (uint32_t j = 0; j < 4; j++) b[p2tc_off(4 * o + j, 4 * i + bb, K)] = (uint8_t)(c >> (8 * j));
        }
}
static inline P2TcTables p2_make_tc_tables() {
    P2TcTables t;
    std::memset(t.b, 0, sizeof t.b);
    const auto pw = p2_m_int_powers();
    uint32_t m[P2TC_AW];
    for (uint32_t r = 1; r <= 20; r++) p2tc_put_output(t.b, P2TC_K1, r - 1, &pw[r][0], 24);  // row 0 of M_I^r
    for (uint32_t b = 1; b < P2TC_NB; b++)
        for (uint32_t r = b * P2TC_BS; r <= 20; r++) {  // c_{r-j} for the deltas j of block b-1
            for (uint32_t i = 0; i < P2TC_BS; i++) m[i] = pw[r - ((b - 1) * P2TC_BS + i)][0];
            p2tc_put_output(t.b + p2tc_blk_boff(b), 4 * P2TC_BW, (4 * (r - 1) - p2tc_blk_c0(b)) / 4, m, P2TC_BS);
        }
    for (uint32_t o = 0; o < 24; o++) {
        std::memset(m, 0, sizeof m);
        for (int i = 0; i < 24; i++) m[i] = pw[21][o * 24 + i];
        for (uint32_t j = 0; j < 21; j++) m[24 + j / P2TC_BS * P2TC_BW + j % P2TC_BS] = pw[21 - j][o * 24];  // (M_I^(21-j) e0)[o]
        p2tc_put_output(t.b + P2TC_B2_OFF, P2TC_K2, o, m, P2TC_AW);
    }
    return t;
}

static inline P2Consts p2_make_consts() {
    P2Consts c;
    for (int i = 0; i < 96; i++) { c.rc_first[i] = to_mont(P2_RC_FULL_FIRST[i]); c.rc_last[i] = to_mont(P2_RC_FULL_LAST[i]); }
    for (int i = 0; i < 21; i++) c.rc_partial[i] = to_mont(P2_RC_PARTIAL[i]);
    for (int i = 0; i < 24; i++) {
        c.diag[i] = to_mont(P2_M_INT_DIAG[i]);
        c.diag_std[i] = P2_M_INT_DIAG[i];
        c.diag_shoup[i] = (uint32_t)(((uint64_t)P2_M_INT_DIAG[i] << 32) / P);
    }
    const auto pw = p2_m_int_powers();
    c.tri_c[0] = 0;
    for (int k = 1; k < 21; k++) {
        const uint32_t v = to_mont(pw[k][0]);
        c.tri_c[k] = v > (P - 1) / 2 ? (int32_t)v - (int32_t)P : (int32_t)v;
    }
    return c;
}

#if !defined(HFB200_EMU)
__constant__ P2Consts g_p2c;
#define P2C_DEV g_p2c
__device__ __align__(16) uint8_t g_p2tc_b[P2TC_B_BYTES];
#endif
static P2Consts g_p2c_host;
static P2TcTables g_p2tc_host;
static inline const P2Consts& p2_host_consts() {
    static const bool once = (g_p2c_host = p2_make_consts(), g_p2tc_host = p2_make_tc_tables(), true);  // thread-safe one-time initialisation
    (void)once;
    return g_p2c_host;
}

HD const P2Consts& p2c() {
#if defined(__CUDA_ARCH__)
    return P2C_DEV;
#else
    return g_p2c_host;
#endif
}

// Pipe steering experiment (B200): 32-bit integer multiplies run only on the heavy half of the FMA pipe, the binding
// unit of this kernel (ncu: sm__pipe_fmaheavy_cycles_active ~92 %).  ptxas splits plain adds between the ALU pipe
// (IADD3) and the FMA pipe (IMAD.IADD).  P2_FADD_ALU=1 pins them to the ALU pipe by writing the add as VIADDMNMX
// (min(a + b, UINT_MAX)); measured on B200 this is 3.7 % SLOWER (28.9 -> 30.0 ms for the 192-column tree), i.e. both
// pipes are already saturated together, so the default stays 0.
#ifndef P2_FADD_ALU
#define P2_FADD_ALU 0
#endif
HD uint32_t padd(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__) && P2_FADD_ALU
    const uint32_t x = __viaddmin_u32(a, b, 0xFFFFFFFFu);
    return __viaddmin_u32(x, 0u - P, x);
#else
    return fadd(a, b);
#endif
}
// Montgomery product left in (0, 2p): one IADD3 instead of subtract + conditional correction.  Valid as ONE operand of a
// following fmul/fmul_lazy whose other operand is canonical (2p * p < p * 2^32).
HD uint32_t fmul_lazy(uint32_t a, uint32_t b) {
    uint64_t o = (uint64_t)a * b;
    uint32_t m = (uint32_t)o * P_INV;
#ifdef __CUDA_ARCH__
    uint32_t mp = __umulhi(m, P);
#else
    uint32_t mp = (uint32_t)(((uint64_t)m * P) >> 32);
#endif
    return (uint32_t)(o >> 32) - mp + P;
}
// x^7 with 4 multiplies; x4 stays lazy (it only meets the canonical x3).
HD uint32_t sbox7(uint32_t x) { uint32_t x2 = fmul(x, x), x3 = fmul(x2, x), x4 = fmul_lazy(x2, x2); return fmul(x3, x4); }
// Signed Montgomery product: for |a * b| < 2^31 * p the value hi(a*b) - hi(m*p), m = lo(a*b) * p^-1 (all signed), is the
// exact quotient (a*b - m*p) / 2^32 and lies in (-p, p): no correction step at all.
HD int32_t smul(int32_t a, int32_t b) {
    const int64_t o = (int64_t)a * b;
    const int32_t m = (int32_t)((uint32_t)o * P_INV);
#ifdef __CUDA_ARCH__
    const int32_t mp = __mulhi(m, (int32_t)P);
#else
    const int32_t mp = (int32_t)(((int64_t)m * (int64_t)P) >> 32);
#endif
    return (int32_t)(o >> 32) - mp;
}
// (s + rc)^7 for canonical s, rc: the sum enters the chain as the signed representative s + rc - p in [-p, p) (one IADD3),
// the four products stay signed in (-p, p) and only the result is made canonical: 4 * 4 + 2 instructions instead of 21.
#ifndef P2_SIGNED_SBOX
#define P2_SIGNED_SBOX 1
#endif
HD uint32_t sbox7_rc(uint32_t s, uint32_t rc) {
#if P2_SIGNED_SBOX
    const int32_t x = (int32_t)(s + rc - P);
    const int32_t x2 = smul(x, x), x3 = smul(x2, x), x4 = smul(x2, x2);
    const uint32_t r = (uint32_t)smul(x3, x4);
    return umin32(r, r + P);
#else
    return sbox7(padd(s, rc));
#endif
}
// x * d mod p for a constant d given as (d, d' = floor(d 2^32 / p)) -- Shoup: no 64-bit product, result already in [0, 2p).
// x may be any residue representation (here Montgomery), d is the canonical constant.
HD uint32_t fmul_const(uint32_t x, uint32_t d, uint32_t dp) {
#ifdef __CUDA_ARCH__
    const uint32_t q = __umulhi(x, dp);
#else
    const uint32_t q = (uint32_t)(((uint64_t)x * dp) >> 32);
#endif
    const uint32_t r = x * d - q * P;
    return umin32(r, r - P);
}

#ifndef P2_DEFERRED_SUM
#define P2_DEFERRED_SUM 1  // 0: plain internal layer; 1: carried row sum, 23 S by a Shoup product; 2: 23 S by doublings
#endif
// External layer: M4 on each 4-chunk (Poseidon2 add/double chain) then add the cross-chunk column sums.
HD void p2_m_ext(uint32_t* s) {
#pragma unroll
    for (int c = 0; c < 24; c += 4) {
        uint32_t a = s[c], b = s[c + 1], cc = s[c + 2], d = s[c + 3];
        uint32_t t0 = padd(a, b), t1 = padd(cc, d);
        uint32_t t2 = padd(padd(b, b), t1), t3 = padd(padd(d, d), t0);
        uint32_t t4 = padd(t1, t1); t4 = padd(padd(t4, t4), t3);
        uint32_t t5 = padd(t0, t0); t5 = padd(padd(t5, t5), t2);
        s[c] = padd(t3, t5); s[c + 1] = t5; s[c + 2] = padd(t2, t4); s[c + 3] = t4;
    }
    uint32_t sum[4];
#pragma unroll
    for (int j = 0; j < 4; j++) sum[j] = padd(padd(padd(s[j], s[4 + j]), padd(s[8 + j], s[12 + j])), padd(s[16 + j], s[20 + j]));
#pragma unroll
    for (int i = 0; i < 24; i++) s[i] = padd(s[i], sum[i & 3]);
}

HD void p2_m_int(uint32_t* s, const P2Consts& k) {
    uint32_t sum = 0;
#pragma unroll
    for (int i = 0; i < 24; i++) sum = padd(sum, s[i]);
#pragma unroll
    for (int i = 0; i < 24; i++) s[i] = padd(sum, fmul_const(s[i], k.diag_std[i], k.diag_shoup[i]));
}

HD void p2_full_rounds(uint32_t* s, const uint32_t* rc) {
#pragma unroll 1
    for (int r = 0; r < 4; r++) {
#pragma unroll
        for (int i = 0; i < 24; i++) s[i] = sbox7_rc(s[i], rc[r * 24 + i]);
        p2_m_ext(s);
    }
}

HD void p2_mix(uint32_t* s) {
    const P2Consts& k = p2c();
    p2_m_ext(s);
    p2_full_rounds(s, k.rc_first);
#if P2_DEFERRED_SUM
    // Partial rounds with the row sum carried instead of recomputed.  The round maps y_i -> mu_i y_i + S with S = sum_i y_i
    // (after the S-box on y_0).  With U = sum_{i>=1} y_i kept canonical:  S = y_0 + U,  t_i = mu_i y_i (Shoup: accepts ANY
    // 32-bit y_i),  U' = sum_{i>=1} t_i + 23 S,  y_0' = t_0 + S (canonical: it meets the S-box),  y_i' = t_i + S left in
    // [0, 2p) for i >= 1 (one add, no range correction: its only reader is the next Shoup product).
    {
        uint32_t U = s[1];
#pragma unroll
        for (int i = 2; i < 24; i++) U = padd(U, s[i]);
#pragma unroll 1
        for (int r = 0; r < 21; r++) {
            s[0] = sbox7_rc(s[0], k.rc_partial[r]);
            const uint32_t S = padd(s[0], U);
            uint32_t t[24];
#pragma unroll
            for (int i = 0; i < 24; i++) t[i] = fmul_const(s[i], k.diag_std[i], k.diag_shoup[i]);
            uint32_t T = t[1];
#pragma unroll
            for (int i = 2; i < 24; i++) T = padd(T, t[i]);
#if P2_DEFERRED_SUM == 2
            uint32_t S2 = padd(S, S), S4 = padd(S2, S2), S8 = padd(S4, S4), S16 = padd(S8, S8);
            const uint32_t S23 = fsub(padd(S16, S8), S);
#else
            const uint32_t S23 = fmul_const(S, 23u, (uint32_t)((23ull << 32) / P));
#endif
            U = padd(T, S23);
            s[0] = padd(t[0], S);
#pragma unroll
            for (int i = 1; i < 24; i++) s[i] = fadd_lazy(t[i], S);
        }
#pragma unroll
        for (int i = 1; i < 24; i++) s[i] = umin32(s[i], s[i] - P);
    }
#else
#pragma unroll 1
    for (int r = 0; r < 21; r++) {
        s[0] = sbox7_rc(s[0], k.rc_partial[r]);
        p2_m_int(s, k);
    }
#endif
    p2_full_rounds(s, k.rc_last);
}

// ---- permutation with the partial rounds on the tensor cores (see "the 21 partial rounds as two linear maps") ---------------
// Device: one CTA of 128 threads = 128 states = the 128 TMEM lanes of a tcgen05.mma (M = 128, kind::i8, cta_group::1).
// Thread t writes its A row (the P2TC_AW words [v | delta blocks]) into shared memory, one thread issues the MMAs,
// tcgen05.commit arrives on an mbarrier, and thread t reads its own row of the int32 planes back with tcgen05.ld.  Every
// thread of the CTA takes part in every permutation (the barriers are CTA-wide), so kernels run idle states on zeros instead
// of returning.  Emulator (and the nvcc host pass): the same row, tables, recombination and REDC, with plain loops in place
// of the MMA accumulating into a per-state column array in place of TMEM.
#ifndef P2_TC
#define P2_TC 1
#endif
static constexpr uint32_t P2TC_A_BYTES = 128 * P2TC_K2;
static constexpr size_t P2TC_SMEM = P2TC_A_BYTES + P2TC_B_BYTES + 32;  // A tile, B operands, 2 mbarriers + the TMEM address
static constexpr uint32_t P2TC_TMEM_COLS = 128;                        // >= N1, N2; 4 CTAs fill an SM's 512 columns

// Phase probe (-DP2_PHASE_PROBE=1, device only): lane 0 of warp 1 of every CTA (a warp that does not issue the MMAs) adds the
// clock64 cycles of each phase of p2_mix_tc to g_p2_probe[phase]; g_p2_probe[P2_PROBE_N] counts the permutations.  Phases:
// 0 first full rounds; per block b: 1 + 3b A row stores + MMA round trip (barrier, issue, commit, mbarrier wait),
// 2 + 3b tcgen05.ld + recombination of the block's rounds, 3 + 3b the block's S-box chain; then 1 + 3 NB GEMM 2 round trip,
// 2 + 3 NB its loads + recombination, 3 + 3 NB last full rounds.  hfb200_p2_probe_read returns and clears the counters.
#ifndef P2_PHASE_PROBE
#define P2_PHASE_PROBE 0
#endif
static constexpr uint32_t P2_PROBE_N = 4 + 3 * P2TC_NB;
#if P2_PHASE_PROBE && !defined(HFB200_EMU)
__device__ unsigned long long g_p2_probe[P2_PROBE_N + 1];
#endif

struct P2Tc {
#ifdef __CUDA_ARCH__
    uint8_t* a;      // A tile, 128 rows x K2 bytes
    uint8_t* b;      // B operands (P2TcTables::b)
    uint64_t* bar;   // [0]: B operands loaded, [1]: MMA done
    uint32_t* tslot; // TMEM base address written by tcgen05.alloc
    uint32_t tmem, phase, row;
    bool b_wait;     // thread 0: B operands not yet waited for
#if P2_PHASE_PROBE
    long long t;     // clock64 at the last phase boundary
#endif
#else
    uint32_t w[P2TC_AW];             // this state's A row
    uint32_t acc[P2TC_TMEM_COLS];    // this state's TMEM lane
#endif
};
HD void p2tc_mark(P2Tc& tc, uint32_t ph) {
#if defined(__CUDA_ARCH__) && P2_PHASE_PROBE
    if (tc.row == 32) {
        const long long t = clock64();
        if (ph < P2_PROBE_N) atomicAdd(&g_p2_probe[ph], (unsigned long long)(t - tc.t));
        else atomicAdd(&g_p2_probe[P2_PROBE_N], 1ull);
        tc.t = t;
    }
#else
    (void)tc; (void)ph;
#endif
}

#ifdef __CUDA_ARCH__
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// K-major, no swizzle (layout of p2tc_off): LBO = 128 B, SBO = 8 K B, bits 46-48 = 0b001 (sm_100 descriptor version)
__device__ __forceinline__ uint64_t p2tc_desc(uint32_t saddr, uint32_t K) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(128u >> 4) << 16) | ((uint64_t)((8u * K) >> 4) << 32) | (1ull << 46);
}
#endif

// Per-CTA set-up: B operands into shared memory (one bulk copy), mbarriers, 128 TMEM columns.  All threads call it.
HD void p2tc_begin(P2Tc& tc, const KCtx& cx, uint32_t* smem) {
#ifdef __CUDA_ARCH__
    uint8_t* base = reinterpret_cast<uint8_t*>(smem);
    tc.a = base;
    tc.b = base + P2TC_A_BYTES;
    tc.bar = reinterpret_cast<uint64_t*>(base + P2TC_A_BYTES + P2TC_B_BYTES);
    tc.tslot = reinterpret_cast<uint32_t*>(tc.bar + 2);
    tc.phase = 0;
    tc.row = (uint32_t)cx.tid;
    tc.b_wait = cx.tid == 0;
    if (cx.tid == 0) {
        mbar_init(&tc.bar[0], 1);
        mbar_init(&tc.bar[1], 1);
        mbar_init_fence();
        mbar_expect_tx(&tc.bar[0], P2TC_B_BYTES);
        tma_bulk_g2s(tc.b, g_p2tc_b, P2TC_B_BYTES, &tc.bar[0]);
    }
    if (cx.tid < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tc.tslot)), "r"(P2TC_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    tc.tmem = *tc.tslot;
#else
    (void)tc; (void)cx; (void)smem;
#endif
}
HD void p2tc_end(P2Tc& tc, const KCtx& cx) {
#ifdef __CUDA_ARCH__
    tc_fence_before();
    __syncthreads();
    if (cx.tid < 32) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tc.tmem), "r"(P2TC_TMEM_COLS) : "memory");
    }
#else
    (void)tc; (void)cx;
#endif
}
// words [w0, w0 + 4 n) of this state's A row
HD void p2tc_put(P2Tc& tc, uint32_t w0, const uint32_t* v, uint32_t n) {
#ifdef __CUDA_ARCH__
#pragma unroll
    for (uint32_t c = 0; c < n; c++)
        *reinterpret_cast<uint4*>(tc.a + p2tc_off(tc.row, 4 * (w0 + 4 * c), P2TC_K2)) = make_uint4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
#else
    for (uint32_t i = 0; i < 4 * n; i++) tc.w[w0 + i] = v[i];
#endif
}
// D[:, c0 .. c0 + N) (+)= A[:, 4 aw0 .. 4 aw0 + K) x B^T over the rows of all threads of the CTA, B the K x N operand at byte
// boff of the tables; accumulate into the TMEM columns when acc.  aw0 is a multiple of 8 (a 32-byte K step), c0 of 16.
// first: the CTA's first GEMM of the permutation, the only one whose issue may still have to wait for the B operands.
HD void p2tc_mma(P2Tc& tc, uint32_t aw0, uint32_t K, uint32_t boff, uint32_t c0, uint32_t N, bool acc, bool first) {
#ifdef __CUDA_ARCH__
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy row stores -> visible to the MMA
    tc_fence_before();                                             // earlier tcgen05.ld of these columns are complete
    __syncthreads();
    if (tc.row == 0) {
        tc_fence_after();
        if (first && tc.b_wait) { mbar_wait(&tc.bar[0], 0); tc.b_wait = false; }
        // kind::i8 instruction descriptor: D s32 (bits 4-5 = 2), A and B unsigned 8-bit, both K-major, N >> 3 at 17, M >> 4 at 24
        const uint32_t idesc = (2u << 4) | ((N >> 3) << 17) | ((128u >> 4) << 24);
        const uint32_t a0 = smem_u32(tc.a) + aw0 / 8 * 256, b0 = smem_u32(tc.b) + boff;
        for (uint32_t kk = 0; kk < K / 32; kk++) {  // K = 32 bytes per MMA: two core matrices along K
            const uint64_t ad = p2tc_desc(a0 + kk * 256, P2TC_K2), bd = p2tc_desc(b0 + kk * 256, K);
            asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n"
                         ::"r"(tc.tmem + c0), "l"(ad), "l"(bd), "r"(idesc), "r"((uint32_t)acc | kk) : "memory");
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&tc.bar[1])) : "memory");
    }
    mbar_wait(&tc.bar[1], tc.phase);
    tc.phase ^= 1;
    tc_fence_after();
#else
    (void)first;
    const uint8_t* a = reinterpret_cast<const uint8_t*>(tc.w) + 4 * aw0;  // little-endian: word i = bytes 4i..4i+3
    const uint8_t* b = g_p2tc_host.b + boff;
    for (uint32_t n = 0; n < N; n++) {
        uint32_t s = acc ? tc.acc[c0 + n] : 0u;
        for (uint32_t k = 0; k < K; k++) s += (uint32_t)a[k] * b[p2tc_off(n, k, K)];
        tc.acc[c0 + n] = s;
    }
#endif
}
#ifdef __CUDA_ARCH__
// issue the load of 16 int32 columns [c0, c0 + 16) of this thread's TMEM lane; the values are valid after p2tc_ld_wait
__device__ __forceinline__ void p2tc_ld16(const P2Tc& tc, uint32_t c0, uint32_t* q) {
    const uint32_t addr = tc.tmem + ((tc.row & ~31u) << 16) + c0;  // a warp reads its own 32 TMEM lanes
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
                 : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]), "=r"(q[4]), "=r"(q[5]), "=r"(q[6]), "=r"(q[7]),
                   "=r"(q[8]), "=r"(q[9]), "=r"(q[10]), "=r"(q[11]), "=r"(q[12]), "=r"(q[13]), "=r"(q[14]), "=r"(q[15])
                 : "r"(addr) : "memory");
}
#endif
// 16 n int32 columns [c0, c0 + 16 n) of this state's TMEM lane: all loads issued, then one wait
HD void p2tc_cols(P2Tc& tc, uint32_t c0, uint32_t n, uint32_t* q) {
#ifdef __CUDA_ARCH__
#pragma unroll
    for (uint32_t i = 0; i < n; i++) p2tc_ld16(tc, c0 + 16 * i, q + 16 * i);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (uint32_t i = 0; i < 16 * n; i++) asm volatile("" : "+r"(q[i]));  // no read of q may move above the wait
#else
    for (uint32_t i = 0; i < 16 * n; i++) q[i] = tc.acc[c0 + i];
#endif
}
// REDC(sum_j 2^(8j) q_j) for planes q_j < 2^24: V < 2^49, split into its low and high words without 64-bit arithmetic.
// Canonical output.
HD uint32_t p2tc_reduce(const uint32_t* q) {
    const uint32_t a = q[1] + (q[0] >> 8), b = q[2] + (a >> 8), c = q[3] + (b >> 8);  // c = V >> 24
    const uint32_t lo = q[0] + (q[1] << 8) + (q[2] << 16) + (q[3] << 24), hi = c >> 8;
    const uint32_t m = lo * P_INV;
#ifdef __CUDA_ARCH__
    const uint32_t mp = __umulhi(m, P);
#else
    const uint32_t mp = (uint32_t)(((uint64_t)m * P) >> 32);
#endif
    const uint32_t r = hi - mp;  // (V - m p) / 2^32 in (-p, 2^17)
    return umin32(r, r + P);
}
// sum_{j<n} c_j d_j for signed |c_j|, |d_j| <= p/2 and n <= 4: |sum| < p^2 < 2^31 p, so one signed REDC lands in (-p, p).
// Canonical output (Montgomery: c_j carries the factor 2^32).
HD uint32_t p2tc_dot4(const int32_t* c, const int32_t* d, int n) {
    int64_t v = 0;
#pragma unroll
    for (int j = 0; j < n; j++) v += (int64_t)c[j] * d[j];
    const int32_t m = (int32_t)((uint32_t)v * P_INV);
#ifdef __CUDA_ARCH__
    const int32_t mp = __mulhi(m, (int32_t)P);
#else
    const int32_t mp = (int32_t)(((int64_t)m * (int64_t)P) >> 32);
#endif
    const uint32_t r = (uint32_t)((int32_t)(v >> 32) - mp);
    return umin32(r, r + P);
}

// out[i] = REDC of the 4 planes in TMEM columns c_lo + 4 i, for c_lo + 4 i < c_hi: x16 loads, one wait per 3 of them
HD void p2tc_read(P2Tc& tc, uint32_t c_lo, uint32_t c_hi, uint32_t* out) {
#pragma unroll
    for (uint32_t g = c_lo & ~15u; g < c_hi; g += 48) {
        uint32_t q[48];
        p2tc_cols(tc, g, umin32((c_hi - g + 15) / 16, 3u), q);
#pragma unroll
        for (uint32_t c = g < c_lo ? c_lo : g; c < c_hi && c < g + 48; c += 4) out[(c - c_lo) / 4] = p2tc_reduce(q + (c - g));
    }
}

HD void p2_mix_tc(uint32_t* s, P2Tc& tc) {
    const P2Consts& k = p2c();
    p2tc_mark(tc, P2_PROBE_N);
    p2_m_ext(s);
    p2_full_rounds(s, k.rc_first);
    p2tc_mark(tc, 0);
    // GEMM 1: a_r . v for r = 1..20 in columns 4(r-1) .. 4(r-1) + 3
    p2tc_put(tc, 0, s, 6);
    p2tc_mma(tc, 0, P2TC_K1, 0, 0, P2TC_N1, false, true);
    p2tc_mark(tc, 1);
    uint32_t w[P2TC_BW];  // the canonical deltas of the current block and its zero padding: its words of the A row
#pragma unroll
    for (uint32_t b = 0; b < P2TC_NB; b++) {
        const uint32_t r0 = b * P2TC_BS, r1 = umin32(r0 + P2TC_BS, 21u), rl = r0 ? r0 : 1;
        if (b > 0) {  // block GEMM b: the deltas of block b - 1 into the columns of rounds >= r0
            p2tc_put(tc, 24 + (b - 1) * P2TC_BW, w, P2TC_BW / 4);
            p2tc_mma(tc, 24 + (b - 1) * P2TC_BW, 4 * P2TC_BW, p2tc_blk_boff(b), p2tc_blk_c0(b), p2tc_blk_n(b), true, false);
            p2tc_mark(tc, 1 + 3 * b);
        }
        // L_r = a_r . v + sum_{j < r0} c_{r-j} delta_j for the rounds of this block
        uint32_t L[P2TC_BS];
        if (b == 0) L[0] = s[0];
        p2tc_read(tc, 4 * (rl - 1), 4 * (r1 - 1), L + (rl - r0));
        p2tc_mark(tc, 2 + 3 * b);
        // the S-box chain inside the block: v_r[0] = L_r + sum_{r0 <= j < r} c_{r-j} delta_j, delta_r kept balanced in (-p/2, p/2]
        int32_t dlt[P2TC_BS];
#pragma unroll
        for (uint32_t r = r0; r < r1; r++) {
            uint32_t y = L[r - r0];
#pragma unroll
            for (uint32_t j0 = r0; j0 < r; j0 += 4) {
                const uint32_t n = umin32(r - j0, 4u);
                int32_t cc[4], dd[4];
#pragma unroll
                for (uint32_t j = 0; j < 4; j++) if (j < n) { cc[j] = k.tri_c[r - j0 - j]; dd[j] = dlt[j0 - r0 + j]; }
                y = fadd(y, p2tc_dot4(cc, dd, (int)n));
            }
            const uint32_t d = fsub(sbox7_rc(y, k.rc_partial[r]), y);
            dlt[r - r0] = d > (P - 1) / 2 ? (int32_t)(d - P) : (int32_t)d;
            w[r - r0] = d;
        }
#pragma unroll
        for (uint32_t t = r1 - r0; t < P2TC_BW; t++) w[t] = 0;
        p2tc_mark(tc, 3 + 3 * b);
    }
    // GEMM 2: v_21 = M_I^21 v + sum_j delta_j M_I^(21-j) e0 (the v bytes and the earlier blocks are still in the A row)
    p2tc_put(tc, 24 + (P2TC_NB - 1) * P2TC_BW, w, P2TC_BW / 4);
    p2tc_mma(tc, 0, P2TC_K2, P2TC_B2_OFF, 0, P2TC_N2, false, false);
    p2tc_mark(tc, 1 + 3 * P2TC_NB);
    p2tc_read(tc, 0, P2TC_N2, s);
    p2tc_mark(tc, 2 + 3 * P2TC_NB);
    p2_full_rounds(s, k.rc_last);
    p2tc_mark(tc, 3 + 3 * P2TC_NB);
}

// The permutation the Merkle / permutation kernels run for one state per thread.  kAll: every thread of the block must
// call mix() (idle states on zeros) and end().
struct P2Perm {
#if P2_TC
    static constexpr bool kAll = true;
    static constexpr int kMinBlocks = 4;  // 4 x 128 TMEM columns per SM; caps registers at 128
    static constexpr size_t kSmem = P2TC_SMEM;
    P2Tc tc;
    HD P2Perm(const KCtx& cx, uint32_t* smem) { p2tc_begin(tc, cx, smem); }
    HD void mix(uint32_t* s) { p2_mix_tc(s, tc); }
    HD void end(const KCtx& cx) { p2tc_end(tc, cx); }
#else
    static constexpr bool kAll = false;
    static constexpr int kMinBlocks = 1;
    static constexpr size_t kSmem = 0;
    HD P2Perm(const KCtx&, uint32_t*) {}
    HD void mix(uint32_t* s) { p2_mix(s); }
    HD void end(const KCtx&) {}
#endif
};

// ---- kernels ------------------------------------------------------------------------------------
// Hal::hash_rows: leaf r = unpadded sponge over matrix[c * col_stride + r], c < cols.  Digest -> nodes[rows + r].
struct HashRowsKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t* smem, const uint32_t* matrix, uint64_t col_stride, uint32_t rows, uint32_t cols, uint32_t* leaves) {
        const uint64_t r = (uint64_t)cx.bx * cx.nt + cx.tid;
        const bool live = r < rows;
        if (!live && !P2Perm::kAll) return;
        P2Perm h(cx, smem);
        uint32_t s[24];
#pragma unroll
        for (int i = 0; i < 24; i++) s[i] = 0;
        const uint32_t* src = matrix + (live ? r : 0);
        uint32_t c = 0;
        for (; c + 16 <= cols; c += 16) {
#pragma unroll
            for (int i = 0; i < 16; i++) s[i] = live ? src[(uint64_t)(c + i) * col_stride] : 0u;
            h.mix(s);
        }
        if (c < cols || cols == 0) {
#pragma unroll
            for (int i = 0; i < 16; i++) s[i] = (live && c + i < cols) ? src[(uint64_t)(c + i) * col_stride] : 0u;
            h.mix(s);
        }
        if (live) {
            uint4* dst = reinterpret_cast<uint4*>(leaves + r * 8);
            dst[0] = make_uint4(s[0], s[1], s[2], s[3]);
            dst[1] = make_uint4(s[4], s[5], s[6], s[7]);
        }
        h.end(cx);
    }
};

// Hal::hash_fold for one level: nodes[i] = H(nodes[2i] || nodes[2i+1]) for i in [level_size, 2*level_size).
struct HashFoldKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t* smem, uint32_t* nodes, uint32_t level_size) {
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        const bool live = t < level_size;
        if (!live && !P2Perm::kAll) return;
        P2Perm h(cx, smem);
        const uint64_t i = level_size + (live ? t : 0);
        uint32_t s[24];
#pragma unroll
        for (int k = 0; k < 24; k++) s[k] = 0;
        if (live) {
            const uint4* in = reinterpret_cast<const uint4*>(nodes + 2 * i * 8);
            uint4 v0 = in[0], v1 = in[1], v2 = in[2], v3 = in[3];
            s[0] = v0.x; s[1] = v0.y; s[2] = v0.z; s[3] = v0.w; s[4] = v1.x; s[5] = v1.y; s[6] = v1.z; s[7] = v1.w;
            s[8] = v2.x; s[9] = v2.y; s[10] = v2.z; s[11] = v2.w; s[12] = v3.x; s[13] = v3.y; s[14] = v3.z; s[15] = v3.w;
        }
        h.mix(s);
        if (live) {
            uint4* dst = reinterpret_cast<uint4*>(nodes + i * 8);
            dst[0] = make_uint4(s[0], s[1], s[2], s[3]);
            dst[1] = make_uint4(s[4], s[5], s[6], s[7]);
        }
        h.end(cx);
    }
};

// The last levels of the tree in one block: levels of size top, top/2, ..., 1 (top <= block threads).
struct HashFoldTailKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* nodes, uint32_t top) {
        for (uint32_t level = top; level >= 1; level >>= 1) {
            for (uint32_t t = cx.tid; t < level; t += cx.nt) {
                const uint64_t i = level + t;
                uint32_t s[24];
#pragma unroll
                for (int k = 0; k < 16; k++) s[k] = nodes[2 * i * 8 + k];
#pragma unroll
                for (int k = 16; k < 24; k++) s[k] = 0;
                p2_mix(s);
#pragma unroll
                for (int k = 0; k < 8; k++) nodes[i * 8 + k] = s[k];
            }
#ifdef __CUDA_ARCH__
            __threadfence_block();
#endif
            cx.sync();
        }
    }
};

// ---- warp-cooperative permutation for the small upper levels of a tree --------------------------------------------
// With one thread per node a level of <= a few thousand nodes is pure latency (one permutation ~17 us, one launch per
// level).  Here a WARP computes one node: lane L < 24 owns state cell L, the S-boxes run 24-wide, the linear layers use
// shuffles (4-lane M4 groups, xor-butterfly column sums, warp all-reduce for the internal layer): ~3.5 us per node.
// 4x more instructions per node than the thread version, so it is used only where latency, not throughput, binds.
#ifdef __CUDA_ARCH__
struct WarpConsts { uint32_t rcf[4], rcl[4], d, dp; };
__device__ __forceinline__ WarpConsts wp2_consts(int lane) {
    const P2Consts& k = p2c();
    WarpConsts w;
    const int l = lane < 24 ? lane : 0;
#pragma unroll
    for (int r = 0; r < 4; r++) { w.rcf[r] = lane < 24 ? k.rc_first[r * 24 + l] : 0u; w.rcl[r] = lane < 24 ? k.rc_last[r * 24 + l] : 0u; }
    w.d = k.diag_std[l]; w.dp = k.diag_shoup[l];
    return w;
}
__device__ __forceinline__ uint32_t wp2_m_ext(uint32_t x, int lane) {
    const int q = lane & ~3;
    const uint32_t a = __shfl_sync(0xffffffffu, x, q), b = __shfl_sync(0xffffffffu, x, q + 1);
    const uint32_t c = __shfl_sync(0xffffffffu, x, q + 2), d = __shfl_sync(0xffffffffu, x, q + 3);
    const uint32_t t0 = fadd(a, b), t1 = fadd(c, d);
    const uint32_t t2 = fadd(fadd(b, b), t1), t3 = fadd(fadd(d, d), t0);
    uint32_t t4 = fadd(t1, t1); t4 = fadd(fadd(t4, t4), t3);
    uint32_t t5 = fadd(t0, t0); t5 = fadd(fadd(t5, t5), t2);
    const int r = lane & 3;
    const uint32_t out = r == 0 ? fadd(t3, t5) : r == 1 ? t5 : r == 2 ? fadd(t2, t4) : t4;
    uint32_t s = out;
    s = fadd(s, __shfl_xor_sync(0xffffffffu, s, 4));
    s = fadd(s, __shfl_xor_sync(0xffffffffu, s, 8));
    s = fadd(s, __shfl_xor_sync(0xffffffffu, s, 16));
    return lane < 24 ? fadd(out, s) : 0u;
}
__device__ __forceinline__ uint32_t wp2_mix(uint32_t x, int lane, const WarpConsts& w) {
    const P2Consts& k = p2c();
    x = wp2_m_ext(x, lane);
#pragma unroll
    for (int r = 0; r < 4; r++) x = wp2_m_ext(sbox7_rc(x, w.rcf[r]), lane);
#pragma unroll 1
    for (int r = 0; r < 21; r++) {
        const uint32_t y = sbox7_rc(x, k.rc_partial[r]);
        if (lane == 0) x = y;
        uint32_t s = x;
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) s = fadd(s, __shfl_xor_sync(0xffffffffu, s, off));
        x = lane < 24 ? fadd(s, fmul_const(x, w.d, w.dp)) : 0u;
    }
#pragma unroll
    for (int r = 0; r < 4; r++) x = wp2_m_ext(sbox7_rc(x, w.rcl[r]), lane);
    return x;
}
__device__ __forceinline__ void wp2_hash_pair(uint32_t* nodes, uint64_t i, int lane, const WarpConsts& w) {
    uint32_t x = lane < 16 ? nodes[2 * i * 8 + lane] : 0u;
    x = wp2_mix(x, lane, w);
    if (lane < 8) nodes[i * 8 + lane] = x;
}
#endif
// one level, one warp per node (device only; the emulator build keeps the thread-per-node path)
struct HashFoldWarpKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* nodes, uint32_t level_size) {
#ifdef __CUDA_ARCH__
        const int lane = cx.tid & 31;
        const uint64_t wid = ((uint64_t)cx.bx * cx.nt + cx.tid) >> 5;
        if (wid >= level_size) return;
        const WarpConsts w = wp2_consts(lane);
        wp2_hash_pair(nodes, (uint64_t)level_size + wid, lane, w);
#else
        (void)cx; (void)nodes; (void)level_size;
#endif
    }
};
// levels top, top/2, ..., 1 in one block of 32 warps
struct HashFoldWarpTailKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* nodes, uint32_t top) {
#ifdef __CUDA_ARCH__
        const int lane = cx.tid & 31, warp = cx.tid >> 5, nwarps = cx.nt >> 5;
        const WarpConsts w = wp2_consts(lane);
        for (uint32_t level = top; level >= 1; level >>= 1) {
            for (uint32_t t = warp; t < level; t += nwarps) wp2_hash_pair(nodes, (uint64_t)level + t, lane, w);
            __threadfence_block();
            __syncthreads();
        }
#else
        (void)cx; (void)nodes; (void)top;
#endif
    }
};

// poseidon2_mix on n independent states (parity probe for the permutation itself).
struct PermuteKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t* smem, uint32_t* states, uint32_t n) {
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        const bool live = t < n;
        if (!live && !P2Perm::kAll) return;
        P2Perm h(cx, smem);
        uint32_t s[24];
        for (int i = 0; i < 24; i++) s[i] = live ? states[t * 24 + i] : 0u;
        h.mix(s);
        if (live)
            for (int i = 0; i < 24; i++) states[t * 24 + i] = s[i];
        h.end(cx);
    }
};

struct Merkle {
    Dev* dev = nullptr;
    void init(Dev* d) {
        dev = d;
        p2_host_consts();
#if !defined(HFB200_EMU)
        CUDA_CHECK(cudaMemcpyToSymbol(g_p2c, &g_p2c_host, sizeof(P2Consts)));
        CUDA_CHECK(cudaMemcpyToSymbol(g_p2tc_b, g_p2tc_host.b, P2TC_B_BYTES));
#endif
    }
    // n independent states (24 words each) permuted in place
    void permute(uint32_t* states, uint32_t n) {
        dev->launch<PermuteKernel, 128, P2Perm::kMinBlocks>((n + 127) / 128, 1, 128, P2Perm::kSmem, states, n);
    }
    // Hal::hash_rows: leaves[r] = digest of row r (8 words each), matrix element (r, c) at matrix[c*col_stride + r]
    void hash_rows(const uint32_t* matrix, uint64_t col_stride, uint32_t rows, uint32_t cols, uint32_t* leaves) {
        const int T = 128;  // = the M of the tensor-core GEMMs (P2Perm)
        dev->launch<HashRowsKernel, 128, P2Perm::kMinBlocks>((rows + T - 1) / T, 1, T, P2Perm::kSmem, matrix, col_stride, rows, cols, leaves);
    }
#ifndef HFB200_EMU
    // big levels: one thread per node (throughput); <= 4096 nodes: one warp per node (latency)
    static uint32_t fold_warp_max() {
        static const uint32_t v = [] { const char* e = std::getenv("HFB200_FOLD_WARP_MAX"); const int x = e ? std::atoi(e) : 0; return x >= 64 ? (uint32_t)x : 4096u; }();
        return v;
    }
#endif
    // Hal::hash_fold of one level: nodes[level + i] = H(nodes[2 (level + i)] || nodes[2 (level + i) + 1]), i < level
    void fold_level(uint32_t* nodes, uint32_t level) {
        const int T = 128;
#ifndef HFB200_EMU
        if (level <= fold_warp_max()) { dev->launch<HashFoldWarpKernel, 256, 1>((level * 32 + 255) / 256, 1, 256, 0, nodes, level); return; }
#endif
        dev->launch<HashFoldKernel, 128, P2Perm::kMinBlocks>((level + T - 1) / T, 1, T, P2Perm::kSmem, nodes, level);
    }
    // nodes: 2*rows digests (heap layout).  matrix element (r, c) at matrix[c*col_stride + r].
    void build(const uint32_t* matrix, uint64_t col_stride, uint32_t rows, uint32_t cols, uint32_t* nodes) {
        hash_rows(matrix, col_stride, rows, cols, nodes + (uint64_t)rows * 8);
        uint32_t level = rows / 2;
#ifndef HFB200_EMU
        // <= 32 nodes: the remaining levels in one block
        for (; level > 32; level >>= 1) fold_level(nodes, level);
        if (level >= 1) dev->launch<HashFoldWarpTailKernel, 1024, 1>(1, 1, 1024, 0, nodes, level);
#else
        for (; level >= 512; level >>= 1) fold_level(nodes, level);
        if (level >= 1) dev->launch<HashFoldTailKernel, 256, 1>(1, 1, 256, 0, nodes, level);
#endif
    }
};

// ---- host-side sponge / RNG for the Fiat-Shamir transcript (WriteIOP) ---------------------------------
struct Digest8 { uint32_t w[8]; };

static inline Digest8 host_hash_elems(const uint32_t* in, size_t n) {
    p2_host_consts();
    uint32_t s[24] = {0};
    size_t used = 0; bool any = false;
    for (size_t i = 0; i < n; i++) {
        s[used++] = in[i];
        if (used == 16) { p2_mix(s); used = 0; any = true; }
    }
    if (used != 0 || !any) { for (size_t k = used; k < 16; k++) s[k] = 0; p2_mix(s); }
    Digest8 d; for (int i = 0; i < 8; i++) d.w[i] = s[i];
    return d;
}

struct HostRng {
    uint32_t cells[24] = {0};
    int pool_used = 0;
    // Poseidon2Rng::mix: a permutation first when elements were drawn since the last mix (upstream: "if switching from squeezing,
    // do a poseidon2 mix"), then add the 8 digest words into the rate and permute
    void mix(const uint32_t* d8) {
        p2_host_consts();
        if (pool_used != 0) { p2_mix(cells); pool_used = 0; }
        for (int i = 0; i < 8; i++) cells[i] = fadd(cells[i], d8[i]);
        p2_mix(cells);
    }
    uint32_t random_elem() { if (pool_used == 16) { p2_mix(cells); pool_used = 0; } return cells[pool_used++]; }
    E4 random_ext() { uint32_t a = random_elem(), b = random_elem(), c = random_elem(), d = random_elem(); return e4(a, b, c, d); }
    uint32_t random_bits(unsigned bits) {
        uint32_t v = from_mont(random_elem());
        for (int i = 0; i < 3; i++) { uint32_t n = from_mont(random_elem()); if (v == 0) v = n; }
        return v & (uint32_t)((1ull << bits) - 1);
    }
};

// ---- transcript header ------------------------------------------------------------------------------------------------
// risc0-circuit-rv32im `SegmentProver::prove` / risc0-zkp `verify`: "At the start of the protocol, seed the Fiat-Shamir
// transcript with context information about the proof system and circuit":
//   commit(H(PROOF_SYSTEM_INFO.encode())); commit(H(CIRCUIT_INFO.encode()));         (`ProtocolInfo`: 16 bytes, one element per byte)
//   header = globals ++ [po2 as a raw word]; commit(H(header)); write header
// Returns the header digest.  Host code, shared by the prover (both transcript modes) and the verifier.
static constexpr char PROOF_SYSTEM_INFO[17] = "RISC0_STARK:v1__";      // risc0-zkp PROOF_SYSTEM_INFO
static constexpr char BUILTIN_CIRCUIT_INFO[17] = "SYNTH_RV32IM:v1_";   // the declared stand-in circuit names itself
static constexpr char DEFAULT_IR_CIRCUIT_INFO[17] = "RV32IM:v2_______"; // data-defined circuits: upstream's rv32im-v2 string unless given
// dst[17] <- the circuit's info string: built-in circuit, data-defined with its own 16 bytes, or data-defined default
static inline void set_circuit_info(char* dst, bool data_defined, const uint8_t* info16) {
    bool given = false;
    if (info16) for (int i = 0; i < 16; i++) given = given || info16[i] != 0;
    if (!data_defined) std::memcpy(dst, BUILTIN_CIRCUIT_INFO, 17);
    else if (given) { std::memcpy(dst, info16, 16); dst[16] = 0; }
    else std::memcpy(dst, DEFAULT_IR_CIRCUIT_INFO, 17);
}
static inline Digest8 protocol_info_digest(const char* info16) {
    uint32_t e[16];
    for (int i = 0; i < 16; i++) e[i] = to_mont((uint32_t)(uint8_t)info16[i]);
    return host_hash_elems(e, 16);
}
static inline Digest8 transcript_header(HostRng& rng, const char* circuit_info16, const uint32_t* globals, size_t n_globals, uint32_t po2) {
    rng.mix(protocol_info_digest(PROOF_SYSTEM_INFO).w);
    rng.mix(protocol_info_digest(circuit_info16).w);
    std::vector<uint32_t> header(globals, globals + n_globals);
    header.push_back(po2);
    const Digest8 d = host_hash_elems(header.data(), header.size());
    rng.mix(d.w);
    return d;
}

}  // namespace hf
