// Circuit plug-in "synth-rv32im-shape v1" on the device: witness stand-in, step_accum, eval_check.
// Plays the role of risc0-circuit-rv32im-sys 4.0.2's generated kernels (witgen steps, `step_accum`,
// `eval_check`/`poly_fp`; /root/reference/Cargo.lock:3121-3132) -- generated code that cannot be obtained
// here, so the circuit is a DECLARED synthetic one with the same shape (DESIGN.md section "circuit").
// Definition (independently restated by oracle/circuit.h):
//   groups: ACCUM=0 (w_accum = 4*n_chains), CODE=1 (w_code), DATA=2 (w_data = 2*n_free)
//   code:   c0 active (rows < N-1994), c1 first-row flag, c2 last-active flag, c3 cycle, c4.. pseudo-random
//   data:   free columns f_0..f_{F-1}; derived columns g_k = expr_k(f taps), k < F
//             k%4==0: A*B + C      1: A*B*C + P'     2: (A+X)*B*C*D     3: P'*B + C*D + X      (P' = back 1)
//   accum:  Fp4 chains: acc_r(i) = (first ? 1 : acc_r(i-1)) * (data[src_r](i) + mix_r)
//   constraints (all gated by `active`, degree <= 5), mixed with successive powers of poly_mix:
//     F derived, 4*n_chains accum components, 1 global tie  first*(f_0 - global_0)
#pragma once
#include <algorithm>
#include "dev.cuh"
#include "blind.cuh"

namespace hf {

static constexpr uint32_t ZK_CYCLES = 1994, N_GLOBAL = 32, CODE_FIXED = 4;
enum { GROUP_ACCUM = 0, GROUP_CODE = 1, GROUP_DATA = 2 };
static constexpr uint64_t CODE_SEED = 0x636F6465ull;

HD uint64_t splitmix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
HD uint32_t synth_value(uint64_t seed, uint32_t col, uint32_t row) {
    return to_mont((uint32_t)(splitmix64(seed ^ (((uint64_t)col << 32) | row)) % P));
}
struct CircuitDev {
    uint32_t w_code, w_data, w_accum, n_free, n_prev, n_chains;
    const uint16_t* picks;      // [n_free][6] : a, b, c, d, p, x   (device memory)
    const uint16_t* chain_src;  // [n_chains]
    HD uint32_t n_constraints() const { return n_free + 4 * n_chains + 1; }
};

HD uint32_t derived_expr(uint32_t k, uint32_t A, uint32_t B, uint32_t C, uint32_t D, uint32_t Pp, uint32_t X) {
    switch (k & 3u) {
        case 0: return fadd(fmul(A, B), C);
        case 1: return fadd(fmul(fmul(A, B), C), Pp);
        case 2: return fmul(fmul(fmul(fadd(A, X), B), C), D);
        default: return fadd(fadd(fmul(Pp, B), fmul(C, D)), X);
    }
}

// ---- witness stand-in ----------------------------------------------------------------------------
struct GenCodeKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* code, uint32_t w_code, uint32_t po2) {
        const uint64_t n = 1ull << po2, act = n - ZK_CYCLES;
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (t >= (uint64_t)w_code * n) return;
        const uint32_t c = (uint32_t)(t >> po2), r = (uint32_t)(t & (n - 1));
        uint32_t v = 0;
        if (r < act) {
            if (c == 0) v = ONE;
            else if (c == 1) v = r == 0 ? ONE : 0u;
            else if (c == 2) v = r == act - 1 ? ONE : 0u;
            else if (c == 3) v = to_mont(r % P);
            else v = synth_value(CODE_SEED, c, r);
        }
        code[t] = v;
    }
};
struct GenFreeKernel {  // free columns (active rows) + blinding rows of every data column
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* data, CircuitDev cd, uint32_t po2, uint64_t trace_seed, BlindKey blind, uint32_t global0) {
        const uint64_t n = 1ull << po2, act = n - ZK_CYCLES;
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (t >= (uint64_t)cd.w_data * n) return;
        const uint32_t c = (uint32_t)(t >> po2), r = (uint32_t)(t & (n - 1));
        if (r >= act) data[t] = blind_value(blind, GROUP_DATA, c, r);
        else if (c < cd.n_free) data[t] = (c == 0 && r == 0) ? global0 : synth_value(trace_seed, c, r);
    }
};
struct GenDerivedKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* data, const uint32_t* code, CircuitDev cd, uint32_t po2) {
        const uint64_t n = 1ull << po2, act = n - ZK_CYCLES;
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (t >= (uint64_t)cd.n_free * n) return;
        const uint32_t k = (uint32_t)(t >> po2), r = (uint32_t)(t & (n - 1));
        if (r >= act) return;
        const uint16_t* pk = cd.picks + 6 * k;
        const uint64_t rp = (r + n - 1) & (n - 1);
        data[(uint64_t)(cd.n_free + k) * n + r] = derived_expr(k, data[(uint64_t)pk[0] * n + r], data[(uint64_t)pk[1] * n + r], data[(uint64_t)pk[2] * n + r],
                                                               data[(uint64_t)pk[3] * n + r], data[(uint64_t)pk[4] * n + rp], code[(uint64_t)pk[5] * n + r]);
    }
};

// ---- step_accum: Fp4 running products (three-phase scan) -----------------------------------------------
// The two scans of hfb200_segment_accum_scan: running products (grand products, Hal::prefix_products) and running sums (LogUp).
enum : int { SCAN_PRODUCT = 0, SCAN_SUM = 1 };
HD E4 scan_op(int kind, const E4& a, const E4& b) { return kind == SCAN_SUM ? e4_add(a, b) : e4_mul(a, b); }
HD E4 scan_identity(int kind) { return kind == SCAN_SUM ? e4_zero() : e4_one(); }

// In-place inclusive scan (Fp4 product, or sum for kind = SCAN_SUM) of buf0[0..n) in shared memory; buf1 is scratch. Result in
// the returned buffer.
HD E4* block_scan_e4(const KCtx& cx, E4* buf0, E4* buf1, uint32_t n, int kind = SCAN_PRODUCT) {
    E4 *src = buf0, *dst = buf1;
    for (uint32_t d = 1; d < n; d <<= 1) {
        for (uint32_t i = cx.tid; i < n; i += cx.nt) dst[i] = i >= d ? scan_op(kind, src[i - d], src[i]) : src[i];
        cx.sync();
        E4* t = src; src = dst; dst = t;
    }
    return src;
}

static constexpr uint32_t ACC_ITEMS = 256, ACC_PER = 8, ACC_RPB = ACC_ITEMS * ACC_PER;  // rows per block

// mode 0: write the block's total product to partial[chain * nblk + blk]
// mode 1: read the exclusive block offset from partial[...] and write the running products (+ blinding rows)
struct AccumKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t* sm, uint32_t* accum, const uint32_t* data, const uint32_t* mix, E4* partial, CircuitDev cd, uint32_t po2, BlindKey blind, int mode,
                       const BlindKey* blind_dev = nullptr) {
        // blind_dev != NULL: the key lives in device memory (CUDA-graph replay: a by-value key would be frozen into the graph)
        if (blind_dev) blind = *blind_dev;
        const uint64_t n = 1ull << po2, act = n - ZK_CYCLES;
        const uint32_t chain = cx.by, blk = cx.bx, nblk = cx.gx;
        const uint32_t* src = data + (uint64_t)cd.chain_src[chain] * n;
        const E4 m = e4(mix[4 * chain], mix[4 * chain + 1], mix[4 * chain + 2], mix[4 * chain + 3]);
        E4* buf0 = reinterpret_cast<E4*>(sm);
        E4* buf1 = buf0 + ACC_ITEMS;
        const uint64_t row0 = (uint64_t)blk * ACC_RPB;
        for (uint32_t it = cx.tid; it < ACC_ITEMS; it += cx.nt) {
            E4 pr = e4_one();
            for (uint32_t j = 0; j < ACC_PER; j++) {
                const uint64_t r = row0 + (uint64_t)it * ACC_PER + j;
                if (r < act) { E4 t = m; t.c[0] = fadd(t.c[0], src[r]); pr = e4_mul(pr, t); }
            }
            buf0[it] = pr;
        }
        cx.sync();
        E4* sc = block_scan_e4(cx, buf0, buf1, ACC_ITEMS);
        if (mode == 0) {
            if (cx.tid == 0) partial[(uint64_t)chain * nblk + blk] = sc[ACC_ITEMS - 1];
            return;
        }
        const E4 off = partial[(uint64_t)chain * nblk + blk];
        for (uint32_t it = cx.tid; it < ACC_ITEMS; it += cx.nt) {
            E4 pr = it == 0 ? off : e4_mul(off, sc[it - 1]);
            for (uint32_t j = 0; j < ACC_PER; j++) {
                const uint64_t r = row0 + (uint64_t)it * ACC_PER + j;
                if (r >= n) break;
                if (r < act) {
                    E4 t = m; t.c[0] = fadd(t.c[0], src[r]); pr = e4_mul(pr, t);
                    for (int k = 0; k < 4; k++) accum[(uint64_t)(4 * chain + k) * n + r] = pr.c[k];
                } else {
                    for (int k = 0; k < 4; k++) accum[(uint64_t)(4 * chain + k) * n + r] = blind_value(blind, GROUP_ACCUM, 4 * chain + k, (uint32_t)r);
                }
            }
        }
    }
};
// Exclusive scan of the per-block products of one chain (grid.y = chain, one block): partial[i] <- prod_{j<i} (sum for SCAN_SUM).
struct AccumOffsetsKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t* sm, E4* partial, uint32_t nblk, int kind = SCAN_PRODUCT) {
        E4* buf0 = reinterpret_cast<E4*>(sm);
        E4* buf1 = buf0 + nblk;
        E4* p = partial + (uint64_t)cx.by * nblk;
        for (uint32_t i = cx.tid; i < nblk; i += cx.nt) buf0[i] = p[i];
        cx.sync();
        E4* sc = block_scan_e4(cx, buf0, buf1, nblk, kind);
        for (uint32_t i = cx.tid; i < nblk; i += cx.nt) p[i] = i == 0 ? scan_identity(kind) : sc[i - 1];
    }
};

// ---- hfb200_segment_accum_scan: the same two-pass scan over terms the CALLER wrote into the accum columns --------------------
// Chain c = first_chain + grid.y lives in columns 4c..4c+3; rows [0, rows) are scanned in place, ACC_RPB rows per block.  The
// block's rows are staged in shared memory with coalesced loads (one E4 of padding every ACC_PER elements, so that the
// per-thread runs of ACC_PER consecutive rows sit in different banks), reduced per thread, scanned across the block, and (mode 1)
// written back with coalesced stores.  mode 0: block totals to partial[chain * nblk + blk]; mode 1: apply the exclusive offsets
// AccumOffsetsKernel left there.
static constexpr uint32_t SCAN_TILE = ACC_RPB + ACC_RPB / ACC_PER;  // padded tile, E4 elements
HD uint32_t scan_slot(uint32_t i) { return i + i / ACC_PER; }
struct AccumScanKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t* sm, uint32_t* accum, uint64_t n, uint64_t rows, uint32_t first_chain, int kind, E4* partial, int mode) {
        const uint32_t chain = first_chain + cx.by, blk = cx.bx, nblk = cx.gx;
        uint32_t* col = accum + (uint64_t)4 * chain * n;
        E4* tile = reinterpret_cast<E4*>(sm);
        E4* buf0 = tile + SCAN_TILE;
        E4* buf1 = buf0 + ACC_ITEMS;
        const uint64_t row0 = (uint64_t)blk * ACC_RPB;
        const uint32_t cnt = (uint32_t)(rows - row0 < ACC_RPB ? rows - row0 : ACC_RPB);
        for (uint32_t i = cx.tid; i < cnt; i += cx.nt) {
            const uint64_t r = row0 + i;
            tile[scan_slot(i)] = e4(col[r], col[n + r], col[2 * n + r], col[3 * n + r]);
        }
        cx.sync();
        for (uint32_t it = cx.tid; it < ACC_ITEMS; it += cx.nt) {
            E4 pr = scan_identity(kind);
            for (uint32_t j = 0; j < ACC_PER; j++) {
                const uint32_t i = it * ACC_PER + j;
                if (i < cnt) pr = scan_op(kind, pr, tile[scan_slot(i)]);
            }
            buf0[it] = pr;
        }
        cx.sync();
        E4* sc = block_scan_e4(cx, buf0, buf1, ACC_ITEMS, kind);
        if (mode == 0) {
            if (cx.tid == 0) partial[(uint64_t)cx.by * nblk + blk] = sc[ACC_ITEMS - 1];
            return;
        }
        const E4 off = partial[(uint64_t)cx.by * nblk + blk];
        for (uint32_t it = cx.tid; it < ACC_ITEMS; it += cx.nt) {
            E4 pr = it == 0 ? off : scan_op(kind, off, sc[it - 1]);
            for (uint32_t j = 0; j < ACC_PER; j++) {
                const uint32_t i = it * ACC_PER + j;
                if (i >= cnt) break;
                pr = scan_op(kind, pr, tile[scan_slot(i)]);
                tile[scan_slot(i)] = pr;
            }
        }
        cx.sync();
        for (uint32_t i = cx.tid; i < cnt; i += cx.nt) {
            const uint64_t r = row0 + i;
            const E4 v = tile[scan_slot(i)];
            col[r] = v.c[0]; col[n + r] = v.c[1]; col[2 * n + r] = v.c[2]; col[3 * n + r] = v.c[3];
        }
    }
};
// The last zk rows of every column of one group from the segment's key, one thread per element, consecutive threads on
// consecutive rows of a column (coalesced stores).  GROUP_ACCUM: hfb200_segment_accum_blind, exactly the values AccumKernel
// mode 1 writes there; GROUP_DATA: hfb200_segment_data_blind, exactly the values GenFreeKernel writes there.
struct BlindRowsKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* cols, uint32_t w, uint32_t po2, uint32_t zk, uint32_t group, BlindKey blind) {
        const uint64_t n = 1ull << po2;
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (t >= (uint64_t)w * zk) return;
        const uint32_t c = (uint32_t)(t / zk), r = (uint32_t)(n - zk + t % zk);
        cols[(uint64_t)c * n + r] = blind_value(blind, group, c, r);
    }
};

// ---- eval_check (CircuitHal::eval_check): constraint polynomial / vanishing polynomial on the LDE domain ----
struct EvalCheckArgs {
    const uint32_t *ev_accum, *ev_code, *ev_data;  // [w][domain]
    uint32_t* check;                               // [4][domain]
    const E4* mixpow;                              // poly_mix^j, j < n_constraints (device)
    const uint32_t* mix;                           // accum mix elems (device) [4*n_chains]
    uint32_t global0;
    const uint32_t* global0_dev;                   // non-NULL: globals[0] is read from device memory instead (CUDA-graph replay)
    uint32_t yinv[4];                              // 1/((3 w_4N^i)^N - 1) depends on i mod 4 only
    uint32_t po2;
    uint32_t rows_per_block;
    CircuitDev cd;
};
// One thread per LDE row; every operand is a coalesced 128-byte line across the warp (served by L2 after the first
// touch).  A shared-memory row-tile variant (stage all 272 columns of 64 rows, two threads per row) was measured at
// 20.2 ms against 3.8 ms for this kernel: 78 KB of tile per 128 threads leaves 8 warps per SM (profiles/README.md).
#ifndef EC_UNROLL
#define EC_UNROLL 4
#endif
static constexpr int kEcUnroll = EC_UNROLL;  // constraints whose operand loads are in flight together
struct EvalCheckKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t* sm, EvalCheckArgs p) {
        const CircuitDev& cd = p.cd;
        const uint32_t nc = cd.n_constraints();
        E4* mp = reinterpret_cast<E4*>(sm);
        uint16_t* spk = reinterpret_cast<uint16_t*>(mp + nc);  // column picks staged in shared memory: the operand addresses
        for (uint32_t i = cx.tid; i < nc; i += cx.nt) mp[i] = p.mixpow[i];       // no longer wait on a global load
        for (uint32_t i = cx.tid; i < 6 * cd.n_free; i += cx.nt) spk[i] = cd.picks[i];
        cx.sync();
        const uint64_t domain = 4ull << p.po2, dmask = domain - 1;
        for (uint32_t rr = cx.tid; rr < p.rows_per_block; rr += cx.nt) {
            const uint64_t i = (uint64_t)cx.bx * p.rows_per_block + rr;
            if (i >= domain) break;
            const uint64_t ib = (i + domain - 4) & dmask;  // back 1 on the x4 domain
            const uint32_t active = p.ev_code[i], first = p.ev_code[domain + i];
            E4A lt = e4a_zero();  // sum_j mixpow[j] * constraint_j in lazy 64-bit accumulators (field.cuh)
            uint32_t j = 0;
#pragma unroll kEcUnroll
            for (uint32_t k = 0; k < cd.n_free; k++, j++) {
                const uint16_t* pk = spk + 6 * k;
                const uint32_t e = derived_expr(k, p.ev_data[(uint64_t)pk[0] * domain + i], p.ev_data[(uint64_t)pk[1] * domain + i], p.ev_data[(uint64_t)pk[2] * domain + i],
                                                p.ev_data[(uint64_t)pk[3] * domain + i], p.ev_data[(uint64_t)pk[4] * domain + ib], p.ev_code[(uint64_t)pk[5] * domain + i]);
                // every constraint but the last carries the selector `active`: it is factored out of the sum (one Fp4 scale
                // at the end instead of one product per constraint; exact arithmetic, same value)
                e4a_mac(lt, mp[j], fsub(p.ev_data[(uint64_t)(cd.n_free + k) * domain + i], e));
            }
            const uint32_t nf = fsub(ONE, first);
            for (uint32_t r = 0; r < cd.n_chains; r++) {
                E4 acc, s, t;
                for (int k = 0; k < 4; k++) {
                    acc.c[k] = p.ev_accum[(uint64_t)(4 * r + k) * domain + i];
                    s.c[k] = fmul(nf, p.ev_accum[(uint64_t)(4 * r + k) * domain + ib]);
                    t.c[k] = p.mix[4 * r + k];
                }
                s.c[0] = fadd(s.c[0], first);
                t.c[0] = fadd(t.c[0], p.ev_data[(uint64_t)cd.chain_src[r] * domain + i]);
                const E4 pr = e4_mul(s, t);
                for (int k = 0; k < 4; k++, j++) e4a_mac(lt, mp[j], fsub(acc.c[k], pr.c[k]));
            }
            E4A lf = e4a_zero();
            e4a_mac(lf, mp[j], fmul(first, fsub(p.ev_data[i], p.global0_dev ? *p.global0_dev : p.global0)));
            const E4 tot = e4_add(e4_scale(e4a_redc(lt), active), e4a_redc(lf));
            const uint32_t yi = p.yinv[i & 3];
            for (int k = 0; k < 4; k++) p.check[(uint64_t)k * domain + i] = fmul(tot.c[k], yi);
        }
    }
};

struct CircuitHost {
    CircuitDev cd{};
    uint32_t n_taps = 0;
    uint16_t* tab_mem = nullptr;
    std::vector<uint16_t> h_picks, h_chain_src;
    void init(Dev* dev, uint32_t wc, uint32_t wd, uint32_t wa) {
        init_host(wc, wd, wa);
        tab_mem = (uint16_t*)dev->alloc((h_picks.size() + h_chain_src.size()) * 2 + 16);
        dev->h2d(tab_mem, h_picks.data(), h_picks.size() * 2);
        dev->h2d(tab_mem + h_picks.size(), h_chain_src.data(), h_chain_src.size() * 2);
        dev->sync();
        cd.picks = tab_mem;
        cd.chain_src = tab_mem + h_picks.size();
    }
    // host tables only (also what the verifier needs)
    void init_host(uint32_t wc, uint32_t wd, uint32_t wa) {
        if (wc < CODE_FIXED + 1 || wd < 8 || (wd & 3) || wa < 4 || (wa & 3) || wc > 4096 || wd > 4096 || wa > 4096) throw Err("circuit: unsupported widths");
        cd.w_code = wc; cd.w_data = wd; cd.w_accum = wa;
        cd.n_free = wd / 2; cd.n_prev = cd.n_free / 2; cd.n_chains = wa / 4;
        const uint32_t F = cd.n_free;
        h_picks.resize(6 * F);
        for (uint32_t k = 0; k < F; k++) {
            h_picks[6 * k + 0] = (uint16_t)(k % F);
            h_picks[6 * k + 1] = (uint16_t)((5 * k + 1) % F);
            h_picks[6 * k + 2] = (uint16_t)((11 * k + 2) % F);
            h_picks[6 * k + 3] = (uint16_t)((17 * k + 3) % F);
            h_picks[6 * k + 4] = (uint16_t)((7 * k + 1) % cd.n_prev);
            h_picks[6 * k + 5] = (uint16_t)(CODE_FIXED + k % (wc - CODE_FIXED));
        }
        h_chain_src.resize(cd.n_chains);
        for (uint32_t r = 0; r < cd.n_chains; r++) h_chain_src[r] = (uint16_t)((13 * r + 5) % wd);
        // taps: accum all {0,1}; code all {0}; data: columns < n_prev {0,1}, others {0}
        n_taps = 2 * wa + wc + wd + cd.n_prev;
    }
    void destroy(Dev* dev) { dev->free(tab_mem); tab_mem = nullptr; }
    // widths only (data-defined circuit: taps / constraints live in GenericCircuitHost)
    uint32_t n_mix_data = 0;
    bool builtin = true;
    void init_widths(uint32_t wc, uint32_t wd, uint32_t wa, uint32_t n_taps_, uint32_t n_mix_) {
        cd = CircuitDev{};
        cd.w_code = wc; cd.w_data = wd; cd.w_accum = wa;
        n_taps = n_taps_; n_mix_data = n_mix_; builtin = false;
    }
    uint32_t group_width(int g) const { return g == GROUP_ACCUM ? cd.w_accum : g == GROUP_CODE ? cd.w_code : cd.w_data; }
    uint32_t group_back1(int g) const { return g == GROUP_ACCUM ? cd.w_accum : g == GROUP_CODE ? 0u : cd.n_prev; }
    uint32_t n_regs() const { return cd.w_accum + cd.w_code + cd.w_data; }
    uint32_t n_mix() const { return builtin ? 4 * cd.n_chains : n_mix_data; }
};

}  // namespace hf

// =====================================================================================================================
// Circuit as DATA: the plug-in form of SURVEY.md section 8b (`hfb200_circuit_register`): a tap table (upstream TapSet:
// sorted (group, offset, back)) and the constraint polynomial as a step list in the shape of upstream's
// `risc0_zkp::adapter::PolyExtStepDef` (Const / Get / GetGlobal / Add / Sub / Mul / True / AndEqz / AndCond).  Upstream
// turns that IR into generated C++/CUDA for the prover; here the host compiles it once into a register-machine bytecode
// (SSA values -> reusable slots by last-use analysis; the `mul` of every MixState is a static power of poly_mix, so only
// `tot` lives at run time) and one interpreter kernel evaluates it per LDE row.  witgen / step_accum of a data-defined
// circuit stay with the caller (two-phase API: segment_begin -> mix -> caller's accum -> segment_finish).
// =====================================================================================================================
namespace hf {

enum : uint32_t { IR_CONST = 0, IR_GET = 1, IR_GET_GLOBAL = 2, IR_ADD = 3, IR_SUB = 4, IR_MUL = 5, IR_TRUE = 6, IR_AND_EQZ = 7, IR_AND_COND = 8 };
struct IrStep { uint32_t op, a, b, c; };
struct IrTap { uint32_t group, offset, back; };

enum : uint16_t { BC_CONST = 0, BC_GET, BC_GETG, BC_ADD, BC_SUB, BC_MUL, BC_MTRUE, BC_MEQZ, BC_MCOND };
struct BcIns { uint16_t op, dst; uint32_t a, b, c; };  // 16 bytes

static constexpr uint32_t GEN_MAX_BACKS = 4;   // distinct `back` values over the whole tap set
static constexpr uint32_t GEN_MAX_COMBOS = 8;  // distinct per-register back sets

struct GenReg { uint32_t group, offset, combo, tap_begin, size; };

struct GenericCircuitHost {
    bool active = false;
    uint32_t w[3] = {0, 0, 0};  // accum, code, data
    uint32_t n_mix = 0;
    std::vector<IrTap> taps;
    std::vector<GenReg> regs;
    std::vector<std::vector<uint32_t>> combos;
    std::vector<uint32_t> combo_begin;
    std::vector<uint32_t> backs;             // distinct back values, sorted (slot s <-> backs[s])
    std::vector<BcIns> prog;   // the whole constraint polynomial as ONE program (verifier, reference for the chunks)
    uint32_t n_fp_slots = 0, n_mix_slots = 0, ret_slot = 0, n_mixpow = 0;
    // The same polynomial cut along its top-level AndEqz / AndCond chain into CHUNKS of ~400 steps: the sum
    // tot = sum_k mix^e_k * term_k splits between any two elements whose chunk does not read one of them as a value (make_chunks),
    // so every chunk is a self-contained program (its Gets re-issued, its chain head starting at the exponent the prefix reached)
    // that adds its partial sum into the check buffer.  At rv32im scale (tens of
    // thousands of steps, a thousand taps) one straight-line kernel does not compile in useful time and keeps ~1000 values
    // live; chunks compile in parallel in seconds and keep the live set small (upstream splits its generated eval_check the same way).
    struct Chunk { std::vector<BcIns> prog; uint32_t n_fp_slots = 0, n_mix_slots = 0, ret_slot = 0; BcIns* d_prog = nullptr; };
    std::vector<Chunk> chunks;
    // device copies
    BcIns* d_prog = nullptr;
    uint8_t* d_colmask[3] = {nullptr, nullptr, nullptr};  // per column: bit s set <=> tapped at backs[s]
    uint8_t* d_regcombo = nullptr;                         // per register (taps order)
    uint32_t* d_regcol = nullptr;                          // per register: group << 28 | offset

    uint32_t back_slot(uint32_t back) const { for (uint32_t s = 0; s < backs.size(); s++) if (backs[s] == back) return s; throw Err("circuit: unknown back"); }

    void init(Dev* dev, uint32_t wc, uint32_t wd, uint32_t wa, uint32_t n_mix_, const IrTap* tp, size_t n_taps, const IrStep* st, size_t n_steps, uint32_t ret) {
        if (!tp || !st || n_taps == 0 || n_steps == 0) throw Err("circuit: empty tap table or step list");
        w[GROUP_ACCUM] = wa; w[GROUP_CODE] = wc; w[GROUP_DATA] = wd; n_mix = n_mix_;
        if (wc == 0 || wd == 0 || wa == 0 || wc > 65535 || wd > 65535 || wa > 65535) throw Err("circuit: bad group widths");
        analyze_taps(tp, n_taps);
        compile(st, n_steps, ret);
        if (!dev) return;  // analysis only (hfb200_ir_source, verifier)
        upload(dev);
    }
    // tap table -> registers, tap sets ("combos"), distinct backs.  w[] must be set.
    void analyze_taps(const IrTap* tp, size_t n_taps) {
        regs.clear(); backs.clear();
        taps.assign(tp, tp + n_taps);
        std::vector<std::vector<uint32_t>> backsets;
        for (size_t i = 0; i < taps.size();) {
            if (taps[i].group > 2 || taps[i].offset >= w[taps[i].group]) throw Err("circuit: tap out of range");
            size_t j = i; std::vector<uint32_t> b;
            while (j < taps.size() && taps[j].group == taps[i].group && taps[j].offset == taps[i].offset) {
                if (j > i && taps[j].back <= taps[j - 1].back) throw Err("circuit: taps must be sorted by (group, offset, back)");
                b.push_back(taps[j++].back);
            }
            if (j < taps.size() && (taps[j].group < taps[i].group || (taps[j].group == taps[i].group && taps[j].offset < taps[i].offset))) throw Err("circuit: taps must be sorted by (group, offset, back)");
            if (b.size() > 4) throw Err("circuit: more than 4 taps on one register");
            regs.push_back(GenReg{taps[i].group, taps[i].offset, 0, (uint32_t)i, (uint32_t)(j - i)});
            backsets.push_back(b);
            for (uint32_t x : b) if (std::find(backs.begin(), backs.end(), x) == backs.end()) backs.push_back(x);
            i = j;
        }
        std::sort(backs.begin(), backs.end());
        if (backs.size() > GEN_MAX_BACKS) throw Err("circuit: more than 4 distinct back values");
        if (backs.back() >= 1024) throw Err("circuit: back too large");
        combos = backsets;
        std::sort(combos.begin(), combos.end());
        combos.erase(std::unique(combos.begin(), combos.end()), combos.end());
        if (combos.size() > GEN_MAX_COMBOS) throw Err("circuit: more than 8 distinct tap sets");
        combo_begin.assign(1, 0);
        for (auto& c : combos) combo_begin.push_back(combo_begin.back() + (uint32_t)c.size());
        for (size_t r = 0; r < regs.size(); r++) regs[r].combo = (uint32_t)(std::lower_bound(combos.begin(), combos.end(), backsets[r]) - combos.begin());
    }
    void upload(Dev* dev) {
        // device tables
        d_prog = (BcIns*)dev->alloc(prog.size() * sizeof(BcIns));
        dev->h2d(d_prog, prog.data(), prog.size() * sizeof(BcIns));
        for (Chunk& c : chunks) {
            c.d_prog = (BcIns*)dev->alloc(c.prog.size() * sizeof(BcIns));
            dev->h2d(c.d_prog, c.prog.data(), c.prog.size() * sizeof(BcIns));
        }
        for (int g = 0; g < 3; g++) {
            std::vector<uint8_t> m(w[g], 0);
            for (const IrTap& t : taps) if ((int)t.group == g) m[t.offset] |= (uint8_t)(1u << back_slot(t.back));
            d_colmask[g] = (uint8_t*)dev->alloc(m.size());
            dev->h2d(d_colmask[g], m.data(), m.size());
        }
        std::vector<uint8_t> rc(regs.size());
        std::vector<uint32_t> rcol(regs.size());
        for (size_t r = 0; r < regs.size(); r++) { rc[r] = (uint8_t)regs[r].combo; rcol[r] = (regs[r].group << 28) | regs[r].offset; }
        d_regcombo = (uint8_t*)dev->alloc(rc.size());
        dev->h2d(d_regcombo, rc.data(), rc.size());
        d_regcol = (uint32_t*)dev->alloc(rcol.size() * 4);
        dev->h2d(d_regcol, rcol.data(), rcol.size() * 4);
        dev->sync();
        active = true;
    }
    void destroy(Dev* dev) {
        if (!active) return;
        dev->free(d_prog); for (auto& p : d_colmask) dev->free(p);
        for (Chunk& c : chunks) { dev->free(c.d_prog); c.d_prog = nullptr; }
        dev->free(d_regcombo); dev->free(d_regcol);
        active = false;
    }

    // SSA step list -> slot-allocated bytecode.
    void compile(const IrStep* st, size_t n, uint32_t ret) {
        std::vector<uint32_t> mix_exp;
        compile_list(st, n, ret, (size_t)-1, 0, prog, n_fp_slots, n_mix_slots, ret_slot, &mix_exp, true);
        n_mixpow = 0;
        for (uint32_t e : mix_exp) if (e + 1 > n_mixpow) n_mixpow = e + 1;
        make_chunks(st, n, ret, mix_exp);
    }
    // `head_idx`: step index of the TRUE that heads the top-level chain of a chunk; its exponent is `base_exp` instead of 0.
    void compile_list(const IrStep* st, size_t n, uint32_t ret, size_t head_idx, uint32_t base_exp, std::vector<BcIns>& out, uint32_t& out_fp_slots,
                      uint32_t& out_mix_slots, uint32_t& out_ret_slot, std::vector<uint32_t>* mix_exp_out, bool validate) const {
        std::vector<int> is_fp(n);                 // 1: pushes an fp var, 0: pushes a mix var
        std::vector<uint32_t> fp_of, mix_of;       // var index -> step index
        for (size_t i = 0; i < n; i++) {
            if (st[i].op > IR_AND_COND) throw Err("circuit: bad poly op");
            is_fp[i] = st[i].op <= IR_MUL;
            (is_fp[i] ? fp_of : mix_of).push_back((uint32_t)i);
        }
        if (ret >= mix_of.size()) throw Err("circuit: ret is not a mix var");
        auto chk_fp = [&](uint32_t v, size_t at) { if (v >= fp_of.size() || fp_of[v] >= at) throw Err("circuit: fp operand used before definition"); };
        auto chk_mx = [&](uint32_t v, size_t at) { if (v >= mix_of.size() || mix_of[v] >= at) throw Err("circuit: mix operand used before definition"); };
        std::vector<size_t> fp_last(fp_of.size(), 0), mix_last(mix_of.size(), 0);
        std::vector<uint32_t> mix_exp(mix_of.size(), 0);
        size_t nm = 0;
        for (size_t i = 0; i < n; i++) {
            const IrStep& s = st[i];
            switch (s.op) {
                case IR_ADD: case IR_SUB: case IR_MUL: chk_fp(s.a, i); chk_fp(s.b, i); fp_last[s.a] = i; fp_last[s.b] = i; break;
                case IR_GET: if (validate && s.a >= taps.size()) throw Err("circuit: Get of an unknown tap"); break;
                case IR_GET_GLOBAL: if (validate && (s.a > 1 || s.b >= (s.a == 0 ? N_GLOBAL : n_mix))) throw Err("circuit: GetGlobal out of range"); break;
                case IR_TRUE: mix_exp[nm++] = i == head_idx ? base_exp : 0; break;
                case IR_AND_EQZ: chk_mx(s.a, i); chk_fp(s.b, i); mix_last[s.a] = i; fp_last[s.b] = i; mix_exp[nm] = mix_exp[s.a] + 1; nm++; break;
                case IR_AND_COND: chk_mx(s.a, i); chk_fp(s.b, i); chk_mx(s.c, i); mix_last[s.a] = i; mix_last[s.c] = i; fp_last[s.b] = i;
                                  mix_exp[nm] = mix_exp[s.a] + mix_exp[s.c]; nm++; break;
                default: break;
            }
        }
        mix_last[ret] = n;  // live to the end
        std::vector<uint32_t> fp_slot(fp_of.size()), mix_slot(mix_of.size());
        std::vector<uint32_t> fp_free, mix_free;
        uint32_t fp_hi = 0, mix_hi = 0, nf = 0; nm = 0;
        auto take = [](std::vector<uint32_t>& fr, uint32_t& hi) { if (!fr.empty()) { uint32_t s = fr.back(); fr.pop_back(); return s; } return hi++; };
        out.clear();
        for (size_t i = 0; i < n; i++) {
            const IrStep& s = st[i];
            BcIns ins{};
            std::vector<uint32_t> rel_fp, rel_mix;
            auto use_fp = [&](uint32_t v) { if (fp_last[v] == i) rel_fp.push_back(fp_slot[v]); return fp_slot[v]; };
            auto use_mx = [&](uint32_t v) { if (mix_last[v] == i) rel_mix.push_back(mix_slot[v]); return mix_slot[v]; };
            switch (s.op) {
                case IR_CONST: ins.op = BC_CONST; ins.a = to_mont(s.a % P); break;
                case IR_GET: ins.op = BC_GET; ins.a = taps[s.a].group; ins.b = taps[s.a].offset; ins.c = taps[s.a].back; break;
                case IR_GET_GLOBAL: ins.op = BC_GETG; ins.a = s.a; ins.b = s.b; break;
                case IR_ADD: ins.op = BC_ADD; ins.a = use_fp(s.a); ins.b = use_fp(s.b); break;
                case IR_SUB: ins.op = BC_SUB; ins.a = use_fp(s.a); ins.b = use_fp(s.b); break;
                case IR_MUL: ins.op = BC_MUL; ins.a = use_fp(s.a); ins.b = use_fp(s.b); break;
                case IR_TRUE: ins.op = BC_MTRUE; break;
                case IR_AND_EQZ: ins.op = BC_MEQZ; ins.a = use_mx(s.a); ins.b = use_fp(s.b); ins.c = mix_exp[s.a]; break;
                case IR_AND_COND: ins.op = BC_MCOND; ins.a = use_mx(s.a); ins.b = use_fp(s.b) | (use_mx(s.c) << 16); ins.c = mix_exp[s.a]; break;
            }
            // operands whose last use is here are released BEFORE the destination is allocated (dst may reuse them:
            // the interpreter reads all operands before it writes)
            std::sort(rel_fp.begin(), rel_fp.end()); rel_fp.erase(std::unique(rel_fp.begin(), rel_fp.end()), rel_fp.end());
            std::sort(rel_mix.begin(), rel_mix.end()); rel_mix.erase(std::unique(rel_mix.begin(), rel_mix.end()), rel_mix.end());
            for (uint32_t x : rel_fp) fp_free.push_back(x);
            for (uint32_t x : rel_mix) mix_free.push_back(x);
            if (is_fp[i]) {
                const uint32_t slot = take(fp_free, fp_hi);
                fp_slot[nf] = slot; ins.dst = (uint16_t)slot;
                if (fp_last[nf] == 0 || fp_last[nf] <= i) fp_free.push_back(slot);  // never used: slot is free again at once
                nf++;
            } else {
                const uint32_t slot = take(mix_free, mix_hi);
                mix_slot[nm] = slot; ins.dst = (uint16_t)slot;
                if (mix_last[nm] <= i && nm != ret) mix_free.push_back(slot);
                nm++;
            }
            if (fp_hi > 4096 || mix_hi > 4096) throw Err("circuit: too many live values");
            out.push_back(ins);
        }
        out_fp_slots = fp_hi ? fp_hi : 1; out_mix_slots = mix_hi ? mix_hi : 1; out_ret_slot = mix_slot[ret];
        if (mix_exp_out) *mix_exp_out = mix_exp;
    }
    // cut the top-level chain into chunks of about GEN_CHUNK_STEPS steps (HFB200_IR_CHUNK overrides) and compile each
    void make_chunks(const IrStep* st, size_t n, uint32_t ret, const std::vector<uint32_t>& mix_exp) {
        // ~400 steps (~2500 SASS instructions, 40 KB) per chunk: the kernel body then stays resident in the instruction cache while
        // every warp loops over its rows; at 3000 steps the stage is bound by instruction fetch from L2 (measured on B200 at
        // po2 = 18, 51 k steps: 104 ms per check stage with 3000-step chunks, 42 ms with 600, 38 ms with 300)
        size_t limit = 400;
        if (const char* env = std::getenv("HFB200_IR_CHUNK")) { const long v = std::atol(env); if (v >= 64) limit = (size_t)v; }
        chunks.clear();
        std::vector<uint32_t> fp_of, mix_of, var_of(n);
        for (size_t i = 0; i < n; i++) { auto& v = st[i].op <= IR_MUL ? fp_of : mix_of; var_of[i] = (uint32_t)v.size(); v.push_back((uint32_t)i); }
        std::vector<uint32_t> chain;  // mix vars of the top-level chain, head first
        for (uint32_t v = ret;;) { chain.push_back(v); const IrStep& s = st[mix_of[v]]; if (s.op == IR_TRUE) break; v = s.a; }
        std::reverse(chain.begin(), chain.end());
        if (n <= limit || chain.size() <= 2) {  // small circuit: the whole program is the one chunk
            Chunk c; c.prog = prog; c.n_fp_slots = n_fp_slots; c.n_mix_slots = n_mix_slots; c.ret_slot = ret_slot;
            chunks.push_back(std::move(c));
            return;
        }
        // Inside a chunk an element of the top-level chain carries a PARTIAL sum (it starts from the chunk's synthetic head), so
        // a step that reads it other than as its chain predecessor (an AndCond inner, the start of another chain) must not sit
        // in the same chunk: it would see the partial sum where the program means the full one.  Such a consumer starts a new
        // chunk instead, where `mark` recomputes the element it reads from the real head.  The first chunk starts at the real
        // head (exponent 0), so its partial sums are the full ones.
        std::vector<uint32_t> chain_pos(n, 0xFFFFFFFFu);
        for (size_t q = 0; q < chain.size(); q++) chain_pos[mix_of[chain[q]]] = (uint32_t)q;
        std::vector<uint32_t> stamp(n, 0);
        std::vector<uint32_t> stack;
        // marks the steps element `var` needs (its own step, its fp operands, its inner chain) -- not its chain predecessor.
        // `reads_from`: set when those steps read a chain element at position >= `lo` other than as a chain predecessor.
        bool reads_from = false;
        auto mark = [&](uint32_t var, uint32_t id, size_t lo) {
            size_t added = 0;
            stack.clear();
            const uint32_t self = mix_of[var];
            if (stamp[self] != id) { stamp[self] = id; added++; }
            const IrStep& e = st[self];
            stack.push_back(fp_of[e.b]);
            if (e.op == IR_AND_COND) stack.push_back(mix_of[e.c]);
            while (!stack.empty()) {
                const uint32_t i = stack.back(); stack.pop_back();
                if (chain_pos[i] != 0xFFFFFFFFu && chain_pos[i] >= lo) reads_from = true;
                if (stamp[i] == id) continue;
                stamp[i] = id; added++;
                const IrStep& s = st[i];
                switch (s.op) {
                    case IR_ADD: case IR_SUB: case IR_MUL: stack.push_back(fp_of[s.a]); stack.push_back(fp_of[s.b]); break;
                    case IR_AND_EQZ: stack.push_back(mix_of[s.a]); stack.push_back(fp_of[s.b]); break;
                    case IR_AND_COND: stack.push_back(mix_of[s.a]); stack.push_back(fp_of[s.b]); stack.push_back(mix_of[s.c]); break;
                    default: break;
                }
            }
            return added;
        };
        size_t k = 1;
        uint32_t id = 0;
        while (k < chain.size()) {
            id++;
            const size_t k0 = k;
            const size_t lo = k0 > 1 ? k0 : chain.size();  // chain elements a consumer in this chunk may not read
            size_t count = 0;
            while (k < chain.size()) {
                // tentative: does element k still fit?  (marking is idempotent within the id, so an overshoot only costs the re-mark below)
                reads_from = false;
                const size_t add = mark(chain[k], id, lo);
                if (k > k0 && (reads_from || count + add > limit)) { break; }
                count += add; k++;
            }
            if (k < chain.size()) {  // the element that did not fit was marked with this id: redo the group cleanly
                id++;
                for (size_t q = k0; q < k; q++) mark(chain[q], id, chain.size());
            }
            // sub-list: synthetic head TRUE, then the marked steps in their original order, operands renumbered
            std::vector<IrStep> sub;
            std::vector<uint32_t> fp_new(fp_of.size(), 0xFFFFFFFFu), mix_new(mix_of.size(), 0xFFFFFFFFu);
            uint32_t nfp = 0, nmx = 0;
            sub.push_back(IrStep{IR_TRUE, 0, 0, 0}); nmx = 1;
            std::vector<char> is_elem(n, 0);
            for (size_t q = k0; q < k; q++) is_elem[mix_of[chain[q]]] = 1;
            uint32_t prev_elem_new = 0;  // the synthetic head
            uint32_t sub_ret = 0;
            // Leaves (Get / Const / GetGlobal) are emitted where they are USED, not where the whole program first used them (that
            // would hoist every tap of a late chunk to its top and keep ~all taps live), and are re-issued when their last copy in
            // this chunk lies more than GEN_REMAT steps back: a Get is one coalesced load of LDE data that later chunks touch
            // anyway, a live value is a register for hundreds of instructions.
            const size_t GEN_REMAT = 192;
            std::vector<size_t> leaf_pos(fp_of.size(), 0);
            auto need_fp = [&](uint32_t v) {
                const IrStep& l = st[fp_of[v]];
                if (l.op > IR_GET_GLOBAL) return;  // computed value: already emitted (original order)
                if (fp_new[v] != 0xFFFFFFFFu && sub.size() - leaf_pos[v] <= GEN_REMAT) return;
                fp_new[v] = nfp++; leaf_pos[v] = sub.size();
                sub.push_back(l);
            };
            for (size_t i = 0; i < n; i++) {
                if (stamp[i] != id) continue;
                IrStep s = st[i];
                if (s.op <= IR_GET_GLOBAL) continue;
                switch (s.op) {
                    case IR_ADD: case IR_SUB: case IR_MUL: need_fp(s.a); need_fp(s.b); s.a = fp_new[s.a]; s.b = fp_new[s.b]; break;
                    case IR_AND_EQZ: need_fp(s.b); s.a = is_elem[i] ? prev_elem_new : mix_new[s.a]; s.b = fp_new[s.b]; break;
                    case IR_AND_COND: need_fp(s.b); s.a = is_elem[i] ? prev_elem_new : mix_new[s.a]; s.b = fp_new[s.b]; s.c = mix_new[s.c]; break;
                    default: break;
                }
                if (s.op <= IR_MUL) fp_new[var_of[i]] = nfp++;
                else { mix_new[var_of[i]] = nmx; if (is_elem[i]) { prev_elem_new = nmx; sub_ret = nmx; } nmx++; }
                sub.push_back(s);
            }
            Chunk c;
            compile_list(sub.data(), sub.size(), sub_ret, 0, mix_exp[chain[k0 - 1]], c.prog, c.n_fp_slots, c.n_mix_slots, c.ret_slot, nullptr, false);
            chunks.push_back(std::move(c));
        }
    }
};

struct GenEvalArgs {
    const uint32_t* ev[3];   // accum, code, data LDEs [w][domain]
    uint32_t* check;         // [4][domain]
    const BcIns* prog; uint32_t n_ins;
    const E4* mixpow;        // poly_mix^k, k < n_mixpow (device)
    const uint32_t* mix;     // accum mix (device)
    const uint32_t* globals; // device copy of the 32 globals
    uint32_t n_mix;
    uint32_t yinv[4];
    uint32_t po2, rows_per_block, n_fp_slots, n_mix_slots, ret_slot;
    uint32_t accumulate;     // 0: store tot / Z; 1: add it to what an earlier chunk left in `check`
};
// One thread per LDE row; fp slots [slot][row] and mix slots in shared memory; the program is read uniformly.
struct GenEvalCheckKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t* sm, GenEvalArgs p) {
        const uint32_t R = p.rows_per_block;
        E4* mslot = reinterpret_cast<E4*>(sm);                                   // [n_mix_slots][R]
        uint32_t* fslot = reinterpret_cast<uint32_t*>(mslot + (size_t)p.n_mix_slots * R);  // [n_fp_slots][R]
        uint32_t* gl = fslot + (size_t)p.n_fp_slots * R;                          // globals then mix
        for (uint32_t i = cx.tid; i < N_GLOBAL; i += cx.nt) gl[i] = p.globals[i];
        for (uint32_t i = cx.tid; i < p.n_mix; i += cx.nt) gl[N_GLOBAL + i] = p.mix[i];
        cx.sync();
        const uint64_t domain = 4ull << p.po2, dmask = domain - 1;
        for (uint32_t rr = cx.tid; rr < R; rr += cx.nt) {
            const uint64_t i = (uint64_t)cx.bx * R + rr;
            if (i >= domain) break;
            for (uint32_t pc = 0; pc < p.n_ins; pc++) {
                const BcIns ins = p.prog[pc];
                switch (ins.op) {
                    case BC_CONST: fslot[ins.dst * R + rr] = ins.a; break;
                    case BC_GET: fslot[ins.dst * R + rr] = p.ev[ins.a][(uint64_t)ins.b * domain + ((i + domain - 4ull * ins.c) & dmask)]; break;
                    case BC_GETG: fslot[ins.dst * R + rr] = gl[ins.a == 0 ? ins.b : N_GLOBAL + ins.b]; break;
                    case BC_ADD: fslot[ins.dst * R + rr] = fadd(fslot[ins.a * R + rr], fslot[ins.b * R + rr]); break;
                    case BC_SUB: fslot[ins.dst * R + rr] = fsub(fslot[ins.a * R + rr], fslot[ins.b * R + rr]); break;
                    case BC_MUL: fslot[ins.dst * R + rr] = fmul(fslot[ins.a * R + rr], fslot[ins.b * R + rr]); break;
                    case BC_MTRUE: mslot[ins.dst * R + rr] = e4_zero(); break;
                    case BC_MEQZ: mslot[ins.dst * R + rr] = e4_add(mslot[ins.a * R + rr], e4_scale(p.mixpow[ins.c], fslot[ins.b * R + rr])); break;
                    default: {  // BC_MCOND: tot = x.tot + cond * inner.tot * mix^k
                        const E4 inner = mslot[(ins.b >> 16) * R + rr];
                        const uint32_t cond = fslot[(ins.b & 0xFFFFu) * R + rr];
                        mslot[ins.dst * R + rr] = e4_add(mslot[ins.a * R + rr], e4_scale(e4_mul(inner, p.mixpow[ins.c]), cond));
                        break;
                    }
                }
            }
            const E4 tot = mslot[p.ret_slot * R + rr];
            const uint32_t yi = p.yinv[i & 3];
            for (int k = 0; k < 4; k++) {
                const uint32_t v = fmul(tot.c[k], yi);
                p.check[(uint64_t)k * domain + i] = p.accumulate ? fadd(p.check[(uint64_t)k * domain + i], v) : v;
            }
        }
    }
};

}  // namespace hf
