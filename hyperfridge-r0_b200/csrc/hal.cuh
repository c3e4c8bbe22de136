// Kernels of the device HAL (hfb200_hal_*): risc0-zkp `Hal` operators on caller device buffers.  The NTT and Merkle
// operators reuse ntt.cuh / poseidon2.cuh on caller pointers; the kernels here are the ones that exist in the segment prover
// only as fused or arena-bound stages.  Fp4 buffers are arrays of 4-word elements (upstream's `Buffer<ExtElem>`).
#pragma once
#include "ntt.cuh"
#include "circuit.cuh"

namespace hf {

static constexpr uint32_t HAL_T = 256;  // threads per block of every kernel below

HD E4 ld_e4(const uint32_t* p, uint64_t i) { return e4(p[4 * i], p[4 * i + 1], p[4 * i + 2], p[4 * i + 3]); }
HD void st_e4(uint32_t* p, uint64_t i, const E4& v) { p[4 * i] = v.c[0]; p[4 * i + 1] = v.c[1]; p[4 * i + 2] = v.c[2]; p[4 * i + 3] = v.c[3]; }

// Hal::zk_shift: the coefficient at bit-reversed position i of every column (true index j = bitrev(i)) times 3^j
struct HalZkShiftKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* io, uint64_t total, uint32_t lg, const uint32_t* p3_lo, const uint32_t* p3_hi) {
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (t >= total) return;
        const uint32_t i = (uint32_t)(t & ((1ull << lg) - 1));
        io[t] = fmul(io[t], tab_pow(p3_lo, p3_hi, brev(i, lg)));
    }
};

// Hal::batch_bit_reverse, in place: the thread of position i swaps it with bitrev(i) when i < bitrev(i)
struct HalBitRevKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* io, uint64_t total, uint32_t lg) {
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (t >= total) return;
        const uint32_t i = (uint32_t)(t & ((1ull << lg) - 1)), j = brev(i, lg);
        if (i >= j) return;
        const uint64_t a = t, b = t - i + j;
        const uint32_t x = io[a];
        io[a] = io[b];
        io[b] = x;
    }
};

// Hal::eltwise_add_elem: out[i] = x[i] + y[i]
struct HalAddElemKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* out, const uint32_t* x, const uint32_t* y, uint64_t count) {
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (t < count) out[t] = fadd(x[t], y[t]);
    }
};

// Hal::eltwise_sum_extelem: out[k * count + i] = (sum_{g < to_add} in[g * count + i]).c[k] (Fp4 in, four base columns out)
struct HalSumExtKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* out, const uint32_t* in, uint64_t count, uint32_t to_add) {
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (t >= count) return;
        E4 s = e4_zero();
        for (uint32_t g = 0; g < to_add; g++) s = e4_add(s, ld_e4(in, (uint64_t)g * count + t));
        for (int k = 0; k < 4; k++) out[(uint64_t)k * count + t] = s.c[k];
    }
};

// Hal::gather_sample: dst[i] = src[idx + i * stride], i < size
struct HalGatherKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* dst, const uint32_t* src, uint64_t idx, uint64_t size, uint64_t stride) {
        const uint64_t t = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (t < size) dst[t] = src[idx + t * stride];
    }
};

// Hal::scatter: for every cycle c < count, into[offsets[j]] = values[j] for j in [index[c], index[c + 1])
struct HalScatterKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, uint32_t* into, const uint32_t* index, const uint32_t* offsets, const uint32_t* values, uint64_t count) {
        const uint64_t c = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (c >= count) return;
        for (uint32_t j = index[c]; j < index[c + 1]; j++) into[offsets[j]] = values[j];
    }
};

// ---- batch_evaluate_any ---------------------------------------------------------------------------------------------
// out[j] = sum_k coeffs[which[j]][k] x_j^k.  grid.x = chunks of HAL_EV_RPB coefficients, grid.y = groups of HAL_EV_PTS
// consecutive points.  Points of one polynomial that are consecutive in `which` (upstream's tap order: the backs of a
// register follow each other) share one read of each coefficient.  Every (thread, point) keeps its own power of x_j and a
// lazy 64-bit accumulator (as DotKernel does): 4 wide multiply-adds and one Fp4 product per coefficient and point.  The block
// sums land in partial[j * nblk + chunk]; HalEvalReduceKernel adds them up.
static constexpr uint32_t HAL_EV_PTS = 4, HAL_EV_STEPS = 64, HAL_EV_RPB = HAL_T * HAL_EV_STEPS;
struct HalEvalKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t* sm, const uint32_t* coeffs, uint64_t n, const uint32_t* which, const uint32_t* xs, uint64_t count, E4* partial) {
        const uint64_t j0 = (uint64_t)cx.by * HAL_EV_PTS;
        const uint32_t npts = (uint32_t)(count - j0 < HAL_EV_PTS ? count - j0 : HAL_EV_PTS);
        const uint64_t base = (uint64_t)cx.bx * HAL_EV_RPB;
        E4* red = reinterpret_cast<E4*>(sm);  // [HAL_EV_PTS][HAL_T]
        E4 x[HAL_EV_PTS], xstep[HAL_EV_PTS];
        const uint32_t* poly[HAL_EV_PTS];
        bool same[HAL_EV_PTS];
        for (uint32_t g = 0; g < HAL_EV_PTS; g++) {
            const uint64_t j = j0 + (g < npts ? g : 0);
            x[g] = ld_e4(xs, j);
            xstep[g] = e4_pow(x[g], HAL_T);
            poly[g] = coeffs + (uint64_t)which[j] * n;
            same[g] = g > 0 && g < npts && which[j] == which[j - 1];
        }
        for (uint32_t t = cx.tid; t < HAL_T; t += cx.nt) {
            E4A acc[HAL_EV_PTS];
            E4 xp[HAL_EV_PTS];
            for (uint32_t g = 0; g < HAL_EV_PTS; g++) { acc[g] = e4a_zero(); xp[g] = e4_pow(x[g], base + t); }
            for (uint32_t s = 0; s < HAL_EV_STEPS; s++) {
                const uint64_t k = base + t + (uint64_t)s * HAL_T;
                if (k >= n) break;
                uint32_t c = 0;
#pragma unroll
                for (uint32_t g = 0; g < HAL_EV_PTS; g++) {
                    if (g >= npts) break;
                    if (!same[g]) c = poly[g][k];
                    e4a_mac(acc[g], xp[g], c);
                    xp[g] = e4_mul(xp[g], xstep[g]);
                }
            }
            for (uint32_t g = 0; g < HAL_EV_PTS; g++) red[g * HAL_T + t] = e4a_redc(acc[g]);
        }
        cx.sync();
        for (uint32_t h = HAL_T / 2; h >= 1; h >>= 1) {
            for (uint32_t t = cx.tid; t < HAL_EV_PTS * h; t += cx.nt) {
                const uint32_t g = t / h, i = t % h;
                red[g * HAL_T + i] = e4_add(red[g * HAL_T + i], red[g * HAL_T + i + h]);
            }
            cx.sync();
        }
        for (uint32_t g = cx.tid; g < npts; g += cx.nt) partial[(j0 + g) * cx.gx + cx.bx] = red[g * HAL_T];
    }
};
struct HalEvalReduceKernel {  // out[j] = sum_b partial[j * nblk + b]
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, const E4* partial, uint32_t nblk, uint64_t count, uint32_t* out) {
        const uint64_t j = (uint64_t)cx.bx * cx.nt + cx.tid;
        if (j >= count) return;
        E4 s = e4_zero();
        for (uint32_t b = 0; b < nblk; b++) s = e4_add(s, partial[j * nblk + b]);
        st_e4(out, j, s);
    }
};

// ---- mix_poly_coeffs --------------------------------------------------------------------------------------------------
// weights w[c] = mix_start * mix^c (one thread per column)
struct HalMixPowKernel {
    static constexpr bool kBarrier = false;
    HD static void run(const KCtx& cx, uint32_t*, E4* w, uint32_t n_cols, E4 mix_start, E4 mix) {
        const uint32_t c = cx.bx * cx.nt + cx.tid;
        if (c < n_cols) w[c] = e4_mul(mix_start, e4_pow(mix, c));
    }
};
// out[combo[c]][i] += w[c] * in[c][i] over every column c, one thread per row i.  The columns are walked in order with one lazy
// accumulator that is flushed into `out` whenever the combo changes, so any column -> combo map costs one pass over the columns.
// Weights and map are staged in shared memory: n_cols E4 + n_cols words.
struct HalMixPolyKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t* sm, uint32_t* out, const E4* w, const uint32_t* in, const uint32_t* combo, uint32_t n_cols, uint64_t n) {
        E4* ws = reinterpret_cast<E4*>(sm);
        uint32_t* cs = sm + 4 * (size_t)n_cols;
        for (uint32_t c = cx.tid; c < n_cols; c += cx.nt) { ws[c] = w[c]; cs[c] = combo[c]; }
        cx.sync();
        for (uint32_t t = cx.tid; t < HAL_T; t += cx.nt) {
            const uint64_t i = (uint64_t)cx.bx * HAL_T + t;
            if (i >= n) break;
            E4A acc = e4a_zero();
            for (uint32_t c = 0; c < n_cols; c++) {
                e4a_mac(acc, ws[c], in[(uint64_t)c * n + i]);
                if (c + 1 == n_cols || cs[c + 1] != cs[c]) {
                    const uint64_t o = (uint64_t)cs[c] * n + i;
                    st_e4(out, o, e4_add(ld_e4(out, o), e4a_redc(acc)));
                    acc = e4a_zero();
                }
            }
        }
    }
};

// ---- two-pass scans: prefix_products and poly_divide -----------------------------------------------------------------
// The shape of AccumScanKernel / AccumOffsetsKernel (HAL_SC_RPB elements per block: each thread folds HAL_SC_PER consecutive
// elements, the block scans the thread aggregates; block totals are scanned by one block, then every block applies its
// offset), over an element type and operator given by Op:
//   Op::T            element type;  Op::id() identity;  Op::op(a, b) = a then b (associative, not commutative)
//   Op::load(a, i)   element i of the scan;  Op::store(a, i, excl, incl) writes element i's result
static constexpr uint32_t HAL_SC_PER = 8, HAL_SC_RPB = HAL_T * HAL_SC_PER;
struct HalScanArgs {
    uint32_t* io;   // Fp4 elements, n of them
    uint64_t n;
    E4 z;           // poly_divide: the root of the divisor x - z
    uint32_t* rem;  // poly_divide: Fp4 remainder
};
struct ProdScan {  // Hal::prefix_products: io[i] <- io[0] * ... * io[i]
    using T = E4;
    HD static T id() { return e4_one(); }
    HD static T op(const T& a, const T& b) { return e4_mul(a, b); }
    HD static T load(const HalScanArgs& a, uint64_t i) { return ld_e4(a.io, i); }
    HD static void store(const HalScanArgs& a, uint64_t i, const T&, const T& incl) { st_e4(a.io, i, incl); }
};
// poly_divide(p, z): upstream's loop `for i in (0..n).rev() { next = z * cur + p[i]; p[i] = cur; cur = next }` is the
// first-order recurrence r_k = c_k + z r_{k+1}, r_n = 0; afterwards p[k] = r_{k+1} (the quotient) and r_0 is the remainder.
// Scan element i is the affine map r -> c_k + z r of k = n - 1 - i; maps compose as (m, a) then (m', a') = (m' m, a' + m' a).
struct Aff { E4 m, a; };
struct DivScan {
    using T = Aff;
    HD static T id() { T t; t.m = e4_one(); t.a = e4_zero(); return t; }
    HD static T op(const T& x, const T& y) { T t; t.m = e4_mul(y.m, x.m); t.a = e4_add(y.a, e4_mul(y.m, x.a)); return t; }
    HD static T load(const HalScanArgs& a, uint64_t i) { T t; t.m = a.z; t.a = ld_e4(a.io, a.n - 1 - i); return t; }
    HD static void store(const HalScanArgs& a, uint64_t i, const T& excl, const T& incl) {
        st_e4(a.io, a.n - 1 - i, excl.a);
        if (i == a.n - 1) st_e4(a.rem, 0, incl.a);
    }
};
// Inclusive Hillis-Steele scan of buf0[0..cnt) in shared memory (buf1: scratch); returns the buffer holding the result.
template <class Op>
HD typename Op::T* hal_block_scan(const KCtx& cx, typename Op::T* buf0, typename Op::T* buf1, uint32_t cnt) {
    typename Op::T *src = buf0, *dst = buf1;
    for (uint32_t d = 1; d < cnt; d <<= 1) {
        for (uint32_t i = cx.tid; i < cnt; i += cx.nt) dst[i] = i >= d ? Op::op(src[i - d], src[i]) : src[i];
        cx.sync();
        typename Op::T* t = src; src = dst; dst = t;
    }
    return src;
}
// mode 0: block totals to partial[blk]; mode 1: apply the exclusive offset partial[blk] and store every element
template <class Op>
struct HalScanKernel {
    static constexpr bool kBarrier = true;
    using T = typename Op::T;
    HD static void run(const KCtx& cx, uint32_t* sm, HalScanArgs a, T* partial, int mode) {
        T* buf0 = reinterpret_cast<T*>(sm);
        T* buf1 = buf0 + HAL_T;
        const uint64_t row0 = (uint64_t)cx.bx * HAL_SC_RPB;
        for (uint32_t t = cx.tid; t < HAL_T; t += cx.nt) {
            T acc = Op::id();
            for (uint32_t s = 0; s < HAL_SC_PER; s++) {
                const uint64_t i = row0 + (uint64_t)t * HAL_SC_PER + s;
                if (i < a.n) acc = Op::op(acc, Op::load(a, i));
            }
            buf0[t] = acc;
        }
        cx.sync();
        T* sc = hal_block_scan<Op>(cx, buf0, buf1, HAL_T);
        if (mode == 0) {
            if (cx.tid == 0) partial[cx.bx] = sc[HAL_T - 1];
            return;
        }
        for (uint32_t t = cx.tid; t < HAL_T; t += cx.nt) {
            T cur = t == 0 ? partial[cx.bx] : Op::op(partial[cx.bx], sc[t - 1]);
            for (uint32_t s = 0; s < HAL_SC_PER; s++) {
                const uint64_t i = row0 + (uint64_t)t * HAL_SC_PER + s;
                if (i >= a.n) break;
                const T next = Op::op(cur, Op::load(a, i));
                Op::store(a, i, cur, next);
                cur = next;
            }
        }
    }
};
// Exclusive scan of the nblk block totals in one block: each thread folds a run of consecutive totals, the block scans the runs.
template <class Op>
struct HalScanOffsetsKernel {
    static constexpr bool kBarrier = true;
    using T = typename Op::T;
    HD static void run(const KCtx& cx, uint32_t* sm, T* partial, uint32_t nblk) {
        T* buf0 = reinterpret_cast<T*>(sm);
        T* buf1 = buf0 + HAL_T;
        const uint32_t per = (nblk + HAL_T - 1) / HAL_T;
        for (uint32_t t = cx.tid; t < HAL_T; t += cx.nt) {
            T acc = Op::id();
            for (uint32_t s = 0; s < per; s++) { const uint32_t b = t * per + s; if (b < nblk) acc = Op::op(acc, partial[b]); }
            buf0[t] = acc;
        }
        cx.sync();
        T* sc = hal_block_scan<Op>(cx, buf0, buf1, HAL_T);
        for (uint32_t t = cx.tid; t < HAL_T; t += cx.nt) {
            T cur = t == 0 ? Op::id() : sc[t - 1];
            for (uint32_t s = 0; s < per; s++) {
                const uint32_t b = t * per + s;
                if (b >= nblk) break;
                const T v = partial[b];
                partial[b] = cur;
                cur = Op::op(cur, v);
            }
        }
    }
};

// Hal::fri_fold with the mix in device memory: FriFoldKernel's fold, the 16 mix powers computed once per block
struct HalFriFoldKernel {
    static constexpr bool kBarrier = true;
    HD static void run(const KCtx& cx, uint32_t* sm, uint32_t* out, const uint32_t* in, uint64_t n, const uint32_t* mix) {
        E4* mp = reinterpret_cast<E4*>(sm);
        if (cx.tid == 0) {
            const E4 m = ld_e4(mix, 0);
            E4 cur = e4_one();
            for (int i = 0; i < 16; i++) { mp[i] = cur; cur = e4_mul(cur, m); }
        }
        cx.sync();
        const uint64_t m = n / 16;
        for (uint32_t t = cx.tid; t < HAL_T; t += cx.nt) {
            const uint64_t idx = (uint64_t)cx.bx * HAL_T + t;
            if (idx >= m) break;
            E4 tot = e4_zero();
#pragma unroll
            for (uint32_t i = 0; i < 16; i++) {
                const uint64_t src = (uint64_t)brev(i, 4) * m + idx;
                tot = e4_add(tot, e4_mul(mp[i], e4(in[src], in[n + src], in[2 * n + src], in[3 * n + src])));
            }
            for (int k = 0; k < 4; k++) out[(uint64_t)k * m + idx] = tot.c[k];
        }
    }
};

}  // namespace hf
