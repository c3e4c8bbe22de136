// Segment-seal verifier of the product: `Receipt::verify` for the seals this library emits.
//
// Mirrors risc0-zkp 3.0.4 `verify::{Verifier::verify, merkle::MerkleTreeVerifier, fri::fri_verify, read_iop::ReadIOP}`
// plus the circuit's `poly_ext` evaluated at the DEEP point (/root/reference/Cargo.lock:3195-3198, not vendored; call
// sites of the reference: /root/reference/host/src/main.rs:622-624 and /root/reference/verifier/src/main.rs:124-126;
// SURVEY.md Appendix A.8).  Like upstream's, it runs on the HOST: verification is O(queries * log N) hashes and a few
// thousand extension-field operations -- there is no data-parallel hot path to put on the GPU, and a verifier must not
// need one.  It shares the field / hash suite / transcript code with the prover's host side (field.cuh, poseidon2.cuh)
// and is independent of oracle/ (tests compare the two verifiers on good and tampered seals).
#pragma once
#include <functional>
#include "circuit.cuh"
#include "poseidon2.cuh"

namespace hf {

static constexpr uint32_t V_QUERIES = 50, V_INV_RATE = 4, V_FRI_FOLD = 16, V_FRI_MIN_DEGREE = 256, V_CHECK_SIZE = 16;

struct VErr : Err { using Err::Err; };
static inline void vfail(const std::string& why) { throw VErr("verify: " + why); }

static inline uint32_t v_rou_fwd(unsigned k) { uint32_t g = to_mont(137); for (unsigned i = k; i < 27; i++) g = fmul(g, g); return g; }
static inline uint32_t v_rou_rev(unsigned k) { return finv(v_rou_fwd(k)); }
static inline unsigned v_log2(uint64_t n) { unsigned k = 0; while ((1ull << k) < n) k++; if ((1ull << k) != n) vfail("size is not a power of two"); return k; }
static inline E4 e4_mul_fp(const E4& a, uint32_t s) { return e4_scale(a, s); }
static inline E4 v_poly_eval(const E4* c, size_t n, const E4& x) { E4 r = e4_zero(); for (size_t i = n; i-- > 0;) r = e4_add(e4_mul(r, x), c[i]); return r; }
static inline bool v_eq(const Digest8& a, const Digest8& b) { for (int i = 0; i < 8; i++) if (a.w[i] != b.w[i]) return false; return true; }

struct VReadIOP {  // verify::read_iop::ReadIOP
    const uint32_t* p; size_t len, pos = 0;
    HostRng rng;  // its suite is the seal's hash suite: every hash of the verifier follows it
    VReadIOP(const uint32_t* s, size_t n, int suite) : p(s), len(n), rng(suite) {}
    void need(size_t n) { if (pos + n > len) vfail("seal truncated"); }
    uint32_t read_u32() { need(1); return p[pos++]; }
    void read_elems(uint32_t* out, size_t n) { need(n); for (size_t i = 0; i < n; i++) { const uint32_t w = p[pos++]; if (w >= P) vfail("non-canonical field element"); out[i] = w; } }
    void read_ext(E4* out, size_t n) { read_elems(reinterpret_cast<uint32_t*>(out), 4 * n); }
    Digest8 read_digest() { need(8); Digest8 d; for (int i = 0; i < 8; i++) d.w[i] = p[pos++]; return d; }
    void commit(const Digest8& d) { rng.mix(d.w); }
    void done() { if (pos != len) vfail("trailing words in seal"); }
};

struct VMerkle {  // verify::merkle::MerkleTreeVerifier (top layer in the seal, paths end there)
    size_t rows, cols, top_size;
    std::vector<Digest8> top;
    VMerkle(VReadIOP& iop, size_t rows_, size_t cols_) : rows(rows_), cols(cols_) {
        const unsigned layers = v_log2(rows);
        unsigned top_layer = 0;
        for (unsigned i = 1; i < layers; i++) { if ((1ull << i) > V_QUERIES) break; top_layer = i; }
        top_size = (size_t)1 << top_layer;
        top.resize(2 * top_size);
        for (size_t i = 0; i < top_size; i++) top[top_size + i] = iop.read_digest();
        for (size_t i = top_size - 1; i >= 1; i--) top[i] = suite_hash_pair(iop.rng.suite, top[2 * i], top[2 * i + 1]);
        iop.commit(top[1]);
    }
    const Digest8& root() const { return top[1]; }
    std::vector<uint32_t> open(VReadIOP& iop, size_t idx) const {
        if (idx >= rows) vfail("merkle index out of range");
        std::vector<uint32_t> row(cols);
        iop.read_elems(row.data(), cols);
        const int s = iop.rng.suite;
        Digest8 cur = suite_hash_elems(s, row.data(), cols);
        size_t i = idx + rows;
        while (i >= 2 * top_size) {
            const Digest8 other = iop.read_digest();
            cur = (i & 1) ? suite_hash_pair(s, other, cur) : suite_hash_pair(s, cur, other);
            i >>= 1;
        }
        if (!v_eq(top[i], cur)) vfail("merkle path does not match the committed top layer");
        return row;
    }
};

// The circuit as the verifier sees it: tap structure (registers, tap sets) + the constraint polynomial at a point.
struct VCircuit {
    GenericCircuitHost g;   // taps / regs / combos (+ bytecode for data-defined circuits); host tables only
    bool builtin = false;
    CircuitHost ch;         // built-in circuit: picks / chain sources (host copies only)
    char info[17] = {0};    // CIRCUIT_INFO hashed into the transcript header

    void init_builtin(uint32_t wc, uint32_t wd, uint32_t wa) {
        builtin = true;
        set_circuit_info(info, false, nullptr);
        ch.init_host(wc, wd, wa);
        std::vector<IrTap> taps;
        for (uint32_t c = 0; c < wa; c++) { taps.push_back(IrTap{GROUP_ACCUM, c, 0}); taps.push_back(IrTap{GROUP_ACCUM, c, 1}); }
        for (uint32_t c = 0; c < wc; c++) taps.push_back(IrTap{GROUP_CODE, c, 0});
        for (uint32_t c = 0; c < wd; c++) { taps.push_back(IrTap{GROUP_DATA, c, 0}); if (c < ch.cd.n_prev) taps.push_back(IrTap{GROUP_DATA, c, 1}); }
        g.w[GROUP_ACCUM] = wa; g.w[GROUP_CODE] = wc; g.w[GROUP_DATA] = wd; g.n_mix = 4 * ch.cd.n_chains;
        g.analyze_taps(taps.data(), taps.size());
    }
    void init_ir(uint32_t wc, uint32_t wd, uint32_t wa, uint32_t n_mix, const IrTap* tp, size_t n_taps, const IrStep* st, size_t n_steps, uint32_t ret,
                 const uint8_t* info16 = nullptr) {
        builtin = false;
        set_circuit_info(info, true, info16);
        g.init(nullptr, wc, wd, wa, n_mix, tp, n_taps, st, n_steps, ret);
    }

    using Get = std::function<E4(uint32_t group, uint32_t offset, uint32_t back)>;

    // Fp4 product formula applied to components that are themselves ring elements (here: evaluations in Fp4)
    static void ext_mul(const E4* a, const E4* b, E4* r) {
        auto nb = [](const E4& x) { return e4_scale(x, NBETA); };
        const E4 t0 = e4_add(e4_add(e4_mul(a[1], b[3]), e4_mul(a[2], b[2])), e4_mul(a[3], b[1]));
        const E4 t1 = e4_add(e4_mul(a[2], b[3]), e4_mul(a[3], b[2]));
        const E4 t2 = e4_mul(a[3], b[3]);
        r[0] = e4_add(e4_mul(a[0], b[0]), nb(t0));
        r[1] = e4_add(e4_add(e4_mul(a[0], b[1]), e4_mul(a[1], b[0])), nb(t1));
        r[2] = e4_add(e4_add(e4_add(e4_mul(a[0], b[2]), e4_mul(a[1], b[1])), e4_mul(a[2], b[0])), nb(t2));
        r[3] = e4_add(e4_add(e4_mul(a[0], b[3]), e4_mul(a[1], b[2])), e4_add(e4_mul(a[2], b[1]), e4_mul(a[3], b[0])));
    }

    E4 poly(const E4& poly_mix, const uint32_t* globals, const uint32_t* mix, const Get& get) const {
        return builtin ? poly_builtin(poly_mix, globals, mix, get) : poly_ir(poly_mix, globals, mix, get);
    }

    // constraint list of "synth-rv32im-shape v1" (the same list EvalCheckKernel evaluates row by row), at one point
    E4 poly_builtin(const E4& poly_mix, const uint32_t* globals, const uint32_t* mix, const Get& get) const {
        const CircuitDev& cd = ch.cd;
        E4 tot = e4_zero(), mp = e4_one();
        auto push = [&](const E4& c) { tot = e4_add(tot, e4_mul(mp, c)); mp = e4_mul(mp, poly_mix); };
        const E4 active = get(GROUP_CODE, 0, 0), first = get(GROUP_CODE, 1, 0);
        for (uint32_t k = 0; k < cd.n_free; k++) {
            const uint16_t* pk = &ch.h_picks[6 * k];
            const E4 A = get(GROUP_DATA, pk[0], 0), B = get(GROUP_DATA, pk[1], 0), C = get(GROUP_DATA, pk[2], 0), D = get(GROUP_DATA, pk[3], 0);
            const E4 Pp = get(GROUP_DATA, pk[4], 1), X = get(GROUP_CODE, pk[5], 0);
            E4 e;
            switch (k & 3u) {
                case 0: e = e4_add(e4_mul(A, B), C); break;
                case 1: e = e4_add(e4_mul(e4_mul(A, B), C), Pp); break;
                case 2: e = e4_mul(e4_mul(e4_mul(e4_add(A, X), B), C), D); break;
                default: e = e4_add(e4_add(e4_mul(Pp, B), e4_mul(C, D)), X); break;
            }
            push(e4_mul(active, e4_sub(get(GROUP_DATA, cd.n_free + k, 0), e)));
        }
        const E4 nf = e4_sub(e4_one(), first);
        for (uint32_t r = 0; r < cd.n_chains; r++) {
            E4 acc[4], s[4], t[4], pr[4];
            for (uint32_t k = 0; k < 4; k++) {
                acc[k] = get(GROUP_ACCUM, 4 * r + k, 0);
                s[k] = e4_mul(nf, get(GROUP_ACCUM, 4 * r + k, 1));
                t[k] = e4_from(mix[4 * r + k]);
            }
            s[0] = e4_add(s[0], first);
            t[0] = e4_add(t[0], get(GROUP_DATA, ch.h_chain_src[r], 0));
            ext_mul(s, t, pr);
            for (uint32_t k = 0; k < 4; k++) push(e4_mul(active, e4_sub(acc[k], pr[k])));
        }
        push(e4_mul(first, e4_sub(get(GROUP_DATA, 0, 0), e4_from(globals[0]))));
        return tot;
    }

    // the register bytecode of a data-defined circuit, over Fp4 values
    E4 poly_ir(const E4& poly_mix, const uint32_t* globals, const uint32_t* mix, const Get& get) const {
        std::vector<E4> mp(g.n_mixpow ? g.n_mixpow : 1);
        E4 cur = e4_one();
        for (auto& m : mp) { m = cur; cur = e4_mul(cur, poly_mix); }
        std::vector<E4> f(g.n_fp_slots, e4_zero()), m(g.n_mix_slots, e4_zero());
        for (const BcIns& ins : g.prog) {
            switch (ins.op) {
                case BC_CONST: f[ins.dst] = e4_from(ins.a); break;
                case BC_GET: f[ins.dst] = get(ins.a, ins.b, ins.c); break;
                case BC_GETG: f[ins.dst] = e4_from(ins.a == 0 ? globals[ins.b] : mix[ins.b]); break;
                case BC_ADD: f[ins.dst] = e4_add(f[ins.a], f[ins.b]); break;
                case BC_SUB: f[ins.dst] = e4_sub(f[ins.a], f[ins.b]); break;
                case BC_MUL: f[ins.dst] = e4_mul(f[ins.a], f[ins.b]); break;
                case BC_MTRUE: m[ins.dst] = e4_zero(); break;
                case BC_MEQZ: m[ins.dst] = e4_add(m[ins.a], e4_mul(mp[ins.c], f[ins.b])); break;
                default: {
                    const E4 inner = m[ins.b >> 16], cond = f[ins.b & 0xFFFFu];
                    m[ins.dst] = e4_add(m[ins.a], e4_mul(e4_mul(inner, mp[ins.c]), cond));
                    break;
                }
            }
        }
        return m[g.ret_slot];
    }
};

struct VFriRound {  // verify::fri::VerifyRoundInfo
    size_t rows;
    VMerkle merkle;
    E4 mix;
    VFriRound(VReadIOP& iop, size_t in_domain) : rows(in_domain / V_FRI_FOLD), merkle(iop, in_domain / V_FRI_FOLD, V_FRI_FOLD * 4) { mix = iop.rng.random_ext(); }
    void query(VReadIOP& iop, size_t& pos, E4& goal) const {
        const size_t quot = pos / rows, group = pos % rows;
        const std::vector<uint32_t> d = merkle.open(iop, group);
        E4 ev[V_FRI_FOLD];
        for (size_t i = 0; i < V_FRI_FOLD; i++) ev[i] = e4(d[i], d[V_FRI_FOLD + i], d[2 * V_FRI_FOLD + i], d[3 * V_FRI_FOLD + i]);
        if (!e4_eq(ev[quot], goal)) vfail("FRI query value does not match the previous layer");
        // the 16 values are f(x0 w16^q): coefficients by the inverse DFT, then sum_i c_i (mix / x0)^i
        const uint32_t w16i = v_rou_rev(4), n_inv = finv(to_mont(V_FRI_FOLD));
        const uint32_t inv_x0 = fpow(v_rou_rev(v_log2(V_FRI_FOLD * rows)), group);
        E4 tot = e4_zero(), mul_mix = e4_one();
        uint32_t mul = ONE;
        for (size_t i = 0; i < V_FRI_FOLD; i++) {
            E4 c = e4_zero();
            const uint32_t wi = fpow(w16i, i);
            uint32_t wij = ONE;
            for (size_t q = 0; q < V_FRI_FOLD; q++) { c = e4_add(c, e4_scale(ev[q], wij)); wij = fmul(wij, wi); }
            c = e4_scale(c, n_inv);
            tot = e4_add(tot, e4_mul(e4_scale(c, mul), mul_mix));
            mul_mix = e4_mul(mul_mix, mix);
            mul = fmul(mul, inv_x0);
        }
        goal = tot;
        pos = group;
    }
};

static inline void v_fri_verify(VReadIOP& iop, size_t degree, const std::function<E4(VReadIOP&, size_t)>& inner) {
    const size_t orig_domain = V_INV_RATE * degree;
    size_t domain = orig_domain;
    std::vector<VFriRound> rounds;
    while (degree > V_FRI_MIN_DEGREE) { rounds.emplace_back(iop, domain); domain /= V_FRI_FOLD; degree /= V_FRI_FOLD; }
    std::vector<uint32_t> fc(4 * degree);
    iop.read_elems(fc.data(), fc.size());
    iop.commit(suite_hash_elems(iop.rng.suite, fc.data(), fc.size()));
    const uint32_t gen = v_rou_fwd(v_log2(domain));
    std::vector<E4> poly(degree);
    for (size_t i = 0; i < degree; i++) poly[i] = e4(fc[i], fc[degree + i], fc[2 * degree + i], fc[3 * degree + i]);
    const unsigned bits = v_log2(orig_domain);
    for (uint32_t q = 0; q < V_QUERIES; q++) {
        size_t pos = iop.rng.random_bits(bits) % orig_domain;
        E4 goal = inner(iop, pos);
        for (const VFriRound& r : rounds) r.query(iop, pos, goal);
        if (!e4_eq(v_poly_eval(poly.data(), degree, e4_from(fpow(gen, pos))), goal)) vfail("FRI final polynomial does not match the folded query");
    }
}

// verify::Verifier::verify for one segment seal.  code_root = the control id of (circuit, po2, suite).
static inline void verify_segment(const VCircuit& vc, const uint32_t* seal, size_t seal_words, const uint32_t* code_root, uint32_t* po2_out,
                                  int suite) {
    const GenericCircuitHost& g = vc.g;
    VReadIOP iop(seal, seal_words, suite);
    uint32_t globals[N_GLOBAL];
    iop.read_elems(globals, N_GLOBAL);
    const uint32_t po2 = iop.read_u32();
    if (po2 < 12 || po2 > 24) vfail("po2 out of range");  // the prover (and the oracle) start at 12
    if (po2_out) *po2_out = po2;
    transcript_header(iop.rng, vc.info, globals, N_GLOBAL, po2);
    const size_t N = (size_t)1 << po2, domain = N * V_INV_RATE;

    VMerkle code_v(iop, domain, g.w[GROUP_CODE]);
    Digest8 want; for (int i = 0; i < 8; i++) want.w[i] = code_root[i];
    if (!v_eq(code_v.root(), want)) vfail("code root is not the control id for this po2");
    VMerkle data_v(iop, domain, g.w[GROUP_DATA]);
    std::vector<uint32_t> mix(g.n_mix);
    for (auto& m : mix) m = iop.rng.random_elem();
    VMerkle accum_v(iop, domain, g.w[GROUP_ACCUM]);
    const E4 poly_mix = iop.rng.random_ext();
    VMerkle check_v(iop, domain, V_CHECK_SIZE);
    const E4 z = iop.rng.random_ext();
    const uint32_t back_one = v_rou_rev(po2);
    const size_t T = g.taps.size();
    std::vector<E4> coeff_u(T + V_CHECK_SIZE);
    iop.read_ext(coeff_u.data(), coeff_u.size());
    iop.commit(suite_hash_elems(suite, reinterpret_cast<const uint32_t*>(coeff_u.data()), 4 * coeff_u.size()));

    // tap evaluations at z w^-back from the per-register interpolants
    std::vector<E4> eval_u(T);
    std::vector<std::vector<int>> reg_of(3);
    for (int gi = 0; gi < 3; gi++) reg_of[gi].assign(g.w[gi], -1);
    for (size_t ri = 0; ri < g.regs.size(); ri++) {
        const GenReg& r = g.regs[ri];
        reg_of[r.group][r.offset] = (int)ri;
        for (uint32_t i = 0; i < r.size; i++) {
            const E4 x = e4_scale(z, fpow(back_one, g.taps[r.tap_begin + i].back));
            eval_u[r.tap_begin + i] = v_poly_eval(&coeff_u[r.tap_begin], r.size, x);
        }
    }
    auto get = [&](uint32_t gi, uint32_t off, uint32_t back) -> E4 {
        if (gi > 2 || off >= g.w[gi] || reg_of[gi][off] < 0) vfail("constraint polynomial reads a register that is not in the tap set");
        const GenReg& r = g.regs[reg_of[gi][off]];
        for (uint32_t k = 0; k < r.size; k++) if (g.taps[r.tap_begin + k].back == back) return eval_u[r.tap_begin + k];
        vfail("constraint polynomial reads a tap that is not in the tap set");
        return e4_zero();
    };
    const E4 result = vc.poly(poly_mix, globals, mix.data(), get);
    // check(z) from the 16 check polynomials at z^4: check_k(y) = sum_i y^i P_{k, rev2(i)}(y^4), combined over the basis x^k
    E4 check = e4_zero();
    for (uint32_t k = 0; k < 4; k++) {
        E4 ck = e4_zero();
        for (uint32_t i = 0; i < V_INV_RATE; i++) ck = e4_add(ck, e4_mul(coeff_u[T + 4 * k + brev(i, 2)], e4_pow(z, i)));
        E4 basis = e4_zero(); basis.c[k] = ONE;
        check = e4_add(check, e4_mul(ck, basis));
    }
    check = e4_mul(check, e4_sub(e4_pow(e4_scale(z, THREE), N), e4_one()));
    if (!e4_eq(check, result)) vfail("constraint polynomial does not match the check polynomial at z");

    const E4 dmix = iop.rng.random_ext();
    const size_t C = g.combos.size(), n_regs = g.regs.size();
    const uint32_t tot_backs = g.combo_begin[C];
    std::vector<E4> combo_u(tot_backs + 1, e4_zero()), reg_mix(n_regs + V_CHECK_SIZE);
    {
        E4 cur = e4_one();
        for (auto& m : reg_mix) { m = cur; cur = e4_mul(cur, dmix); }
        for (size_t ri = 0; ri < n_regs; ri++) {
            const GenReg& r = g.regs[ri];
            for (uint32_t i = 0; i < r.size; i++) combo_u[g.combo_begin[r.combo] + i] = e4_add(combo_u[g.combo_begin[r.combo] + i], e4_mul(reg_mix[ri], coeff_u[r.tap_begin + i]));
        }
        for (size_t c = 0; c < V_CHECK_SIZE; c++) combo_u[tot_backs] = e4_add(combo_u[tot_backs], e4_mul(reg_mix[n_regs + c], coeff_u[T + c]));
    }
    const E4 z4 = e4_pow(z, 4);
    const uint32_t gen = v_rou_fwd(po2 + 2);
    const VMerkle* gv[3] = {&accum_v, &code_v, &data_v};
    v_fri_verify(iop, N, [&](VReadIOP& r, size_t idx) -> E4 {
        const E4 x = e4_from(fpow(gen, idx));
        std::vector<uint32_t> rows[3];
        for (int gi = 0; gi < 3; gi++) rows[gi] = gv[gi]->open(r, idx);
        const std::vector<uint32_t> check_row = check_v.open(r, idx);
        std::vector<E4> tot(C + 1, e4_zero());
        for (size_t ri = 0; ri < n_regs; ri++) {
            const GenReg& rg = g.regs[ri];
            tot[rg.combo] = e4_add(tot[rg.combo], e4_scale(reg_mix[ri], rows[rg.group][rg.offset]));
        }
        for (size_t c = 0; c < V_CHECK_SIZE; c++) tot[C] = e4_add(tot[C], e4_scale(reg_mix[n_regs + c], check_row[c]));
        E4 ret = e4_zero();
        for (size_t c = 0; c < C; c++) {
            const E4 num = e4_sub(tot[c], v_poly_eval(&combo_u[g.combo_begin[c]], g.combos[c].size(), x));
            E4 div = e4_one();
            for (uint32_t back : g.combos[c]) div = e4_mul(div, e4_sub(x, e4_scale(z, fpow(back_one, back))));
            ret = e4_add(ret, e4_mul(num, e4_inv(div)));
        }
        ret = e4_add(ret, e4_mul(e4_sub(tot[C], combo_u[tot_backs]), e4_inv(e4_sub(x, z4))));
        return ret;
    });
    iop.done();
}

}  // namespace hf
