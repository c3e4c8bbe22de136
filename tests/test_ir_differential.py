"""Differential tests of data-defined circuits (`hfb200_init_ir`): seeded random tap tables and constraint programs, proved by the
product and by the CPU oracle interpreting the same data, seals compared word for word.

The programs cover what the fixed generators of oracle/synth_ir.py never produce: up to 4 distinct `back` values anywhere in
[0, 1023] (sometimes without 0), up to 8 tap sets, untapped columns, widths that are not multiples of 8, every op, operands far
back (so that the chunker re-issues leaves), non-canonical `Const` values, `GetGlobal` over both arrays, AndCond nested up to 3
deep, AndCond inners that are top-level chain elements or are used twice, chains that continue an existing mix value, dead steps
and a `ret` that is not the last step.  Each program runs at several chunk limits (`HFB200_IR_CHUNK`), so the compiler's cut of
the polynomial into chunks is checked against the oracle, which evaluates the whole program.

Satisfiable random circuits (constraints `code[0] * (D_k - e_k(taps))`, the output columns D_k filled by a numpy evaluator of
e_k) check the other direction: the product verifier, which also evaluates the whole program, accepts the chunked prover's seal.
"""
import itertools
import os
import random
import re
import time

import numpy as np
import pytest
from conftest import SMALL

P = 2013265921
CONST, GET, GETG, ADD, SUB, MUL, TRUE, EQZ, COND = range(9)
ACCUM, CODE, DATA = 0, 1, 2
ZK_CYCLES = 1994
N_GLOBAL = 32
CHUNKS = (None, "64", "97", "100000")      # None: the default limit
WIDTHS = [SMALL, (7, 20, 12), (5, 12, 4), (13, 28, 20)]
SEEDS = range(20)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class _Prog:
    """SSA step list: fp values and mix values are two index spaces; every step pushes one value."""

    def __init__(self):
        self.steps, self.nfp, self.nmx = [], 0, 0

    def fp(self, op, a=0, b=0, c=0):
        self.steps.append((op, a, b, c))
        self.nfp += 1
        return self.nfp - 1

    def mx(self, op, a=0, b=0, c=0):
        self.steps.append((op, a, b, c))
        self.nmx += 1
        return self.nmx - 1


def _tap_sets(rnd, full, zero=False):
    """Distinct back values (1-4 from [0, 1023]) and 1-8 distinct tap sets over them; `full`: the declared limits exactly (4
    backs, 8 sets, the first one holding all 4 backs); `zero`: back 0 is one of the backs."""
    pool = [0, 0, 1, 2, 3, 5, 9, 64, 193, 511, 1000, 1023, rnd.randrange(1024)]
    backs = {0} if zero else set()
    while len(backs) < (4 if full else rnd.randint(1, 4)):
        backs.add(rnd.choice(pool))
    backs = sorted(backs)
    subsets = [s for k in range(len(backs), 0, -1) for s in itertools.combinations(backs, k)]
    head, rest = subsets[:1], subsets[1:]
    rnd.shuffle(rest)
    subsets = head + rest if full else rest + head
    return subsets[:8 if full else rnd.randint(1, min(8, len(subsets)))]


def _tap_table(rnd, widths, sets, keep=()):
    """Sorted (group, offset, back) rows; each register gets one of `sets`, ~15% of the columns stay untapped (never one in `keep`)."""
    wc, wd, wa = widths
    taps = []
    for g, w in ((ACCUM, wa), (CODE, wc), (DATA, wd)):
        cols = [c for c in range(w) if (g, c) in keep or rnd.random() > 0.15] or [rnd.randrange(w)]
        for c in cols:
            taps += [(g, c, b) for b in rnd.choice(sets)]
    return taps


def random_ir(seed, widths=None, n_cons=60):
    """A seeded random constraint program in the PolyExtStep shape, not satisfiable: only compared with the oracle."""
    rnd = random.Random(seed)
    widths = widths or WIDTHS[seed % len(WIDTHS)]
    wc, wd, wa = widths
    taps = _tap_table(rnd, widths, _tap_sets(rnd, full=seed % 4 == 0))
    p = _Prog()

    def leaf():
        r = rnd.random()
        if r < 0.55:
            return p.fp(GET, rnd.randrange(len(taps)))
        if r < 0.75:
            return p.fp(CONST, rnd.choice([0, 1, P - 1, P, P + 1, 0xFFFFFFFF, rnd.randrange(1 << 32)]))
        if r < 0.88:
            return p.fp(GETG, 0, rnd.randrange(N_GLOBAL))
        return p.fp(GETG, 1, rnd.randrange(wa))

    def operand():
        r = rnd.random()
        if r < 0.6 or p.nfp < 2:
            return leaf()
        if r < 0.85:
            return rnd.randrange(p.nfp)
        return rnd.randrange(max(1, p.nfp // 4))      # far back: hundreds of steps in a 2000-step program

    def expr():
        v = operand()
        for _ in range(rnd.randint(1, 5)):
            u = operand()
            op = rnd.choice((ADD, SUB, MUL))
            v = p.fp(op, v, u) if rnd.random() < 0.5 else p.fp(op, u, v)
        return v

    def chain(depth, head=None):
        m = p.mx(TRUE) if head is None else head
        for _ in range(rnd.randint(1, 4)):
            if depth > 0 and rnd.random() < 0.4:
                m = p.mx(COND, m, expr(), chain(depth - 1))
            else:
                m = p.mx(EQZ, m, expr())
        return m

    top, inners = [p.mx(TRUE)], []
    for _ in range(n_cons):
        r = rnd.random()
        if r < 0.1:
            inner = rnd.choice(top)                                   # a top-level chain element (its full sum)
        elif r < 0.16 and inners:
            inner = rnd.choice(inners)                                # an inner used a second time
        elif r < 0.22:
            inner = chain(rnd.randint(0, 2), head=rnd.randrange(p.nmx))  # a chain continuing an existing mix value
        elif r < 0.45:
            inner = chain(rnd.randint(0, 2))                          # AndCond nested 1-3 deep
        else:
            inner = None
        if rnd.random() < 0.05:
            expr()                                                    # dead fp steps
        if rnd.random() < 0.03:
            chain(1)                                                  # a dead mix chain
        if inner is None:
            top.append(p.mx(EQZ, top[-1], expr()))
        else:
            inners.append(inner)
            top.append(p.mx(COND, top[-1], expr(), inner))
    ret = top[-1]
    expr()
    chain(1)                                                          # ret is not the last step
    return {"taps": np.array(taps, np.uint32), "steps": np.array(p.steps, np.uint32), "ret": ret, "n_globals": N_GLOBAL,
            "n_mix": wa, "widths": tuple(widths), "info": None}


# ---- satisfiable random circuits ----------------------------------------------------------------------------------------------
def _canon(words):
    """Montgomery words -> canonical values as uint64 (room for one product below 2^64)."""
    import oracle
    return oracle.decode(words).astype(np.uint64)


def satisfiable_ir(seed, widths, po2, n_out, n_cons):
    """A random circuit together with a trace that satisfies it: constraints code[0] * (D_k - e_k(taps)), where e_k reads code
    columns, free data columns and globals[0..32) at any tapped back, and the output columns D_k (the last `n_out` data columns,
    which no e_k reads) hold e_k on the active rows.  A tap at back b reads row (r - b) mod n, so the first rows read the blinding
    rows at the end of the trace.  Returns (ir, globals, code, data) with code from the oracle's control columns."""
    import oracle
    rnd = random.Random(seed)
    wc, wd, wa = widths
    n = 1 << po2
    act = n - ZK_CYCLES
    free = wd - n_out
    sets = _tap_sets(rnd, full=True, zero=True)
    with_zero = [s for s in sets if 0 in s]
    taps = _tap_table(rnd, widths, sets, keep={(CODE, 0)} | {(DATA, c) for c in range(free, wd)})
    # code[0] and the outputs are read at back 0: give them a tap set with 0
    regs = {}
    for g, c, b in taps:
        regs.setdefault((g, c), []).append(b)
    for key in [(CODE, 0)] + [(DATA, c) for c in range(free, wd)]:
        if 0 not in regs[key]:
            regs[key] = list(rnd.choice(with_zero))
    taps = sorted((g, c, b) for (g, c), bs in regs.items() for b in bs)
    tap_index = {t: i for i, t in enumerate(taps)}
    readable = [t for t in taps if t[0] == CODE or (t[0] == DATA and t[1] < free)]

    cir = oracle.Circuit(*widths)
    code = cir.gen_code(po2)
    g = cir.gen_globals(seed)
    data = np.random.default_rng(seed).integers(0, P, size=(wd, n), dtype=np.uint32)   # random witness and blinding rows (Montgomery words)
    code_c, g_c = [None] * wc, _canon(g)

    def column(grp, c):
        if grp == CODE:
            if code_c[c] is None:
                code_c[c] = _canon(code[c])
            return code_c[c]
        return _canon(data[c])

    p = _Prog()

    def expr(max_deg):
        """Random e of degree <= max_deg over readable taps / constants / globals, built as steps and evaluated on all n rows.
        The constraint polynomial may have degree 5 at most (its quotient by the vanishing polynomial lives on the 4x domain)."""
        vals, deg = [], []

        def leaf():
            r = rnd.random()
            if r < 0.65 and max_deg > 0:
                t = rnd.choice(readable)
                vals.append(np.roll(column(t[0], t[1]), t[2]))
                deg.append(1)
                return p.fp(GET, tap_index[t])
            deg.append(0)
            if r < 0.85:
                v = rnd.choice([0, 1, P - 1, P, P + 3, 0xFFFFFFFF, rnd.randrange(1 << 32)])
                vals.append(np.full(n, v % P, np.uint64))
                return p.fp(CONST, v)
            i = rnd.randrange(N_GLOBAL)
            vals.append(np.full(n, g_c[i], np.uint64))
            return p.fp(GETG, 0, i)

        base = p.nfp
        v = leaf()
        for _ in range(rnd.randint(1, 4)):
            u = leaf() if rnd.random() < 0.7 else base + rnd.randrange(p.nfp - base)
            a, b = (v, u) if rnd.random() < 0.5 else (u, v)
            da, db = deg[a - base], deg[b - base]
            op = rnd.choice((ADD, SUB, MUL) if da + db <= max_deg else (ADD, SUB))
            x, y = vals[a - base], vals[b - base]
            vals.append((x + y) % P if op == ADD else (x + (P - y)) % P if op == SUB else (x * y) % P)
            deg.append(da + db if op == MUL else max(da, db))
            v = p.fp(op, a, b)
        return v, vals[v - base]

    outs = list(range(free, wd))
    rnd.shuffle(outs)
    out_iter = itertools.cycle(outs)
    solved = {}

    def diff():
        """D_k - e_k for the next output column k: the first time k comes up, D_k is solved for a new e_k; later constraints on
        D_k reuse that e_k's value (an operand from far back)."""
        k = next(out_iter)
        if k not in solved:
            e, ev = expr(2)
            data[k, :act] = oracle.encode(ev[:act])
            solved[k] = e
        return p.fp(SUB, p.fp(GET, tap_index[(DATA, k, 0)]), solved[k])

    active = p.fp(GET, tap_index[(CODE, 0, 0)])
    top, raw_inners = [p.mx(TRUE)], []

    # degrees: D_k - e_k <= 2, under code[0] (1) and at most two nested conds of degree <= 1: <= 5
    def raw_chain(depth):
        """Chain whose terms vanish on the active rows only: must sit under a cond that is 0 on the blinding rows."""
        m = p.mx(TRUE)
        for _ in range(rnd.randint(1, 3)):
            if depth > 0 and rnd.random() < 0.4:
                m = p.mx(COND, m, expr(1)[0], raw_chain(depth - 1))   # any cond inside: the outer code[0] gates it
            else:
                m = p.mx(EQZ, m, diff())
        return m

    for _ in range(n_cons):
        r = rnd.random()
        if r < 0.12:                     # a top-level chain element: 0 on every row, so any (constant: degree) cond keeps it so
            top.append(p.mx(COND, top[-1], expr(0)[0], rnd.choice(top)))
        elif r < 0.2 and raw_inners:      # an inner used a second time
            top.append(p.mx(COND, top[-1], active, rnd.choice(raw_inners)))
        elif r < 0.45:
            inner = raw_chain(rnd.randint(0, 2))                   # AndCond nested 1-3 deep
            raw_inners.append(inner)
            top.append(p.mx(COND, top[-1], active, inner))
        else:
            top.append(p.mx(EQZ, top[-1], p.fp(MUL, active, diff())))
    ret = top[-1]
    expr(2)                                # dead steps after ret
    ir = {"taps": np.array(taps, np.uint32), "steps": np.array(p.steps, np.uint32), "ret": ret, "n_globals": N_GLOBAL,
          "n_mix": wa, "widths": tuple(widths), "info": None}
    return ir, g, code, data


# ---- helpers ------------------------------------------------------------------------------------------------------------------
def _segment_inputs(orc, widths, po2, seed):
    cir = orc.Circuit(*widths)
    code = cir.gen_code(po2)
    g = cir.gen_globals(seed)
    data = cir.gen_data(po2, code, g, seed, 1)
    return g, code, data


def _oracle_prove(orc, ir, po2, g, code, data):
    cir = orc.Circuit(*ir["widths"])
    cir.set_ir(ir["taps"], ir["steps"], ir["ret"], ir.get("info"))
    seal, cps, _ = cir.prove(po2, g, code, data, 1)
    return cir, seal, cps["code_root"]


def _prove(pkg, lib, orc, ir, po2, g, code, data, max_po2=None, jit=None):
    """Two-phase proof with the oracle's step_accum (the caller's for a data-defined circuit)."""
    with pkg.Context(0, max_po2 or po2, ir["widths"], lib=lib, ir=ir) as c:
        if jit is not None:
            assert c.ir_jit_active()[0] == jit
        mix = c.segment_begin(po2, g, code, data, 1)
        return c.segment_finish(orc.Circuit(*ir["widths"]).step_accum(po2, data, mix, 1))


def _assert_same(seal, oseal, what):
    assert len(seal) == len(oseal), what
    bad = np.nonzero(seal != oseal)[0]
    assert bad.size == 0, "%s: %d of %d seal words differ, first at %d" % (what, bad.size, len(seal), bad[0])


def _set_chunk(monkeypatch, chunk):
    if chunk is None:
        monkeypatch.delenv("HFB200_IR_CHUNK", raising=False)
    else:
        monkeypatch.setenv("HFB200_IR_CHUNK", chunk)


def _golden_shared_chain_element():
    z = np.load(os.path.join(GOLDEN, "ir_shared_chain_element.npz"))
    return {"taps": z["taps"], "steps": z["steps"], "ret": int(z["ret"]), "n_globals": N_GLOBAL, "n_mix": 8, "widths": SMALL,
            "info": None}


# ---- the generators produce what they claim -----------------------------------------------------------------------------------
def test_random_programs_cover_the_shapes():
    """Over the seeds of the CPU tier the generator really produces every shape the module docstring names."""
    seen = set()
    for seed in SEEDS:
        ir = random_ir(seed)
        taps, steps, ret = ir["taps"], ir["steps"], ir["ret"]
        backs = sorted(set(taps[:, 2].tolist()))
        regs = {}
        for g, c, b in taps.tolist():
            regs.setdefault((g, c), []).append(b)
        sets = {tuple(v) for v in regs.values()}
        seen |= {("backs", len(backs)), ("sets", len(sets))}
        seen.add(("no back 0", 0 not in backs))
        seen.add(("back >= 512", backs[-1] >= 512))
        seen.add(("4 taps on a register", max(len(v) for v in regs.values()) == 4))
        wc, wd, wa = ir["widths"]
        seen.add(("untapped column", len(regs) < wc + wd + wa))
        seen.add(("width not a multiple of 8", any(w % 8 for w in ir["widths"])))
        ops = set(steps[:, 0].tolist())
        seen.add(("every op", ops == set(range(9))))
        fp_of = [i for i, s in enumerate(steps) if s[0] <= MUL]
        mix_of = [i for i, s in enumerate(steps) if s[0] > MUL]
        seen.add(("ret not last", mix_of[ret] != len(steps) - 1))
        far = any(s[0] in (ADD, SUB, MUL) and i - fp_of[min(s[1], s[2])] > 192 for i, s in enumerate(steps))
        seen.add(("operand > 192 steps back", far))
        consts = {int(s[1]) for s in steps if s[0] == CONST}
        seen.add(("Const 0, 1, P-1, P and >= P", {0, 1, P - 1, P, 0xFFFFFFFF} <= consts))
        seen.add(("GetGlobal both arrays", {int(s[1]) for s in steps if s[0] == GETG} == {0, 1}))
        top, v = [], ret
        while steps[mix_of[v]][0] != TRUE:
            top.append(v)
            v = int(steps[mix_of[v]][1])
        top.append(v)
        inner_uses = {}
        for s in steps:
            if s[0] == COND:
                inner_uses[int(s[3])] = inner_uses.get(int(s[3]), 0) + 1
        seen.add(("inner used twice", any(k > 1 for k in inner_uses.values())))
        seen.add(("inner is a top-level element", any(u in top for u in inner_uses)))

        def depth(v):   # AndCond nesting of an inner chain (not counting what it continues from the top-level chain)
            s = steps[mix_of[v]]
            if v in top or s[0] == TRUE:
                return 0
            d = depth(int(s[1]))
            return max(d, 1 + depth(int(s[3]))) if s[0] == COND else d
        seen.add(("AndCond 3 deep", max(1 + depth(int(steps[mix_of[t]][3])) for t in top if steps[mix_of[t]][0] == COND) >= 3))
        live = set()
        stack = [mix_of[ret]]
        while stack:
            i = stack.pop()
            if i in live:
                continue
            live.add(i)
            s = steps[i]
            if s[0] in (ADD, SUB, MUL):
                stack += [fp_of[s[1]], fp_of[s[2]]]
            elif s[0] == EQZ:
                stack += [mix_of[s[1]], fp_of[s[2]]]
            elif s[0] == COND:
                stack += [mix_of[s[1]], fp_of[s[2]], mix_of[s[3]]]
        seen.add(("dead steps", len(live) < len(steps)))
    for what in ["no back 0", "back >= 512", "4 taps on a register", "untapped column", "width not a multiple of 8", "every op",
                 "ret not last", "operand > 192 steps back", "Const 0, 1, P-1, P and >= P", "GetGlobal both arrays", "inner used twice",
                 "inner is a top-level element", "AndCond 3 deep", "dead steps"]:
        assert (what, True) in seen, what
    assert {("backs", k) for k in (1, 2, 3, 4)} <= seen and ("sets", 8) in seen and ("sets", 1) in seen


# ---- CPU tier: host emulator of the kernel sources (interpreter kernel) ---------------------------------------------------------
@pytest.mark.parametrize("seed", SEEDS)
def test_random_program_matches_oracle(pkg, emu_lib, orc, monkeypatch, seed):
    ir, po2 = random_ir(seed), 12
    g, code, data = _segment_inputs(orc, ir["widths"], po2, seed)
    _, oseal, _ = _oracle_prove(orc, ir, po2, g, code, data)
    for chunk in CHUNKS:
        _set_chunk(monkeypatch, chunk)
        _assert_same(_prove(pkg, emu_lib, orc, ir, po2, g, code, data), oseal, "chunk limit %s" % chunk)
    monkeypatch.setenv("HFB200_IR_CHUNK", "64")
    assert pkg.ir_source(ir, ir["widths"], lib=emu_lib).count("__global__") >= 4   # the program really was cut


@pytest.mark.parametrize("chunk", [None, "200", "400", "2000", "64", "100000"])
def test_and_cond_on_a_chain_element_of_the_same_chunk(pkg, emu_lib, orc, monkeypatch, chunk):
    """Regression: an AndCond whose inner is a top-level chain element of the same chunk read that element's partial sum (the
    chunk starts its chain at a synthetic head), so the default limit of 400 and a limit of 200 gave a seal the oracle and both
    verifiers reject.  A 2034-step program over widths (8, 16, 8) with such inners (tests/golden/ir_shared_chain_element.npz)."""
    ir, po2, seed = _golden_shared_chain_element(), 12, 15
    g, code, data = _segment_inputs(orc, SMALL, po2, seed)
    cir, oseal, root = _oracle_prove(orc, ir, po2, g, code, data)
    _set_chunk(monkeypatch, chunk)
    seal = _prove(pkg, emu_lib, orc, ir, po2, g, code, data)
    _assert_same(seal, oseal, "chunk limit %s" % chunk)
    # the oracle's constraint polynomial is not zero on this trace, so neither verifier may accept the seal
    with pytest.raises(RuntimeError, match="constraint polynomial"):
        cir.verify(seal, root)
    with pytest.raises(pkg.Hfb200Error, match="constraint polynomial"):
        pkg.verify_segment(seal, root, SMALL, ir=ir, lib=emu_lib)


SAT_CASES = [(0, (8, 24, 8), 6), (1, (7, 20, 12), 5), (2, (13, 36, 4), 9)]


@pytest.mark.parametrize("seed,widths,n_out", SAT_CASES)
def test_satisfiable_random_circuit_verifies(pkg, emu_lib, orc, monkeypatch, seed, widths, n_out):
    """The chunked prover agrees with the whole-program verifiers: a satisfiable random circuit gives the oracle's seal at every
    chunk limit, the product's and the oracle's verifiers accept it, and a one-word change of the seal is rejected by both."""
    po2 = 12
    ir, g, code, data = satisfiable_ir(seed, widths, po2, n_out, n_cons=70)
    cir, oseal, root = _oracle_prove(orc, ir, po2, g, code, data)
    assert cir.verify(oseal, root) == po2                        # the trace satisfies the circuit
    for chunk in CHUNKS:
        _set_chunk(monkeypatch, chunk)
        seal = _prove(pkg, emu_lib, orc, ir, po2, g, code, data)
        _assert_same(seal, oseal, "chunk limit %s" % chunk)
    assert pkg.verify_segment(seal, root, widths, ir=ir, lib=emu_lib) == po2
    rnd = random.Random(seed)
    for pos in [len(seal) // 2, len(seal) - 1] + [rnd.randrange(len(seal)) for _ in range(2)]:
        bad = seal.copy()
        bad[pos] ^= 1 << rnd.randrange(31)
        with pytest.raises(pkg.Hfb200Error):
            pkg.verify_segment(bad, root, widths, ir=ir, lib=emu_lib)
        with pytest.raises(RuntimeError):
            cir.verify(bad, root)


def test_unsatisfied_random_circuit_is_rejected(pkg, emu_lib, orc):
    """The same construction with one output word of an active row changed proves (the prover does not check the witness) but
    neither verifier accepts the seal."""
    widths, po2 = (8, 24, 8), 12
    ir, g, code, data = satisfiable_ir(0, widths, po2, 6, n_cons=70)
    data[widths[1] - 6:, 777] = (data[widths[1] - 6:, 777] + 1) % P        # every output column, one active row
    cir, oseal, root = _oracle_prove(orc, ir, po2, g, code, data)
    seal = _prove(pkg, emu_lib, orc, ir, po2, g, code, data)
    _assert_same(seal, oseal, "unsatisfied trace")
    with pytest.raises(pkg.Hfb200Error, match="constraint polynomial"):
        pkg.verify_segment(seal, root, widths, ir=ir, lib=emu_lib)
    with pytest.raises(RuntimeError, match="constraint polynomial"):
        cir.verify(seal, root)


# ---- refusals -----------------------------------------------------------------------------------------------------------------
_OK_TAPS = [(CODE, 0, 0), (DATA, 0, 0), (DATA, 0, 1)]
_OK_STEPS = [(GET, 0, 0, 0), (TRUE, 0, 0, 0), (EQZ, 0, 0, 0)]


def _nine_sets():
    subsets = [s for k in (1, 2, 3) for s in itertools.combinations((0, 1, 2, 3), k)][:9]
    return [(DATA, c, b) for c, s in enumerate(subsets) for b in s]


REFUSALS = {
    "five_backs": ([(DATA, 0, b) for b in (0, 1, 2, 3)] + [(DATA, 1, 4)], _OK_STEPS, 1, "circuit: more than 4 distinct back values"),
    "nine_tap_sets": (_nine_sets(), _OK_STEPS, 1, "circuit: more than 8 distinct tap sets"),
    "five_taps_on_a_register": ([(DATA, 0, b) for b in (0, 1, 2, 3, 4)], _OK_STEPS, 1, "circuit: more than 4 taps on one register"),
    "back_1024": ([(DATA, 0, 0), (DATA, 0, 1024)], _OK_STEPS, 1, "circuit: back too large"),
    "unsorted_registers": ([(DATA, 1, 0), (DATA, 0, 0)], _OK_STEPS, 1, "circuit: taps must be sorted by (group, offset, back)"),
    "unsorted_backs": ([(DATA, 0, 1), (DATA, 0, 0)], _OK_STEPS, 1, "circuit: taps must be sorted by (group, offset, back)"),
    "fp_use_before_definition": (_OK_TAPS, [(GET, 0, 0, 0), (ADD, 0, 1, 0), (TRUE, 0, 0, 0), (EQZ, 0, 1, 0)], 1,
                                 "circuit: fp operand used before definition"),
    "mix_use_before_definition": (_OK_TAPS, [(GET, 0, 0, 0), (TRUE, 0, 0, 0), (COND, 0, 0, 1)], 1,
                                  "circuit: mix operand used before definition"),
    "global_out_of_range": (_OK_TAPS, [(GETG, 0, N_GLOBAL, 0), (TRUE, 0, 0, 0), (EQZ, 0, 0, 0)], 1, "circuit: GetGlobal out of range"),
    "mix_out_of_range": (_OK_TAPS, [(GETG, 1, 8, 0), (TRUE, 0, 0, 0), (EQZ, 0, 0, 0)], 1, "circuit: GetGlobal out of range"),
    "global_array_2": (_OK_TAPS, [(GETG, 2, 0, 0), (TRUE, 0, 0, 0), (EQZ, 0, 0, 0)], 1, "circuit: GetGlobal out of range"),
    "ret_not_a_mix_value": (_OK_TAPS, _OK_STEPS, 2, "circuit: ret is not a mix var"),
}


@pytest.mark.parametrize("case", sorted(REFUSALS))
def test_refused_programs_name_the_reason(pkg, emu_lib, case):
    """Programs outside the declared limits are refused at registration and by the verifier with the exact reason, and no
    context (so no seal) comes into being."""
    taps, steps, ret, msg = REFUSALS[case]
    ir = {"taps": np.array(taps, np.uint32), "steps": np.array(steps, np.uint32), "ret": ret, "n_mix": 8, "info": None}
    with pytest.raises(pkg.Hfb200Error, match="^" + re.escape(msg) + "$"):
        pkg.Context(0, 12, SMALL, lib=emu_lib, ir=ir)
    with pytest.raises(pkg.Hfb200Error, match="^" + re.escape(msg) + "$"):
        pkg.verify_segment(np.zeros(1000, np.uint32), np.zeros(8, np.uint32), SMALL, ir=ir, lib=emu_lib)


def test_limits_themselves_are_accepted(pkg, emu_lib, orc):
    """4 distinct backs including 1023, 8 tap sets and 4 taps on one register are inside the limits: a satisfiable circuit at
    exactly those limits proves to the oracle's seal and verifies."""
    widths, po2 = (8, 24, 8), 12
    ir, g, code, data = satisfiable_ir(4, widths, po2, 6, n_cons=30)
    taps = ir["taps"]
    regs = {}
    for gr, c, b in taps.tolist():
        regs.setdefault((gr, c), []).append(b)
    assert len(set(taps[:, 2].tolist())) == 4 and len({tuple(v) for v in regs.values()}) == 8
    assert max(len(v) for v in regs.values()) == 4
    cir, oseal, root = _oracle_prove(orc, ir, po2, g, code, data)
    seal = _prove(pkg, emu_lib, orc, ir, po2, g, code, data)
    _assert_same(seal, oseal, "limits")
    assert pkg.verify_segment(seal, root, widths, ir=ir, lib=emu_lib) == po2 == cir.verify(seal, root)


# ---- GPU tier: NVRTC chunk kernels and the interpreter kernel -------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_random_program_matches_oracle_on_gpu(pkg, gpu_lib, orc, monkeypatch, seed):
    ir, po2 = random_ir(seed), 12
    g, code, data = _segment_inputs(orc, ir["widths"], po2, seed)
    _, oseal, _ = _oracle_prove(orc, ir, po2, g, code, data)
    for chunk in (None, "64"):
        _set_chunk(monkeypatch, chunk)
        for jit in ("1", "0"):
            monkeypatch.setenv("HFB200_IR_JIT", jit)
            seal = _prove(pkg, gpu_lib, orc, ir, po2, g, code, data, jit=jit == "1")
            _assert_same(seal, oseal, "chunk limit %s, HFB200_IR_JIT=%s" % (chunk, jit))


@pytest.mark.gpu
def test_random_programs_at_two_sizes_on_gpu(pkg, gpu_lib, orc, monkeypatch):
    """One context proves po2 14 and then 13: each size has its own NVRTC build, both give the oracle's seals, as does the
    interpreter."""
    for jit in ("1", "0"):
        monkeypatch.setenv("HFB200_IR_JIT", jit)
        for seed in (15, 16):
            ir = random_ir(seed)
            with pkg.Context(0, 14, ir["widths"], lib=gpu_lib, ir=ir) as c:
                assert c.ir_jit_active()[0] == (jit == "1")
                for po2 in (14, 13):
                    g, code, data = _segment_inputs(orc, ir["widths"], po2, seed + po2)
                    _, oseal, _ = _oracle_prove(orc, ir, po2, g, code, data)
                    mix = c.segment_begin(po2, g, code, data, 1)
                    seal = c.segment_finish(orc.Circuit(*ir["widths"]).step_accum(po2, data, mix, 1))
                    _assert_same(seal, oseal, "seed %d po2 %d HFB200_IR_JIT=%s" % (seed, po2, jit))


@pytest.mark.gpu
@pytest.mark.parametrize("seed,widths,n_out", SAT_CASES)
def test_satisfiable_random_circuit_verifies_on_gpu(pkg, gpu_lib, orc, monkeypatch, seed, widths, n_out):
    po2 = 13
    ir, g, code, data = satisfiable_ir(seed, widths, po2, n_out, n_cons=70)
    cir, oseal, root = _oracle_prove(orc, ir, po2, g, code, data)
    for jit in ("1", "0"):
        monkeypatch.setenv("HFB200_IR_JIT", jit)
        seal = _prove(pkg, gpu_lib, orc, ir, po2, g, code, data, jit=jit == "1")
        _assert_same(seal, oseal, "HFB200_IR_JIT=%s" % jit)
    assert pkg.verify_segment(seal, root, widths, ir=ir, lib=gpu_lib) == po2 == cir.verify(seal, root)
    bad = seal.copy()
    bad[len(bad) // 3] ^= 1
    with pytest.raises(pkg.Hfb200Error):
        pkg.verify_segment(bad, root, widths, ir=ir, lib=gpu_lib)
    with pytest.raises(RuntimeError):
        cir.verify(bad, root)


# ---- scale (GPU): the rv32im-v2-sized circuit at the segment sizes it is quoted at ----------------------------------------------
@pytest.mark.gpu
def test_rv32im_scale_program_at_po2_18_matches_oracle_on_gpu(pkg, gpu_lib, orc, monkeypatch):
    """The 51 k-step, W = 400 program of build_scaled(560) at po2 18: NVRTC chunk kernels and interpreter both give the oracle's seal."""
    from oracle import synth_ir
    ir = synth_ir.build_scaled(n_groups=560)
    W, po2 = ir["widths"], 18
    cir = orc.Circuit(*W)
    code = cir.gen_code(po2)
    g = cir.gen_globals(9)
    data = np.random.default_rng(18).integers(0, P, size=(W[1], 1 << po2), dtype=np.uint32)
    t = time.time()
    _, oseal, _ = _oracle_prove(orc, ir, po2, g, code, data)
    print("rv32im-scale IR at po2 18: oracle proof %.1f s on %d host threads" % (time.time() - t, os.cpu_count()))
    for jit in ("1", "0"):
        monkeypatch.setenv("HFB200_IR_JIT", jit)
        _assert_same(_prove(pkg, gpu_lib, orc, ir, po2, g, code, data, jit=jit == "1"), oseal, "HFB200_IR_JIT=%s" % jit)


@pytest.mark.gpu
def test_rv32im_scale_program_at_po2_20_jit_equals_interpreter(pkg, gpu_lib, orc, monkeypatch):
    from oracle import synth_ir
    ir = synth_ir.build_scaled(n_groups=560)
    W, po2 = ir["widths"], 20
    cir = orc.Circuit(*W)
    code = cir.gen_code(po2)
    g = cir.gen_globals(9)
    data = np.random.default_rng(20).integers(0, P, size=(W[1], 1 << po2), dtype=np.uint32)
    seals = {}
    for jit in ("1", "0"):
        monkeypatch.setenv("HFB200_IR_JIT", jit)
        seals[jit] = _prove(pkg, gpu_lib, orc, ir, po2, g, code, data, jit=jit == "1")
    _assert_same(seals["1"], seals["0"], "JIT against interpreter")


@pytest.mark.gpu
@pytest.mark.parametrize("po2", [21, 22])
def test_satisfiable_w400_circuit_at_large_segments_on_gpu(pkg, gpu_lib, orc, monkeypatch, po2):
    """A satisfiable W = 400 (24 / 320 / 56) circuit at po2 21 and 22, where element indices of the data group's LDE pass 2^31
    (320 * 2^23) and 2^32 (320 * 2^24): both verifiers accept the seal and the NVRTC kernels equal the interpreter."""
    W = (24, 320, 56)
    t = time.time()
    ir, g, code, data = satisfiable_ir(21, W, po2, n_out=40, n_cons=60)
    print("W = 400 satisfiable circuit at po2 %d: %d steps, trace built in %.1f s" % (po2, len(ir["steps"]), time.time() - t))
    seals = {}
    for jit in ("1", "0"):
        monkeypatch.setenv("HFB200_IR_JIT", jit)
        t = time.time()
        seals[jit] = _prove(pkg, gpu_lib, orc, ir, po2, g, code, data, jit=jit == "1")
        print("  HFB200_IR_JIT=%s: context + proof %.1f s" % (jit, time.time() - t))
    _assert_same(seals["1"], seals["0"], "JIT against interpreter")
    root = orc.Circuit(*W).control_id(po2)
    assert pkg.verify_segment(seals["1"], root, W, ir=ir, lib=gpu_lib) == po2
    cir = orc.Circuit(*W)
    cir.set_ir(ir["taps"], ir["steps"], ir["ret"], ir.get("info"))
    assert cir.verify(seals["1"], root) == po2
