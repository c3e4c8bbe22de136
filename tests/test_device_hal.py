"""The device HAL (hfb200_hal_*): risc0-zkp `Hal` operators on caller device buffers, queued on the context's stream.

CPU tier: the host emulator (device memory is host memory, buffers are numpy arrays), every operator against a first-principles
reference (the oracle's NTT / Merkle, Python Horner, scans and folds over Fp4), two compositions (the control root through the
HAL; the DEEP combos of a satisfied segment divide exactly), and the refusals.  GPU tier: torch CUDA tensors at production
sizes, against the host-buffer operators, the segment prover's roots and the emulator."""
import ctypes as C
import threading

import numpy as np
import pytest
from conftest import SMALL, DEFAULT, make_segment, rand_elems

P = 2013265921
R = (1 << 32) % P
RINV = pow(R, P - 2, P)


# ---- Fp / Fp4 in canonical form (Python ints); the library works in Montgomery form -----------------------------------------

def enc(x):
    return (np.asarray(x, dtype=np.uint64) % P * np.uint64(R) % np.uint64(P)).astype(np.uint32)


def dec(m):
    return (np.asarray(m, dtype=np.uint64) * np.uint64(RINV) % np.uint64(P)).astype(np.uint32)


def f4(m4):
    """Fp4 tuple (canonical ints) from 4 Montgomery words."""
    return tuple(int(v) for v in dec(np.asarray(m4).reshape(4)))


def m4(a):
    return enc(np.array(a, dtype=np.uint64))


def add4(a, b):
    return tuple((x + y) % P for x, y in zip(a, b))


def sub4(a, b):
    return tuple((x - y) % P for x, y in zip(a, b))


def mul4(a, b):
    c = [0] * 7
    for i in range(4):
        for j in range(4):
            c[i + j] += a[i] * b[j]
    return tuple((c[i] - 11 * (c[i + 4] if i < 3 else 0)) % P for i in range(4))


def pow4(a, e):
    r, b = (1, 0, 0, 0), a
    while e:
        if e & 1:
            r = mul4(r, b)
        b = mul4(b, b)
        e >>= 1
    return r


def inv4(a):
    return pow4(a, P ** 4 - 2)


def scal4(a, s):
    return tuple(x * s % P for x in a)


ZERO4, ONE4 = (0, 0, 0, 0), (1, 0, 0, 0)


def rand4(rng):
    return tuple(int(v) for v in rng.integers(0, P, 4))


def horner(coeffs_canon, x):
    acc = ZERO4
    for c in reversed(coeffs_canon):
        acc = add4(mul4(acc, x), (int(c), 0, 0, 0))
    return acc


# ---- fixtures ----------------------------------------------------------------------------------------------------------------

@pytest.fixture()
def emu(pkg, emu_lib):
    with pkg.Context(0, 12, SMALL, lib=emu_lib, deterministic=True) as c:
        yield c, pkg.Hal(c)


def U(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


# ---- CPU tier: every operator against its reference --------------------------------------------------------------------------

@pytest.mark.parametrize("count,n", [(1, 2), (3, 16), (2, 1 << 12), (1, 1 << 13)])
def test_interpolate_shift_bitrev_expand(emu, orc, count, n):
    _, hal = emu
    rng = np.random.default_rng(n + count)
    x = U(rand_elems(rng, (count, n)))
    io = x.copy()
    hal.batch_interpolate_ntt(io)
    want = orc.interpolate_ntt(x)
    assert (io == want).all()
    hal.zk_shift(io)
    want = orc.zk_shift(want)
    assert (io == want).all()
    for bits in (0, 2):
        out = np.zeros((count, n << bits), np.uint32)
        hal.batch_expand_into_evaluate_ntt(out, io, bits)
        assert (out == orc.expand_ntt(want, bits)).all()
    hal.batch_bit_reverse(io)
    assert (io == orc.bit_reverse(want)).all()


def test_zk_shift_and_bit_reverse_single_element(emu):
    _, hal = emu
    io = U([[5], [7]])
    hal.zk_shift(io)
    hal.batch_bit_reverse(io)
    assert io.tolist() == [[5], [7]]


@pytest.mark.parametrize("rows,cols", [(77, 20), (1, 1), (130, 16), (300, 33)])
def test_hash_rows_ragged(emu, orc, rows, cols):
    _, hal = emu
    m = U(rand_elems(np.random.default_rng(rows), (cols, rows)))
    dig = np.zeros((rows, 8), np.uint32)
    hal.hash_rows(dig, m)
    for r in (0, rows // 2, rows - 1):
        assert (dig[r] == orc.hash_elems(m[:, r])).all()


@pytest.mark.parametrize("rows,cols", [(2, 3), (64, 24), (1 << 11, 17)])
def test_hash_rows_and_folds_equal_merkle(emu, orc, rows, cols):
    ctx, hal = emu
    m = U(rand_elems(np.random.default_rng(cols), (cols, rows)))
    nodes = np.zeros((2 * rows, 8), np.uint32)
    hal.merkle_tree(nodes, m)
    root, want = orc.merkle(m, want_nodes=True)
    assert (nodes[1:] == want[1:]).all() and (nodes[1] == root).all()
    assert (nodes[1:] == ctx.op_merkle(m)[1:]).all()


@pytest.mark.parametrize("poly_count,n,count", [(1, 1, 1), (3, 100, 9), (2, (1 << 14) + 37, 5)])
def test_batch_evaluate_any(emu, poly_count, n, count):
    _, hal = emu
    rng = np.random.default_rng(n)
    coeffs = U(rand_elems(rng, (poly_count, n)))
    which = U(np.sort(rng.integers(0, poly_count, count)))  # tap order: points of one polynomial follow each other
    if count > 2:
        which[1] = which[0]
    xs_c = [rand4(rng) for _ in range(count)]
    xs = U(np.stack([m4(x) for x in xs_c]))
    out = np.zeros((count, 4), np.uint32)
    hal.batch_evaluate_any(coeffs, which, xs, out)
    canon = dec(coeffs)
    for j in range(count):
        assert f4(out[j]) == horner(canon[which[j]].tolist(), xs_c[j]), j


def test_batch_evaluate_any_unsorted_points(emu):
    _, hal = emu
    rng = np.random.default_rng(5)
    coeffs = U(rand_elems(rng, (4, 50)))
    which = U([3, 0, 3, 3, 1, 0, 2])
    xs_c = [rand4(rng) for _ in range(7)]
    out = np.zeros((7, 4), np.uint32)
    hal.batch_evaluate_any(coeffs, which, U(np.stack([m4(x) for x in xs_c])), out)
    canon = dec(coeffs)
    assert [f4(o) for o in out] == [horner(canon[w].tolist(), x) for w, x in zip(which, xs_c)]


def test_mix_poly_coeffs_arbitrary_map(emu):
    _, hal = emu
    rng = np.random.default_rng(9)
    n_cols, n, n_combos = 7, 50, 3
    inp = U(rand_elems(rng, (n_cols, n)))
    combo = U([2, 0, 0, 1, 2, 2, 0])
    out0 = U(rand_elems(rng, (n_combos, n, 4)))
    out = out0.copy()
    ms, mx = rand4(rng), rand4(rng)
    hal.mix_poly_coeffs(out, m4(ms), m4(mx), inp, combo)
    want = [[f4(out0[g, i]) for i in range(n)] for g in range(n_combos)]
    canon = dec(inp)
    for c in range(n_cols):
        w = mul4(ms, pow4(mx, c))
        for i in range(n):
            want[combo[c]][i] = add4(want[combo[c]][i], scal4(w, int(canon[c, i])))
    assert [[f4(out[g, i]) for i in range(n)] for g in range(n_combos)] == want


def poly_divide_ref(p, z):
    p = list(p)
    cur = ZERO4
    for i in reversed(range(len(p))):
        nxt = add4(mul4(z, cur), p[i])
        p[i] = cur
        cur = nxt
    return p, cur


@pytest.mark.parametrize("n", [1, 2, 5, 2048, 2049, 5000])
def test_poly_divide(emu, n):
    _, hal = emu
    rng = np.random.default_rng(n)
    poly = U(rand_elems(rng, (n, 4)))
    z = rand4(rng)
    rem = np.zeros(4, np.uint32)
    want, wrem = poly_divide_ref([f4(v) for v in poly], z)
    hal.poly_divide(poly, m4(z), rem)
    assert [f4(v) for v in poly] == want
    assert f4(rem) == wrem and wrem != ZERO4  # a nonzero remainder: p(z)


@pytest.mark.parametrize("n", [1, 2, 3, 2048, 4097])
def test_prefix_products(emu, n):
    _, hal = emu
    io = U(rand_elems(np.random.default_rng(n), (n, 4)))
    want, acc = [], ONE4
    for v in io:
        acc = mul4(acc, f4(v))
        want.append(acc)
    hal.prefix_products(io)
    assert [f4(v) for v in io] == want


def test_eltwise_gather_scatter(emu):
    _, hal = emu
    rng = np.random.default_rng(3)
    x, y = U(rand_elems(rng, 1000)), U(rand_elems(rng, 1000))
    out = np.zeros(1000, np.uint32)
    hal.eltwise_add_elem(out, x, y)
    assert (out.astype(np.uint64) == (x.astype(np.uint64) + y) % P).all()
    hal.eltwise_copy_elem(out, x)
    assert (out == x).all()
    hal.eltwise_zeroize_elem(out)
    assert (out == 0).all()
    ext = U(rand_elems(rng, (3, 10, 4)))
    s4 = np.zeros((4, 10), np.uint32)
    hal.eltwise_sum_extelem(s4, ext)
    assert (s4.T.astype(np.uint64) == ext.astype(np.uint64).sum(axis=0) % P).all()
    src = U(rand_elems(rng, 100))
    dst = np.zeros(9, np.uint32)
    hal.gather_sample(dst, src, 5, 11)
    assert (dst == src[5::11][:9]).all()
    into = np.zeros(20, np.uint32)
    index, offsets, values = U([0, 2, 2, 5]), U([3, 7, 0, 19, 11]), U([1, 2, 3, 4, 5])
    hal.scatter(into, index, offsets, values)
    want = np.zeros(20, np.uint32)
    want[offsets] = values
    assert (into == want).all()


def test_fri_fold_matches_host_operator(emu):
    ctx, hal = emu
    rng = np.random.default_rng(4)
    n = 16 * 300
    inp = U(rand_elems(rng, (4, n)))
    mix = U(rand_elems(rng, 4))
    out = np.zeros((4, n // 16), np.uint32)
    hal.fri_fold(out, inp, mix)
    assert (out == ctx.op_fri_fold(inp, mix)).all()


# ---- CPU tier: compositions --------------------------------------------------------------------------------------------------

def commit_through_hal(hal, cols, po2):
    """interpolate, zk_shift, expand x4, hash_rows, every fold: the root of a group's commitment."""
    w, n = cols.shape
    io = U(cols).copy()
    hal.batch_interpolate_ntt(io)
    hal.zk_shift(io)
    ev = np.zeros((w, 4 * n), np.uint32)
    hal.batch_expand_into_evaluate_ntt(ev, io, 2)
    nodes = np.zeros((8 * n, 8), np.uint32)
    hal.merkle_tree(nodes, ev)
    return nodes[1]


@pytest.mark.parametrize("po2", [12, 13, 14])
def test_control_root_through_hal(pkg, emu_lib, orc, po2):
    cir = orc.Circuit(*SMALL)
    code = cir.gen_code(po2)
    with pkg.Context(0, po2, SMALL, lib=emu_lib, deterministic=True) as ctx:
        root = commit_through_hal(pkg.Hal(ctx), code, po2)
        assert (root == ctx.control_root(po2, code)).all()
    assert (root == cir.control_id(po2)).all()


def _deep_remainders(pkg, ctx, orc, cir, po2, groups, corrupt):
    """DEEP combos of the segment's polynomials through the HAL, minus the interpolants of the GOOD trace's values at each
    combo's points, divided by (x - z w^-back) for every back: the remainders."""
    hal = pkg.Hal(ctx)
    n = 1 << po2
    taps = cir.taps()  # (group, offset, back), sorted; group ids 0 accum, 1 code, 2 data
    col_base = {0: 0, 1: groups[0].shape[0], 2: groups[0].shape[0] + groups[1].shape[0]}
    regs = {}
    for g, off, back in taps.tolist():
        regs.setdefault((g, off), []).append(back)
    combos = sorted(set(tuple(b) for b in regs.values()))
    n_cols = sum(x.shape[0] for x in groups)
    combo_of_col = np.zeros(n_cols, np.uint32)
    for (g, off), backs in regs.items():
        combo_of_col[col_base[g] + off] = combos.index(tuple(backs))
    rng = np.random.default_rng(po2)
    z, ms, mx = rand4(rng), rand4(rng), rand4(rng)
    w = pow(137, (P - 1) >> po2, P)  # a primitive N-th root of unity
    point = lambda b: scal4(z, pow(w, (P - 1 - b) % (P - 1), P))

    def coefficients(cols):
        c = U(np.concatenate(cols)).copy()
        hal.batch_interpolate_ntt(c)
        hal.zk_shift(c)
        hal.batch_bit_reverse(c)  # natural order
        return c

    good = coefficients(groups)
    # the tap values: batch_evaluate_any over the good polynomials
    which = U([col_base[g] + off for g, off, _ in taps.tolist()])
    xs_c = [point(b) for _, _, b in taps.tolist()]
    vals = np.zeros((len(which), 4), np.uint32)
    hal.batch_evaluate_any(good, which, U(np.stack([m4(x) for x in xs_c])), vals)
    v = {(int(which[i]), int(taps[i][2])): f4(vals[i]) for i in range(len(which))}
    coeffs = good
    if corrupt:
        bad = [x.copy() for x in groups]
        bad[2][0, 5] = (int(bad[2][0, 5]) + 1) % P
        coeffs = coefficients(bad)
    out = np.zeros((len(combos), n, 4), np.uint32)
    hal.mix_poly_coeffs(out, m4(ms), m4(mx), coeffs, combo_of_col)
    rems = []
    for k, backs in enumerate(combos):
        cols = [c for c in range(n_cols) if combo_of_col[c] == k and any(col_base[g] + off == c for g, off in regs)]
        pts = [point(b) for b in backs]
        ys = []
        for b in backs:
            y = ZERO4
            for c in cols:
                y = add4(y, mul4(mul4(ms, pow4(mx, c)), v[(c, b)]))
            ys.append(y)
        # Lagrange interpolant U(x) of degree < len(backs) through (pts, ys), coefficients low to high
        ucoef = [ZERO4] * len(pts)
        for i, (xi, yi) in enumerate(zip(pts, ys)):
            num, den = [ONE4], ONE4
            for j, xj in enumerate(pts):
                if j == i:
                    continue
                num = [add4(a, b) for a, b in zip([ZERO4] + num, [mul4(sub4(ZERO4, xj), t) for t in num] + [ZERO4])]
                den = mul4(den, sub4(xi, xj))
            s = mul4(yi, inv4(den))
            ucoef = [add4(u, mul4(s, t)) for u, t in zip(ucoef, num)]
        for d, u in enumerate(ucoef):
            out[k, d] = m4(sub4(f4(out[k, d]), u))
        poly = U(out[k]).copy()
        for x in pts:
            rem = np.zeros(4, np.uint32)
            hal.poly_divide(poly, m4(x), rem)
            rems.append(f4(rem))
    return rems


@pytest.mark.parametrize("corrupt", [False, True])
def test_deep_combos_divide_exactly(pkg, emu_lib, orc, corrupt):
    po2 = 12
    cir, g, code, data = make_segment(orc, SMALL, po2)
    with pkg.Context(0, po2, SMALL, lib=emu_lib, deterministic=True) as ctx:
        ctx.prove_segment(po2, g, code, data, 1)
        groups = [ctx.read_group(0), ctx.read_group(1), ctx.read_group(2)]
        assert (groups[2] == data).all()
        rems = _deep_remainders(pkg, ctx, orc, cir, po2, groups, corrupt)
    if corrupt:
        assert any(r != ZERO4 for r in rems)
    else:
        assert all(r == ZERO4 for r in rems), rems


# ---- CPU tier: refusals ------------------------------------------------------------------------------------------------------

def _err(lib, e):
    assert e, "expected a refusal"
    msg = C.cast(e, C.c_char_p).value.decode()
    lib.hfb200_free_error(e)
    return msg


def test_refusals(emu):
    ctx, hal = emu
    lib, h = ctx.lib, ctx._h
    buf = np.zeros(1 << 12, np.uint32)
    a = buf.ctypes.data
    assert "NULL ctx" in _err(lib, lib.hfb200_hal_zk_shift(None, a, 1, 16))
    assert "io is NULL" in _err(lib, lib.hfb200_hal_batch_interpolate_ntt(h, None, 1, 16))
    assert "digests is NULL" in _err(lib, lib.hfb200_hal_hash_rows(h, None, a, 4, 4))
    assert "remainder_out is NULL" in _err(lib, lib.hfb200_hal_poly_divide(h, a, 4, a, None))
    assert "z is NULL" in _err(lib, lib.hfb200_hal_poly_divide(h, a, 4, None, a))
    assert "mix is NULL" in _err(lib, lib.hfb200_hal_fri_fold(h, a, a, 32, None))
    assert "not a power of two" in _err(lib, lib.hfb200_hal_batch_interpolate_ntt(h, a, 1, 24))
    assert "not a power of two" in _err(lib, lib.hfb200_hal_zk_shift(h, a, 1, 3))
    assert "not a power of two" in _err(lib, lib.hfb200_hal_batch_bit_reverse(h, a, 1, 100))
    assert "not a power of two" in _err(lib, lib.hfb200_hal_batch_expand_into_evaluate_ntt(h, a, a + 4096, 1, 12, 2))
    assert "expand_bits = 1 is not supported" in _err(lib, lib.hfb200_hal_batch_expand_into_evaluate_ntt(h, a, a + 4096, 1, 16, 1))
    assert "expand_bits = 3 is not supported" in _err(lib, lib.hfb200_hal_batch_expand_into_evaluate_ntt(h, a, a + 4096, 1, 16, 3))
    assert "out and in overlap" in _err(lib, lib.hfb200_hal_batch_expand_into_evaluate_ntt(h, a, a + 16, 1, 16, 2))
    # sizes are checked before pointers: a bad size with a NULL pointer reports the size
    assert "not a power of two" in _err(lib, lib.hfb200_hal_batch_interpolate_ntt(h, None, 1, 24))
    assert "input_size must be 2 * output_size" in _err(lib, lib.hfb200_hal_hash_fold(h, a, 8, 3))
    assert "multiple of 16" in _err(lib, lib.hfb200_hal_fri_fold(h, a, a, 40, a))
    assert "16-byte aligned" in _err(lib, lib.hfb200_hal_hash_rows(h, a + 4, a, 4, 4))
    bad = np.array([P, 0, 0, 0], np.uint32)
    assert "non-canonical" in _err(lib, lib.hfb200_hal_poly_divide(h, a, 4, bad.ctypes.data, a))
    with pytest.raises(pkg_error(ctx), match="contiguous uint32 numpy"):
        hal.zk_shift(np.zeros((2, 8), np.int64))


def pkg_error(ctx):
    import hfb200_loader
    return hfb200_loader.load().Hfb200Error


def test_host_syncs_flat_in_emulator(emu):
    ctx, hal = emu
    cols = U(rand_elems(np.random.default_rng(1), (2, 256)))
    commit_through_hal(hal, cols, 8)  # grows nothing: no synchronisation
    s0 = hal.host_syncs()
    commit_through_hal(hal, cols, 8)
    assert hal.host_syncs() == s0
    hal.sync()
    assert hal.host_syncs() == s0 + 1


# ---- GPU tier ------------------------------------------------------------------------------------------------------------------

def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).cuda()


def _np(t):
    return t.cpu().numpy().view(np.uint32)


@pytest.mark.gpu
def test_gpu_ntt_and_leaves_at_production_size(pkg, gpu_lib):
    import torch
    po2, w = 20, 192
    n = 1 << po2
    rng = np.random.default_rng(20)
    cols = U(rand_elems(rng, (w, n)))
    with pkg.Context(0, 12, SMALL, lib=gpu_lib, deterministic=True) as ctx:
        hal = pkg.Hal(ctx)
        io = _t(cols)
        hal.batch_interpolate_ntt(io)
        hal.sync()
        coeffs = ctx.op_interpolate_ntt(cols)
        assert (_np(io) == coeffs).all()
        ev = torch.empty((w, 4 * n), dtype=torch.int32, device="cuda")
        hal.batch_expand_into_evaluate_ntt(ev, io, 2)
        ev0 = torch.empty((w, n), dtype=torch.int32, device="cuda")
        hal.batch_expand_into_evaluate_ntt(ev0, io, 0)
        hal.sync()
        assert (_np(ev0) == ctx.op_expand_ntt(coeffs, 0)).all()
        ev_h = _np(ev)
        assert (ev_h == ctx.op_expand_ntt(coeffs, 2)).all()
        del ev0, io
        dig = torch.empty((4 * n, 8), dtype=torch.int32, device="cuda")
        hal.hash_rows(dig, ev)
        hal.sync()
        assert (_np(dig) == ctx.op_merkle(ev_h)[4 * n:]).all()


@pytest.mark.gpu
def test_gpu_roots_equal_segment_checkpoints(pkg, gpu_lib):
    import torch
    po2 = 20
    n = 1 << po2
    with pkg.Context(0, po2, DEFAULT, lib=gpu_lib, deterministic=True) as seg:
        g = seg.witgen_synth(po2, 0x48595046, 1)
        seg.prove_resident(1)
        want = {"code_root": seg.checkpoint("code_root"), "data_root": seg.checkpoint("data_root")}
        groups = {"code_root": seg.read_group(1), "data_root": seg.read_group(2)}
        assert g.size == 32
    with pkg.Context(0, 12, SMALL, lib=gpu_lib, deterministic=True) as ctx:
        hal = pkg.Hal(ctx)
        for name, cols in groups.items():
            w = cols.shape[0]
            io = _t(cols)
            hal.batch_interpolate_ntt(io)
            hal.zk_shift(io)
            ev = torch.empty((w, 4 * n), dtype=torch.int32, device="cuda")
            hal.batch_expand_into_evaluate_ntt(ev, io, 2)
            nodes = torch.empty((8 * n, 8), dtype=torch.int32, device="cuda")
            hal.merkle_tree(nodes, ev)
            hal.sync()
            assert (_np(nodes[1]) == want[name]).all(), name


def _hal_buffers(src, n):
    import torch
    w = src.shape[0]
    return src.clone(), torch.empty((w, 4 * n), dtype=torch.int32, device=src.device), torch.empty((8 * n, 8), dtype=torch.int32, device=src.device)


def _commit_sequence(hal, bufs):
    io, ev, nodes = bufs
    hal.batch_interpolate_ntt(io)
    hal.zk_shift(io)
    hal.batch_expand_into_evaluate_ntt(ev, io, 2)
    hal.merkle_tree(nodes, ev)


@pytest.mark.gpu
def test_gpu_two_contexts_concurrent_and_no_hidden_syncs(pkg, gpu_lib):
    import torch
    po2, w = 18, 64
    n = 1 << po2
    src = _t(U(rand_elems(np.random.default_rng(18), (w, n))))
    bufs = {k: _hal_buffers(src, n) for k in "ab"}
    torch.cuda.synchronize()  # the copies above ran on torch's stream; the HAL streams read them
    with pkg.Context(0, 12, SMALL, lib=gpu_lib) as a, pkg.Context(0, 12, SMALL, lib=gpu_lib) as b:
        hals = {"a": pkg.Hal(a), "b": pkg.Hal(b)}
        assert hals["a"].stream != hals["b"].stream
        before = {k: h.host_syncs() for k, h in hals.items()}
        th = [threading.Thread(target=_commit_sequence, args=(hals[k], bufs[k])) for k in "ab"]
        for t in th:
            t.start()
        for t in th:
            t.join()
        assert {k: h.host_syncs() for k, h in hals.items()} == before
        for h in hals.values():
            h.sync()
        assert {k: h.host_syncs() for k, h in hals.items()} == {k: v + 1 for k, v in before.items()}
        ra, rb = _np(bufs["a"][2]), _np(bufs["b"][2])
        assert (ra[1:] == rb[1:]).all()
        assert (ra[1] == a.op_merkle(_np(_expand_ref(pkg, a, src, n)))[1]).all()


def _expand_ref(pkg, ctx, src, n):
    cols = _np(src)
    return _t(ctx.op_expand_ntt(ctx.op_interpolate_ntt(cols, zk_shift=True), 2))


@pytest.mark.gpu
def test_gpu_operators_match_emulator(pkg, gpu_lib, emu_lib):
    """The scan / evaluation / mix kernels at production sizes against the same sources run by the host emulator."""
    import torch
    n = 1 << 20
    rng = np.random.default_rng(7)
    with pkg.Context(0, 12, SMALL, lib=gpu_lib) as gctx, pkg.Context(0, 12, SMALL, lib=emu_lib) as ectx:
        gh, eh = pkg.Hal(gctx), pkg.Hal(ectx)
        poly = U(rand_elems(rng, (n, 4)))
        z = rand4(rng)
        gp, grem = _t(poly), torch.zeros(4, dtype=torch.int32, device="cuda")
        ep, erem = poly.copy(), np.zeros(4, np.uint32)
        gh.poly_divide(gp, m4(z), grem)
        eh.poly_divide(ep, m4(z), erem)
        pp_g, pp_e = _t(poly), poly.copy()
        gh.prefix_products(pp_g)
        eh.prefix_products(pp_e)
        coeffs = U(rand_elems(rng, (24, n)))
        which = U(np.repeat(np.arange(24), 3)[:64])
        xs = U(rand_elems(rng, (64, 4)))
        gout, eout = torch.zeros((64, 4), dtype=torch.int32, device="cuda"), np.zeros((64, 4), np.uint32)
        gh.batch_evaluate_any(_t(coeffs), _t(which), _t(xs), gout)
        eh.batch_evaluate_any(coeffs, which, xs, eout)
        combo = U(rng.integers(0, 3, 24))
        gm, em = torch.zeros((3, n, 4), dtype=torch.int32, device="cuda"), np.zeros((3, n, 4), np.uint32)
        ms, mx = rand4(rng), rand4(rng)
        gh.mix_poly_coeffs(gm, m4(ms), m4(mx), _t(coeffs), _t(combo))
        eh.mix_poly_coeffs(em, m4(ms), m4(mx), coeffs, combo)
        fin = U(rand_elems(rng, (4, n)))
        mix = U(rand_elems(rng, 4))
        gf = torch.zeros((4, n // 16), dtype=torch.int32, device="cuda")
        gh.fri_fold(gf, _t(fin), _t(mix))
        gh.sync()
        assert (_np(gp) == ep).all() and (_np(grem) == erem).all()
        assert (_np(pp_g) == pp_e).all()
        assert (_np(gout) == eout).all()
        assert (_np(gm) == em).all()
        assert (_np(gf) == gctx.op_fri_fold(fin, mix)).all()


@pytest.mark.gpu
def test_gpu_refuses_host_pointers(pkg, gpu_lib):
    with pkg.Context(0, 12, SMALL, lib=gpu_lib) as ctx:
        host = np.zeros(1 << 12, np.uint32)
        msg = _err(gpu_lib, gpu_lib.hfb200_hal_zk_shift(ctx._h, host.ctypes.data, 1, 1 << 12))
        assert "io is not device memory of device 0" in msg
        hal = pkg.Hal(ctx)
        with pytest.raises(pkg.Hfb200Error, match="torch CUDA tensor"):
            hal.zk_shift(host.reshape(1, -1))
