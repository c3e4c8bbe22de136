"""Poseidon2 partial rounds as two exact int8 GEMMs (csrc/poseidon2.cuh, "the 21 partial rounds as two linear maps").

CPU tier: the composed maps against step-by-step partial rounds in exact integers; the byte-plane GEMM arithmetic and its
accumulator bound on adversarial words (every byte 0xFF, p - 1, its Montgomery form, the largest delta) in a numpy model built
the same way as the C++ tables (the words entering the partial rounds cannot be chosen through the permutation's input); the
emulator's tensor-form permutation, i.e. the C++ tables, against the oracle.  GPU tier: the tcgen05 kernels against the oracle
on 2^20 states (partly idle last CTAs) and on Merkle trees with fewer leaves than a CTA or with levels large enough for
HashFoldKernel."""
import numpy as np
import pytest
from conftest import SMALL, rand_elems
from test_poseidon2 import _gen

P = 2013265921
R = (1 << 32) % P
P_INV = 0x88000001
K1, N1, K2, N2 = 96, 80, 192, 96


def _consts():
    g = _gen()
    rc = g.grain_constants(1, 0, 31, 24, 8, 21, 213, P)
    return [int(d) for d in g.M_INT_DIAG], rc[96:117]


DIAG, RC_PART = _consts()


def m_int(v):
    s = sum(v) % P
    return [(s + DIAG[i] * v[i]) % P for i in range(24)]


def m_int_powers():
    pw = [[[int(i == j) for j in range(24)] for i in range(24)]]
    for _ in range(21):
        prev = pw[-1]
        pw.append([[(sum(prev[l][i] for l in range(24)) + DIAG[o] * prev[o][i]) % P for i in range(24)] for o in range(24)])
    return pw


PW = m_int_powers()


def planes(coeffs, K):
    """Logical B operand [4 * outputs, K] of outputs o = sum_i coeffs[o][i] x_i: bytes j of 2^(8b) m 2^32 mod p at (4o + j, 4i + b)."""
    b = np.zeros((4 * len(coeffs), K), np.int64)
    for o, row in enumerate(coeffs):
        for i, m in enumerate(row):
            for bb in range(4):
                c = m * (1 << (8 * bb)) % P * R % P
                for j in range(4):
                    b[4 * o + j, 4 * i + bb] = (c >> (8 * j)) & 255
    return b


B1 = planes([PW[r][0] for r in range(1, 21)], K1)
B2 = planes([PW[21][o] + [PW[21 - j][o][0] for j in range(21)] for o in range(24)], K2)


def gemm(words, b):
    """words [n, K/4] u32 -> int32 planes [n, N]: the tensor-core product, bytes of the words against the byte planes."""
    a = np.ascontiguousarray(words.astype("<u4")).view(np.uint8).astype(np.int64)
    q = a @ b.T
    assert q.max() < 1 << 24  # plane accumulators: at most 180 * 255^2
    return q


def reduce(q):
    """REDC(sum_j 2^(8j) Q_j), canonical (the kernel's p2tc_reduce, in exact integers)."""
    q = q.reshape(q.shape[0], -1, 4).astype(object)
    v = q[..., 0] + (q[..., 1] << 8) + (q[..., 2] << 16) + (q[..., 3] << 24)
    assert (v < P << 32).all()
    m = (v & 0xFFFFFFFF) * P_INV & 0xFFFFFFFF
    return ((v - m * P) >> 32) % P


def test_composed_maps_equal_repeated_internal_layer():
    rng = np.random.default_rng(1)
    for trial in range(20):
        v = [int(x) for x in rng.integers(0, P, 24)]
        dl = [int(x) for x in rng.integers(0, P, 21)]
        if trial == 0:
            v, dl = [P - 1] * 24, [P - 1] * 21
        st = list(v)
        for r in range(21):
            tri = sum(PW[r - j][0][0] * dl[j] for j in range(r))
            assert st[0] == (sum(PW[r][0][i] * v[i] for i in range(24)) + tri) % P
            st[0] = (st[0] + dl[r]) % P
            st = m_int(st)
        exp = [(sum(PW[21][o][i] * v[i] for i in range(24)) + sum(PW[21 - j][o][0] * dl[j] for j in range(21))) % P for o in range(24)]
        assert st == exp


def test_byte_plane_gemms_exact_on_adversarial_words():
    rng = np.random.default_rng(2)
    n = 4096
    v = rng.integers(0, 1 << 32, (n, 24), dtype=np.uint64).astype(np.uint32)
    d = rng.integers(0, P, (n, 21), dtype=np.uint32)
    v[0], d[0] = 0xFFFFFFFF, P - 1          # every input byte 0xFF; the largest canonical delta
    v[1], d[1] = P - 1, (P - 1) // 2
    v[2], d[2] = (P - 1) * R % P, 0         # Montgomery form of p - 1
    v[3], d[3] = 0, 0
    got1 = reduce(gemm(v, B1))
    w = np.concatenate([v, d, np.zeros((n, 3), np.uint32)], axis=1)
    got2 = reduce(gemm(w, B2))
    vi, di = v.astype(object), d.astype(object)
    a = np.array([PW[r][0] for r in range(1, 21)], dtype=object)
    assert (got1 == (vi @ a.T) % P).all()
    full = np.array([PW[21][o] + [PW[21 - j][o][0] for j in range(21)] for o in range(24)], dtype=object)
    assert (got2 == (np.concatenate([vi, di], axis=1) @ full.T) % P).all()


def test_triangular_term_signed_groups_of_four():
    """sum_{j<r} c_{r-j} delta_j in groups of <= 4 balanced products, one signed REDC each (p2tc_dot4)."""
    half = (P - 1) // 2
    c = [0] + [(PW[k][0][0] * R % P) for k in range(1, 21)]
    c = [x - P if x > half else x for x in c]
    rng = np.random.default_rng(3)
    for trial in range(200):
        dl = [int(x) for x in rng.integers(0, P, 21)] if trial else [half + 1] * 21  # trial 0: the most negative balanced delta
        db = [x - P if x > half else x for x in dl]
        for r in range(1, 21):
            acc = 0
            for j0 in range(0, r, 4):
                vsum = sum(c[r - j] * db[j] for j in range(j0, min(r, j0 + 4)))
                assert abs(vsum) < (1 << 31) * P
                m = (vsum & 0xFFFFFFFF) * P_INV & 0xFFFFFFFF
                m = m - (1 << 32) if m >= 1 << 31 else m
                t = (vsum >> 32) - ((m * P) >> 32)
                assert -P < t < P
                acc += t
            assert acc % P == sum(PW[r - j][0][0] * dl[j] for j in range(r)) % P


def _adversarial_states(orc):
    st = [np.zeros(24, np.uint32), np.full(24, P - 1, np.uint32), np.array(orc.encode([P - 1] * 24), np.uint32),
          np.array(orc.encode(list(range(24))), np.uint32),
          np.full(24, 0x77FFFFFF, np.uint32)]  # the canonical word with the most 0xFF bytes
    return np.stack(st)


def test_emulator_tensor_form_permutation_matches_oracle(pkg, emu_lib, orc):
    st = np.concatenate([_adversarial_states(orc), rand_elems(np.random.default_rng(4), (100_000, 24))])
    with pkg.Context(0, 12, SMALL, lib=emu_lib) as c:
        got = c.op_poseidon2(st)
    exp = np.stack([orc.poseidon2_mix(s) for s in st])
    assert (got == exp).all()


@pytest.mark.gpu
def test_tensor_core_permutation_on_gpu(pkg, gpu_lib, orc):
    st = np.concatenate([_adversarial_states(orc), rand_elems(np.random.default_rng(5), ((1 << 20) - 5, 24))])
    with pkg.Context(0, 12, SMALL, lib=gpu_lib) as c:
        got = c.op_poseidon2(st)
        for n in (1, 127, 129, 1000):  # the last CTA partly idle
            assert (c.op_poseidon2(st[:n]) == got[:n]).all()
    exp = np.stack([orc.poseidon2_mix(s) for s in st])
    assert (got == exp).all()


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols", [(2, 40), (32, 16), (64, 33), (1 << 14, 7)])  # 2^14 rows: a level of 8192 in HashFoldKernel
def test_tensor_core_merkle_ragged_on_gpu(pkg, gpu_lib, orc, rows, cols):
    m = rand_elems(np.random.default_rng(rows * cols), (cols, rows))
    _, nodes = orc.merkle(m, True)
    with pkg.Context(0, 12, SMALL, lib=gpu_lib) as c:
        assert (c.op_merkle(m)[1:] == nodes[1:]).all()
