"""Blocked S-box chain of the tensor-core Poseidon2 partial rounds (csrc/poseidon2.cuh, P2TC_BLOCKS).

The 21 partial rounds are cut into blocks; after each block one small GEMM adds the block's deltas to the TMEM planes of all
later rounds, so SIMT sums only the terms inside a block.  CPU tier: the blocked chain against the full triangular sum and
step-by-step rounds in exact integers; a numpy model of the block and GEMM 2 tables built like the C++ tables (including
GEMM 2's reordered rows) with the accumulator bound on adversarial words; the emulator's permutation against the oracle for
every block count 1..4.  GPU tier: PermuteKernel on 2^20 states with a partly idle CTA, and a Merkle tree of 2^14 rows x
192 columns, the bench's column count, whose 8192-node level runs through HashFoldKernel.
"""
import os
import subprocess

import numpy as np
import pytest
from conftest import ROOT, SMALL, rand_elems
from test_p2_partial_gemm import B1, P, P_INV, PW, R, RC_PART, K1, N1, N2, _adversarial_states, m_int, planes, reduce

HALF = (P - 1) // 2


def layout(nb):
    """(rounds per block, A words per block, A row words) -- P2TC_BS, P2TC_BW, P2TC_AW."""
    bs = -(-21 // nb)
    bw = -(-bs // 8) * 8
    return bs, bw, 24 + nb * bw


def blk_c0(nb, b):
    return (4 * (b * layout(nb)[0] - 1)) & ~15


def block_table(nb, b):
    """Logical B operand of block GEMM b (A = the deltas of block b - 1): rows = planes of TMEM columns [c0, 80)."""
    bs, bw, _ = layout(nb)
    c0 = blk_c0(nb, b)
    rows = []
    for o in range((N1 - c0) // 4):
        r = (c0 + 4 * o) // 4 + 1
        rows.append([PW[r - ((b - 1) * bs + i)][0][0] for i in range(bs)] + [0] * (bw - bs) if r >= b * bs else [0] * bw)
    return planes(rows, 4 * bw)


def gemm2_table(nb):
    bs, bw, aw = layout(nb)
    rows = []
    for o in range(24):
        m = list(PW[21][o]) + [0] * (aw - 24)
        for j in range(21):
            m[24 + j // bs * bw + j % bs] = PW[21 - j][o][0]
        rows.append(m)
    return planes(rows, 4 * aw)


def a_row(nb, v, d):
    """[v | delta blocks, zero-padded] as the kernel writes it."""
    bs, bw, aw = layout(nb)
    w = np.zeros((v.shape[0], aw), np.uint32)
    w[:, :24] = v
    for j in range(21):
        w[:, 24 + j // bs * bw + j % bs] = d[:, j]
    return w


def planes_of(words, b):
    a = np.ascontiguousarray(words.astype("<u4")).view(np.uint8).astype(np.int64)
    return a @ b.T


def sbox_delta(y, r):
    return (pow((y + RC_PART[r]) % P, 7, P) - y) % P


@pytest.mark.parametrize("nb", [1, 2, 3, 4])
def test_blocked_chain_equals_full_triangular_sum(nb):
    """In exact integers: v_r[0] from the block-entry values plus the in-block sum, with deltas from the S-box, gives the
    same chain and the same v_21 as 21 step-by-step partial rounds; the in-block terms in signed groups of <= 4 stay in
    range of one signed REDC each (p2tc_dot4)."""
    bs = layout(nb)[0]
    c_mont = [0] + [PW[k][0][0] * R % P for k in range(1, 21)]
    c_bal = [x - P if x > HALF else x for x in c_mont]
    rng = np.random.default_rng(10 + nb)
    for trial in range(30):
        v = [int(x) for x in rng.integers(0, P, 24)] if trial else [P - 1] * 24
        st, ref_d = list(v), []
        for r in range(21):
            ref_d.append(sbox_delta(st[0], r))
            st[0] = (st[0] + ref_d[-1]) % P
            st = m_int(st)
        d = []
        for b in range(nb):
            r0, r1 = b * bs, min(b * bs + bs, 21)
            entry = [(sum(PW[r][0][i] * v[i] for i in range(24)) + sum(PW[r - j][0][0] * d[j] for j in range(r0))) % P
                     for r in range(r0, r1)]  # what TMEM holds after GEMM 1 and the block GEMMs before block b
            for r in range(r0, r1):
                db = [x - P if x > HALF else x for x in d]
                y = entry[r - r0]
                for j0 in range(r0, r, 4):
                    vsum = sum(c_bal[r - j] * db[j] for j in range(j0, min(r, j0 + 4)))
                    assert abs(vsum) < (1 << 31) * P
                    m = (vsum & 0xFFFFFFFF) * P_INV & 0xFFFFFFFF
                    m = m - (1 << 32) if m >= 1 << 31 else m
                    t = (vsum >> 32) - ((m * P) >> 32)
                    assert -P < t < P
                    y = (y + t) % P  # c carries 2^32, the REDC takes it off: t = sum c_{r-j} delta_j mod p
                d.append(sbox_delta(y, r))
        assert d == ref_d
        assert st == [(sum(PW[21][o][i] * v[i] for i in range(24)) + sum(PW[21 - j][o][0] * d[j] for j in range(21))) % P
                      for o in range(24)]


@pytest.mark.parametrize("nb", [1, 2, 3, 4])
def test_block_tables_accumulate_exactly_on_adversarial_words(nb):
    """GEMM 1 plus the block GEMMs accumulated into the same columns give a_r . v + sum_{j < block start} c_{r-j} delta_j
    for every round; GEMM 2 over the reordered A row gives v_21; no plane reaches 2^24 on all-0xFF bytes, p - 1, its
    Montgomery form or the largest delta."""
    bs, bw, aw = layout(nb)
    rng = np.random.default_rng(20 + nb)
    n = 2048
    v = rng.integers(0, 1 << 32, (n, 24), dtype=np.uint64).astype(np.uint32)
    d = rng.integers(0, P, (n, 21), dtype=np.uint32)
    v[0], d[0] = 0xFFFFFFFF, P - 1
    v[1], d[1] = P - 1, HALF
    v[2], d[2] = (P - 1) * R % P, P - 1
    v[3], d[3] = 0x77FFFFFF, 0x77FFFFFF  # the canonical word with the most 0xFF bytes
    w = a_row(nb, v, d)
    tm = np.zeros((n, 128), np.int64)
    tm[:, :N1] = planes_of(v, B1)
    for b in range(1, nb):
        c0 = blk_c0(nb, b)
        tm[:, c0:N1] += planes_of(w[:, 24 + (b - 1) * bw: 24 + b * bw], block_table(nb, b))
    assert tm.max() < 1 << 24
    got1 = reduce(tm[:, :N1])
    vi, di = v.astype(object), d.astype(object)
    for r in range(1, 21):
        r0 = r // bs * bs
        exp = (vi @ np.array(PW[r][0], dtype=object) + sum(di[:, j] * PW[r - j][0][0] for j in range(r0))) % P
        assert (got1[:, r - 1] == exp).all()
    q2 = planes_of(w, gemm2_table(nb))
    assert q2.shape[1] == N2 and q2.max() < 1 << 24
    full = np.array([PW[21][o] + [PW[21 - j][o][0] for j in range(21)] for o in range(24)], dtype=object)
    assert (reduce(q2) == (np.concatenate([vi, di], axis=1) @ full.T) % P).all()


@pytest.mark.parametrize("nb", [1, 2, 3, 4])
def test_block_layout_fits_the_tensor_core_shapes(nb):
    """Each block starts on a 32-byte K step, block GEMMs write whole 16-column groups inside GEMM 1's 80 columns (N a
    multiple of 16 in [16, 256] for M = 128), and GEMM 2's K covers the row in 32-byte steps."""
    bs, bw, aw = layout(nb)
    assert bw % 8 == 0 and (4 * aw) % 32 == 0 and (4 * 24) % 32 == 0
    for b in range(1, nb):
        c0 = blk_c0(nb, b)
        assert c0 % 16 == 0 and c0 <= 4 * (b * bs - 1) and (N1 - c0) % 16 == 0 and 16 <= N1 - c0 <= 256
    assert K1 == 96


@pytest.fixture(scope="module")
def emu_variants(pkg, tmp_path_factory):
    """The host emulator built for every block count."""
    out = tmp_path_factory.mktemp("emu_blocks")
    src = os.path.join(ROOT, "hyperfridge-r0_b200", "csrc", "hfb200.cu")
    procs = {}
    for nb in (1, 2, 3, 4):
        so = str(out / ("libhfb200_emu_b%d.so" % nb))
        procs[nb] = (so, subprocess.Popen(["g++", "-x", "c++", "-DHFB200_EMU", "-DP2TC_BLOCKS=%d" % nb, "-O2", "-std=c++17", "-fPIC",
                                           "-fopenmp", "-Wno-unknown-pragmas", "-I/usr/local/cuda/include", "-shared", "-o", so, src]))
    libs = {}
    for nb, (so, p) in procs.items():
        assert p.wait() == 0
        libs[nb] = pkg.load_library(so)
    return libs


@pytest.mark.parametrize("nb", [1, 2, 3, 4])
def test_emulator_blocked_permutation_matches_oracle(pkg, emu_variants, orc, nb):
    lib = emu_variants[nb]
    st = np.concatenate([_adversarial_states(orc), rand_elems(np.random.default_rng(30 + nb), (100_000, 24))])
    with pkg.Context(0, 12, SMALL, lib=lib) as c:
        got = c.op_poseidon2(st)
    exp = np.stack([orc.poseidon2_mix(s) for s in st])
    assert (got == exp).all()


@pytest.mark.gpu
def test_blocked_permute_kernel_on_gpu(pkg, gpu_lib, orc):
    st = np.concatenate([_adversarial_states(orc), rand_elems(np.random.default_rng(40), ((1 << 20) - 5, 24))])
    exp = np.stack([orc.poseidon2_mix(s) for s in st])
    with pkg.Context(0, 12, SMALL, lib=gpu_lib) as c:
        assert (c.op_poseidon2(st) == exp).all()
        assert (c.op_poseidon2(st[:200]) == exp[:200]).all()  # the second CTA runs 56 idle states


@pytest.mark.gpu
def test_blocked_merkle_192_columns_on_gpu(pkg, gpu_lib, orc):
    m = rand_elems(np.random.default_rng(41), (192, 1 << 14))
    _, nodes = orc.merkle(m, True)
    with pkg.Context(0, 12, SMALL, lib=gpu_lib) as c:
        assert (c.op_merkle(m)[1:] == nodes[1:]).all()
