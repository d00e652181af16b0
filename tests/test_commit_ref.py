"""Pins tests/_commit_ref.py, the exact CPU reference of the NTT, LDE and Merkle kernels: field operations against Python
ints, every transform against the big-int sums of tests/_naive.py, the quotient slices against the C++ oracle, and the MMCS
restatement against test_oracle_hash.py's and the golden values of tests/golden/pcs_refs.json. No GPU needed."""
import json
import os
import random

import numpy as np
import pytest

from tests import _commit_ref as R
from tests import _naive as N
from tests.test_oracle_hash import py_mmcs_commit

P = R.P
EDGES = [0, 1, P - 1, P - 2, P - 2**32, 2**32 - 1, 2**32, 2**63, 2**63 + 1, 2**32 + 1]


def _vals(seed, k=300):
    rng = random.Random(seed)
    return EDGES + [rng.randrange(P) for _ in range(k)] + [P - 1 - rng.randrange(2**33) for _ in range(20)]


@pytest.mark.parametrize("op,ref", [(R.add, lambda a, b: (a + b) % P), (R.sub, lambda a, b: (a - b) % P),
                                    (R.mul, lambda a, b: a * b % P)])
def test_field_ops_against_python_ints(op, ref):
    v = _vals(1)
    A, B = np.meshgrid(np.array(v, dtype=np.uint64), np.array(v, dtype=np.uint64))
    got = op(A, B)
    want = np.array([[ref(int(a), int(b)) for a, b in zip(ra, rb)] for ra, rb in zip(A, B)], dtype=np.uint64)
    assert np.array_equal(got, want)
    assert (got < np.uint64(P)).all()


def test_generators_and_powers():
    for k in range(0, 33):
        g = R.two_adic_generator(k)
        assert g == N.two_adic_generator(k)
        assert pow(g, 1 << k, P) == 1 and (k == 0 or pow(g, 1 << (k - 1), P) == P - 1)
    assert [int(x) for x in R.powers(7, 70)] == [pow(7, i, P) for i in range(70)]
    assert [int(x) for x in R.rev_perm(4)] == [N.rev(i, 4) for i in range(16)]


def _cols(seed, n, w):
    rng = random.Random(seed)
    cols = [[rng.randrange(P) for _ in range(n)] for _ in range(w)]
    cols[0][:min(n, 3)] = [P - 1, 0, P - 1][:min(n, 3)]
    return cols, np.array(cols, dtype=np.uint64).T.copy()


@pytest.mark.parametrize("log_n", range(0, 7))
def test_dft_idft_against_naive(log_n):
    n = 1 << log_n
    cols, m = _cols(log_n, n, 3)
    y = R.dft(m)
    assert [[int(x) for x in y[:, c]] for c in range(3)] == [N.dft(col) for col in cols]
    assert [[int(x) for x in R.idft(m)[:, c]] for c in range(3)] == [N.idft(col) for col in cols]
    br = R.dft_bitrev(m)
    assert np.array_equal(br, y[[N.rev(i, log_n) for i in range(n)]])
    assert np.array_equal(R.idft(y), m)


@pytest.mark.parametrize("log_n", [0, 1, 2, 3, 5])
@pytest.mark.parametrize("added_bits", [0, 1, 2, 3])
def test_coset_lde_against_naive(log_n, added_bits):
    n = 1 << log_n
    cols, m = _cols(10 * log_n + added_bits, n, 2)
    for shift in (7, 1, P - 1, 0x1234567890ABCDEF % P):
        got = R.coset_lde_bitrev(m, added_bits, shift)
        assert [[int(x) for x in got[:, c]] for c in range(2)] == [N.coset_lde_bitrev(col, added_bits, shift) for col in cols]


@pytest.mark.parametrize("log_n,added_bits", [(0, 2), (2, 1), (3, 3), (5, 0), (4, 2)])
def test_lde_from_shifted_coefficients_against_naive(log_n, added_bits):
    """Zero-padded coefficients, one DFT: stored[i] = poly(w_{nB}^{rev(i)})."""
    n = 1 << log_n
    cols, m = _cols(log_n, n, 2)
    got = R.lde_from_shifted_coefficients(m, added_bits)
    lb = log_n + added_bits
    w = N.two_adic_generator(lb)
    for c in range(2):
        assert [int(x) for x in got[:, c]] == [N.poly_eval(cols[c], pow(w, N.rev(i, lb), P)) for i in range(n << added_bits)]


@pytest.mark.parametrize("log_nq,q,d", [(0, 1, 1), (2, 2, 3), (4, 4, 2), (6, 2, 1), (10, 4, 2), (12, 1, 2)])
def test_shifted_quotient_slices_against_oracle(oracle, log_nq, q, d):
    m = np.random.default_rng(log_nq).integers(0, P, size=(1 << log_nq, d), dtype=np.uint64)
    want = np.empty(((1 << log_nq) // q, q * d), dtype=np.uint64)
    oracle.orc_shifted_quotient_slices(m, m.shape[0], d, q, want)
    assert np.array_equal(R.shifted_quotient_slices(m, q), want)


@pytest.mark.parametrize("shapes", [[(16, 1)], [(16, 3), (16, 2)], [(4, 5), (32, 1), (32, 9), (8, 2)], [(2, 140)],
                                    [(64, 14), (2, 1)], [(8, 300), (8, 1), (4, 129)], [(8, 0), (8, 2), (2, 0), (1, 3)]])
def test_mmcs_against_python_restatement(shapes):
    rng = np.random.default_rng(len(shapes))
    mats = [rng.integers(0, P, size=s, dtype=np.uint64) for s in shapes]
    layers = R.mmcs_commit(mats)
    want = py_mmcs_commit(mats)
    assert [[bytes(d) for d in l] for l in layers] == want
    max_h = max(h for h, _ in shapes)
    for i in {0, 1 % max_h, max_h - 1}:
        assert [int(x) for x in R.open_rows(mats, i)] == \
            [int(v) for m in mats for v in m[i >> ((max_h.bit_length() - 1) - (m.shape[0].bit_length() - 1))]]
        assert [bytes(d) for d in R.open_path(layers, i)] == [want[l][(i >> l) ^ 1] for l in range(len(want) - 1)]


def test_mmcs_against_golden_pcs_refs():
    """The 3-matrix case of gen_pcs_refs (heights 8/4/2, opened at 5) and the single-row leaves."""
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "pcs_refs.json")))
    limbs = lambda d: [int(x) for x in np.frombuffer(bytes(d), dtype="<u8")]
    m0 = np.zeros((8, 2), dtype=np.uint64); m0[5] = [11, 12]
    m1 = np.zeros((4, 3), dtype=np.uint64); m1[2] = [107, 108, 109]
    m2 = np.zeros((2, 1), dtype=np.uint64); m2[1] = [202]
    layers = R.mmcs_commit([m0, m1, m2])
    assert limbs(layers[-1][0]) == g["COMMIT"]
    assert [int(x) for x in R.open_rows([m0, m1, m2], 5)] == sum(g["OPENED"], [])
    for i, s in enumerate(R.open_path(layers, 5)):
        assert limbs(s) == g["SIB%d" % i]
    for n in (3, 17, 22, 20):
        assert limbs(R.mmcs_commit([np.arange(1, n + 1, dtype=np.uint64).reshape(1, n)])[-1][0]) == g["LEAF%d" % n]


def test_open_batch_multi_layout():
    """Per tree: the rows of every query, then (after all trees' rows) the paths of every query, tree after tree; a
    rows-only part contributes no path and a paths-only tree no row."""
    rng = np.random.default_rng(3)
    a = [rng.integers(0, P, size=(8, 2), dtype=np.uint64), rng.integers(0, P, size=(2, 1), dtype=np.uint64)]
    b = [rng.integers(0, P, size=(4, 3), dtype=np.uint64)]
    la, lb = R.mmcs_commit(a), R.mmcs_commit(b)
    o, p = R.open_batch_multi([(a, la), (b, None), ([], lb)], [0, 1, 1], [7, 0, 7])
    assert [int(x) for x in o] == [int(v) for i in (7, 0, 7) for v in R.open_rows(a, i)] + \
        [int(v) for i in (3, 0, 3) for v in b[0][i]]
    assert p.shape == (3 * 3 + 3 * 2, 32)
    assert np.array_equal(p[:3], R.open_path(la, 7)) and np.array_equal(p[9:11], R.open_path(lb, 3))
