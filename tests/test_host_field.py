"""The host Goldilocks field (multi_stark_b200/host/goldilocks.hpp) and the CPU oracle's SIMD field ops (oracle/cpu_simd.hpp)
over the operand table of tests/_gl_model.py, against Python ints.

goldilocks.hpp is the field of the host prover layer and of the CPU oracle that every GPU parity test compares with, and
cpu_simd.hpp's row kernels carry the oracle's DFT: a wrong rare branch there would sit in the product and in the reference
alike, where parity cannot see it. The row kernels run at widths 1..17 (vector bodies and masked tails), with the AVX-512
kernels and, in a subprocess with ORC_NO_AVX512=1, the auto-vectorised clones."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import _gl_model as G
from tests import _naive as nv
from tests import _oracle as orc

P = G.P
M64 = G.M64
FP_FROM, FP_ADD, FP_SUB, FP_NEG, FP_MUL, FP_POW, FP_INV, FP_HALVE, SIMD_MUL, SIMD_ADD, SIMD_SUB, REDUCE128 = range(12)


@pytest.fixture(scope="module")
def L():
    return _lib()


def _lib():
    L = orc.lib()
    for name, args in {"orc_fp_op": [C.c_int, orc.u64p, orc.u64p, orc.u64p, C.c_uint64],
                       "orc_fp2_op": [C.c_int, orc.u64p, orc.u64p, orc.u64p, C.c_uint64],
                       "orc_fp_batch_inverse": [orc.u64p, orc.u64p, C.c_uint64],
                       "orc_dif_butterfly_row": [orc.u64p, orc.u64p, C.c_uint64, C.c_uint64],
                       "orc_scale_row": [orc.u64p, orc.u64p, C.c_uint64, C.c_uint64]}.items():
        getattr(L, name).argtypes = args
        getattr(L, name).restype = None
    return L


def _u64(xs):
    return np.ascontiguousarray(np.array([int(x) for x in xs], dtype=np.uint64))


def fp(L, op, a, b=None):
    a = _u64(a)
    b = _u64(b) if b is not None else np.zeros_like(a)
    out = np.empty_like(a)
    L.orc_fp_op(op, a, b, out, len(a))
    return [int(v) for v in out]


def _pairs(xs, ys):
    return [x for x in xs for y in ys], [y for x in xs for y in ys]


def _random(n, seed):
    rng = np.random.default_rng(seed)
    return [int(v) for v in rng.integers(0, 2**64, size=n, dtype=np.uint64)]


def _check(name, got, want, args):
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, "%s%r = %d, want %d" % (name, tuple(a[i] for a in args), g, w)


def test_fp_from_non_canonical_u64(L):
    xs = G.ANY_U64 + _random(10000, 1)
    _check("Fp(u64)", fp(L, FP_FROM, xs), [x % P for x in xs], (xs,))


def test_fp_arithmetic(L):
    ra, rb = _random(20000, 2), _random(20000, 3)
    a, b = _pairs(G.CLASSES, G.CLASSES)
    a, b = a + [x % P for x in ra], b + [x % P for x in rb]
    a += [x for x, _, _ in G.TARGETED.values()]
    b += [y for _, y, _ in G.TARGETED.values()]
    _check("+", fp(L, FP_ADD, a, b), [(x + y) % P for x, y in zip(a, b)], (a, b))
    _check("-", fp(L, FP_SUB, a, b), [(x - y) % P for x, y in zip(a, b)], (a, b))
    _check("*", fp(L, FP_MUL, a, b), [x * y % P for x, y in zip(a, b)], (a, b))
    _check("unary -", fp(L, FP_NEG, a), [-x % P for x in a], (a,))
    _check("halve", fp(L, FP_HALVE, a), [x * (P + 1) // 2 % P for x in a], (a,))
    # operands given non-canonical are reduced by Fp(u64) first
    na, nb = _pairs(G.ANY_U64, G.ANY_U64)
    _check("Fp(a) * Fp(b)", fp(L, FP_MUL, na, nb), [x * y % P for x, y in zip(na, nb)], (na, nb))
    _check("Fp(a) + Fp(b)", fp(L, FP_ADD, na, nb), [(x + y) % P for x, y in zip(na, nb)], (na, nb))


@pytest.mark.parametrize("e", [0, 1, 2, P - 2, P - 1, 2**64 - 1])
def test_fp_pow(L, e):
    xs = G.ANY_U64
    _check("pow(., %d)" % e, fp(L, FP_POW, xs, [e] * len(xs)), [pow(x, e, P) for x in xs], (xs,))


def test_fp_inverse_and_batch_inverse(L):
    xs = [x for x in G.ANY_U64 if x % P] + [x % P or 1 for x in _random(1000, 4)]
    want = [pow(x, P - 2, P) for x in xs]
    _check("inverse", fp(L, FP_INV, xs), want, (xs,))
    for n in (1, 2, 7, len(xs)):
        out = np.empty(n, dtype=np.uint64)
        L.orc_fp_batch_inverse(_u64(xs[:n]), out, n)
        assert [int(v) for v in out] == want[:n], n


def fp2(L, op, xs, ys):
    a = _u64([v for x in xs for v in x])
    b = _u64([v for y in ys for v in y])
    out = np.empty_like(a)
    L.orc_fp2_op(op, a, b, out, len(xs))
    return [(int(out[2 * i]), int(out[2 * i + 1])) for i in range(len(xs))]


def test_fp2(L):
    xs, ys = _pairs(G.E2_TABLE, G.E2_TABLE)
    for x, y, g in zip(xs, ys, fp2(L, 0, xs, ys)):
        assert g == nv.e_mul(x, y), ("*", x, y)
    nz = [x for x in G.E2_TABLE if x != (0, 0)]
    for x, g in zip(nz, fp2(L, 1, nz, nz)):
        assert g == nv.e_inv(x), ("inverse", x)
    for x, g in zip(G.E2_TABLE, fp2(L, 2, G.E2_TABLE, G.E2_TABLE)):
        assert g == (x[0] * (P + 1) // 2 % P, x[1] * (P + 1) // 2 % P), ("halve", x)


def test_simd_scalar_ops(L):
    ra, rb = _random(20000, 5), _random(20000, 6)
    a, b = _pairs(G.ANY_U64, G.ANY_U64)
    a, b = a + ra, b + rb
    _check("simd::gl_mul", fp(L, SIMD_MUL, a, b), [x * y % P for x, y in zip(a, b)], (a, b))
    ca, cb = _pairs(G.CLASSES, G.CLASSES)
    ca, cb = ca + [x % P for x in ra], cb + [x % P for x in rb]
    _check("simd::gl_add", fp(L, SIMD_ADD, ca, cb), [(x + y) % P for x, y in zip(ca, cb)], (ca, cb))
    _check("simd::gl_sub", fp(L, SIMD_SUB, ca, cb), [(x - y) % P for x, y in zip(ca, cb)], (ca, cb))


def _reduce128_branches(x):
    """gl_reduce128's three conditions, transcribed: lo < hi_hi (borrow), t0 + t1 overflows, r >= p."""
    lo, hi = x & M64, x >> 64
    hi_hi, hi_lo = hi >> 32, hi & G.M32
    borrow = lo < hi_hi
    t0 = (lo - hi_hi - (G.EPS if borrow else 0)) & M64
    t1 = hi_lo * G.EPS
    carry = t0 + t1 > M64
    r = (t0 + t1 + (G.EPS if carry else 0)) & M64
    return borrow, carry, r >= P


def test_gl_reduce128_reaches_every_branch(L):
    a, b = _pairs(G.CLASSES, G.CLASSES)
    a += [x for x, _, _ in G.TARGETED.values()]
    b += [y for _, y, _ in G.TARGETED.values()]
    prods = [x * y for x, y in zip(a, b)]
    seen = [set() for _ in range(3)]
    for x in prods:
        for k, c in enumerate(_reduce128_branches(x)):
            seen[k].add(c)
    assert seen == [{False, True}] * 3, seen
    # and gl_reduce128 itself, on those products and on any 128-bit (hi, lo) of the table
    lo, hi = [x & M64 for x in prods], [x >> 64 for x in prods]
    _check("gl_reduce128", fp(L, REDUCE128, lo, hi), [x % P for x in prods], (lo, hi))
    lo, hi = _pairs(G.ANY_U64, G.ANY_U64)
    _check("gl_reduce128", fp(L, REDUCE128, lo, hi), [(x + (y << 64)) % P for x, y in zip(lo, hi)], (lo, hi))


def row_kernel_failures():
    """The table through dif_butterfly_row and scale_row at widths 1..17; returns the mismatches (lanes past the width
    must stay untouched)."""
    L = _lib()
    fails = []
    cs, anys = G.CLASSES, G.ANY_U64
    sentinel = 0xA5A5A5A5A5A5A5A5
    for w in range(1, 18):
        for k in range(len(cs)):
            xa = [cs[(k + c) % len(cs)] for c in range(w)]
            xb = [cs[(3 * k + 5 * c + 1) % len(cs)] for c in range(w)]
            t = cs[(7 * k + w) % len(cs)]
            a, b = _u64(xa + [sentinel] * 8), _u64(xb + [sentinel] * 8)
            L.orc_dif_butterfly_row(a, b, t, w)
            want_a = [(x + y) % P for x, y in zip(xa, xb)] + [sentinel] * 8
            want_b = [(x - y) * t % P for x, y in zip(xa, xb)] + [sentinel] * 8
            if [int(v) for v in a] != want_a or [int(v) for v in b] != want_b:
                fails.append(("dif_butterfly_row", w, xa, xb, t))
            src = _u64([anys[(k + c) % len(anys)] for c in range(w)] + [sentinel] * 8)
            dst = _u64([sentinel] * (w + 8))
            L.orc_scale_row(dst, src, t, w)
            if [int(v) for v in dst] != [int(x) * t % P for x in src[:w]] + [sentinel] * 8:
                fails.append(("scale_row", w, [int(x) for x in src[:w]], t))
    return fails


def test_row_kernels(L):
    assert row_kernel_failures() == []


def test_row_kernels_without_avx512():
    code = ("import sys, json; sys.path.insert(0, %r); from tests import test_host_field as T; "
            "print(json.dumps(T.row_kernel_failures()))") % orc.ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=dict(os.environ, ORC_NO_AVX512="1"))
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout.strip().splitlines()[-1]) == []
