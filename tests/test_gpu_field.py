"""The compiled Goldilocks primitives of csrc/gl.cuh on the GPU against Python ints.

tests/gl_harness.cu (test-only, not part of libmsgpu) is compiled here with the library's own nvcc flags and runs each
primitive over the operand table of tests/_gl_model.py: every pair of edge classes and non-canonical values, the targeted
pairs, the Acc160 limb states and the extension-field elements. test_field_model.py shows on the CPU that this table drives
every carry and borrow of gl.cuh's asm both ways (or never, where a comment says so), so the same operands do it here.
Random bulk (2^22 seeded pairs per binary op) is checked against tests/_commit_ref.py's numpy field."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import _commit_ref as R
from tests import _gl_model as G
from tests import _naive as nv

pytestmark = pytest.mark.gpu

P = G.P
HERE = os.path.dirname(os.path.abspath(__file__))
(CANON, ADD_LAZY, SUB_LAZY, ADD, SUB, NEG, REDUCE128_LAZY, MUL, MUL_LAZY, SQR, POW, INV, HALVE, GF_ADD, GF_SUB,
 GF_REDUCE128, GF_MUL, MUL7, POW2_MOD_P, REV_BITS, E2_ADD, E2_SUB, E2_MUL, E2_MUL_BASE, E2_INV) = range(25)
N_BULK = 1 << 22

u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")
u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")


@pytest.fixture(scope="module")
def gh(tmp_path_factory):
    from multi_stark_b200 import build
    so = str(tmp_path_factory.mktemp("gl_harness") / "gl_harness.so")
    subprocess.run([build.NVCC, *build.FLAGS, "-shared", "-o", so, os.path.join(HERE, "gl_harness.cu")], check=True)
    L = C.CDLL(so)
    for name, args in {"gh_base": [C.c_int, u64p, u64p, u64p, C.c_uint64],
                       "gh_e2": [C.c_int, u64p, u64p, u64p, C.c_uint64],
                       "gh_mul_pow2": [C.c_int, u64p, u64p, C.c_uint64],
                       "gh_acc_mac": [u32p, u64p, u64p, u32p, u64p, C.c_uint64],
                       "gh_acc_repeat": [C.c_uint64, C.c_uint64, C.c_uint64, u32p, u64p],
                       "gh_pow_lookup": [u64p, C.c_uint64, u64p, C.c_uint64, C.c_uint32, u64p, u64p, C.c_uint64]}.items():
        getattr(L, name).argtypes = args
        getattr(L, name).restype = C.c_int
    return L


def _u64(xs):
    return np.ascontiguousarray(np.array([int(x) for x in xs], dtype=np.uint64))


def base(gh, op, a, b=None):
    a = _u64(a)
    b = _u64(b) if b is not None else np.zeros_like(a)
    out = np.empty_like(a)
    assert gh.gh_base(op, a, b, out, len(a)) == 0
    return [int(v) for v in out]


def _pairs(xs, ys):
    return [x for x in xs for y in ys], [y for x in xs for y in ys]


def _check(name, got, want, args, lazy=False):
    for i, (g, w) in enumerate(zip(got, want)):
        ok = (g % P == w % P) if lazy else (g == w)
        assert ok, "%s%r = %d, want %d" % (name, tuple(a[i] for a in args), g, w)


# ---- the operand table ----------------------------------------------------------------------------------------------------
def test_base_field_table(gh):
    xs = G.ANY_U64
    aa, ab = _pairs(G.ANY_U64, G.ANY_U64)
    ca, cb = _pairs(G.CLASSES, G.CLASSES)
    la, lb = _pairs(G.ANY_U64, G.CLASSES + [P])  # sub_lazy takes b in [0, p]; add_lazy b < p
    lbc = [b % P for b in lb]
    _check("canon", base(gh, CANON, xs), [x % P for x in xs], (xs,))
    _check("add_lazy", base(gh, ADD_LAZY, la, lbc), [a + b for a, b in zip(la, lbc)], (la, lbc), lazy=True)
    _check("sub_lazy", base(gh, SUB_LAZY, la, lb), [a - b for a, b in zip(la, lb)], (la, lb), lazy=True)
    for name, op in (("add", ADD), ("gf::add", GF_ADD)):
        _check(name, base(gh, op, ca, cb), [(a + b) % P for a, b in zip(ca, cb)], (ca, cb))
    for name, op in (("sub", SUB), ("gf::sub", GF_SUB)):
        _check(name, base(gh, op, ca, cb), [(a - b) % P for a, b in zip(ca, cb)], (ca, cb))
    cs = G.CLASSES
    _check("neg", base(gh, NEG, cs), [-x % P for x in cs], (cs,))
    _check("halve", base(gh, HALVE, cs), [x * (P + 1) // 2 % P for x in cs], (cs,))
    _check("mul7", base(gh, MUL7, cs), [7 * x % P for x in cs], (cs,))
    _check("reduce128_lazy", base(gh, REDUCE128_LAZY, aa, ab), [lo + (hi << 64) for lo, hi in zip(aa, ab)], (aa, ab),
           lazy=True)
    _check("gf::reduce128", base(gh, GF_REDUCE128, aa, ab), [(lo + (hi << 64)) % P for lo, hi in zip(aa, ab)], (aa, ab))
    ma = aa + [a for a, _, _ in G.TARGETED.values()]
    mb = ab + [b for _, b, _ in G.TARGETED.values()]
    for name, op in (("mul", MUL), ("gf::mul", GF_MUL)):
        _check(name, base(gh, op, ma, mb), [a * b % P for a, b in zip(ma, mb)], (ma, mb))
    _check("mul_lazy", base(gh, MUL_LAZY, ma, mb), [a * b for a, b in zip(ma, mb)], (ma, mb), lazy=True)
    _check("sqr", base(gh, SQR, xs), [x * x % P for x in xs], (xs,))


def test_lazy_results_stay_in_u64_and_canonical_ones_below_p(gh):
    """gl::sub(a, b) with canonical operands is canonical: sub_lazy's one fix-up suffices."""
    ca, cb = _pairs(G.CLASSES, G.CLASSES)
    assert all(r < P for r in base(gh, SUB_LAZY, ca, cb))


@pytest.mark.parametrize("e", [0, 1, P - 2, P - 1, 2**64 - 1])
def test_pow(gh, e):
    xs = G.ANY_U64
    _check("pow(., %d)" % e, base(gh, POW, xs, [e] * len(xs)), [pow(x, e, P) for x in xs], (xs,))


def test_inv(gh):
    xs = G.ANY_U64
    _check("inv", base(gh, INV, xs), [pow(x, P - 2, P) for x in xs], (xs,))  # inv(0) = 0 (and inv(p) = 0)


def test_mul_pow2_every_exponent(gh):
    xs = _u64(G.ANY_U64 + [int(v) for v in np.random.default_rng(3).integers(0, 2**64, size=4096, dtype=np.uint64)])
    out = np.empty_like(xs)
    for e in range(1, 96):
        assert gh.gh_mul_pow2(e, xs, out, len(xs)) == 0
        _check("gf::mul_pow2(., %d)" % e, [int(v) for v in out], [(int(x) << e) % P for x in xs], (xs,))
    assert gh.gh_mul_pow2(0, xs, out, len(xs)) != 0 and gh.gh_mul_pow2(96, xs, out, len(xs)) != 0


def test_pow2_mod_p(gh):
    es = list(range(96))
    _check("gf::pow2_mod_p", base(gh, POW2_MOD_P, es), [pow(2, e, P) for e in es], (es,))


# ---- Acc160 ---------------------------------------------------------------------------------------------------------------
def test_acc160_limb_states(gh):
    sa, sb = _pairs(G.CLASSES, G.CLASSES)
    lanes = [(s, a, b) for s in G.acc_states() for a, b in zip(sa, sb) if G.limbs_value(s) + a * b < 2**160]
    st = np.ascontiguousarray(np.array([s for s, _, _ in lanes], dtype=np.uint32).reshape(-1))
    a, b = _u64([a for _, a, _ in lanes]), _u64([b for _, _, b in lanes])
    out_st = np.empty_like(st)
    out = np.empty(2 * len(lanes), dtype=np.uint64)
    assert gh.gh_acc_mac(st, a, b, out_st, out, len(lanes)) == 0
    out_st = out_st.reshape(-1, 5)
    for k, (s, x, y) in enumerate(lanes):
        want = G.limbs_value(s) + x * y
        assert G.limbs_value(out_st[k]) == want, (s, x, y)
        assert int(out[2 * k]) == G.limbs_value(s) % P, s
        assert int(out[2 * k + 1]) == want % P, (s, x, y)
    # every state's l4 fed through acc_reduce, including 0xffffffff
    assert {s[4] for s, _, _ in lanes} == {0, 1, G.M32}


def test_acc160_many_terms(gh):
    """One thread, 2^20 terms of (p - 1)^2: l4 and the carries into it run far past any one term."""
    terms = 1 << 20
    st, out = np.zeros(5, dtype=np.uint32), np.zeros(1, dtype=np.uint64)
    assert gh.gh_acc_repeat(P - 1, P - 1, terms, st, out) == 0
    want = terms * (P - 1)**2
    assert G.limbs_value(st) == want
    assert int(out[0]) == want % P


# ---- extension field ------------------------------------------------------------------------------------------------------
def e2(gh, op, xs, ys):
    a = _u64([v for x in xs for v in x])
    b = _u64([v for y in ys for v in y])
    out = np.empty_like(a)
    assert gh.gh_e2(op, a, b, out, len(xs)) == 0
    return [(int(out[2 * i]), int(out[2 * i + 1])) for i in range(len(xs))]


def test_extension_field(gh):
    xs, ys = _pairs(G.E2_TABLE, G.E2_TABLE)
    for name, op, ref in (("e2_add", E2_ADD, nv.e_add), ("e2_sub", E2_SUB, nv.e_sub), ("e2_mul", E2_MUL, nv.e_mul)):
        got = e2(gh, op, xs, ys)
        for x, y, g in zip(xs, ys, got):
            assert g == ref(x, y), (name, x, y)
    for x, y, g in zip(xs, ys, e2(gh, E2_MUL_BASE, xs, ys)):
        assert g == (x[0] * y[0] % P, x[1] * y[0] % P), ("e2_mul_base", x, y[0])
    for x, g in zip(G.E2_TABLE, e2(gh, E2_INV, G.E2_TABLE, G.E2_TABLE)):
        assert g == nv.e_inv(x), ("e2_inv", x)  # (0, 0) -> (0, 0)


# ---- indexing helpers -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("h1", [0, 1, 5, 10])
def test_pow_lookup(gh, h1):
    g, c, log_n = nv.two_adic_generator(12), 7, 12
    lo = _u64([c * pow(g, i, P) % P for i in range(1 << h1)])
    hi = _u64([pow(g, i << h1, P) for i in range((1 << log_n) >> h1)])
    es = _u64(range(1 << log_n))
    out = np.empty_like(es)
    assert gh.gh_pow_lookup(lo, len(lo), hi, len(hi), h1, es, out, len(es)) == 0
    assert [int(v) for v in out] == [c * pow(g, e, P) % P for e in range(1 << log_n)]


def test_rev_bits(gh):
    xs, bits = [], []
    for nb in (0, 1, 31, 32):
        for x in (0, 1, 2, 0x12345678 & ((1 << nb) - 1), (1 << nb) - 1, 0x80000000 >> (32 - nb) if nb else 0):
            xs.append(x)
            bits.append(nb)
    want = [nv.rev(x, nb) for x, nb in zip(xs, bits)]
    assert base(gh, REV_BITS, xs, bits) == want


# ---- random bulk against the numpy field ----------------------------------------------------------------------------------
def _bulk(gh, op, a, b):
    out = np.empty_like(a)
    assert gh.gh_base(op, a, b, out, len(a)) == 0
    return out


def _canon_np(x):
    return np.where(x >= R._P, x - R._P, x)


def test_random_bulk(gh):
    rng = np.random.default_rng(22)
    a = rng.integers(0, 2**64, size=N_BULK, dtype=np.uint64)
    b = rng.integers(0, 2**64, size=N_BULK, dtype=np.uint64)
    ca, cb = _canon_np(a), _canon_np(b)
    for name, op, want in (("add", ADD, R.add(ca, cb)), ("gf::add", GF_ADD, R.add(ca, cb)),
                           ("sub", SUB, R.sub(ca, cb)), ("gf::sub", GF_SUB, R.sub(ca, cb)),
                           ("mul", MUL, R.mul(ca, cb)), ("gf::mul", GF_MUL, R.mul(ca, cb))):
        got = _bulk(gh, op, ca, cb)
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, (name, int(ca[bad[0]]), int(cb[bad[0]]), int(got[bad[0]]))
    # any-u64 operands; lazy forms compared after one reduction
    for name, op, x, y, want, lazy in (
            ("mul(any)", MUL, a, b, R.mul(a, b), False), ("mul_lazy", MUL_LAZY, a, b, R.mul(a, b), True),
            ("add_lazy", ADD_LAZY, a, cb, R.add(_canon_np(a), cb), True),
            ("sub_lazy", SUB_LAZY, a, cb, R.sub(_canon_np(a), cb), True),
            ("gf::reduce128", GF_REDUCE128, a, b, R.add(R.mul(_canon_np(b), R._EPS), _canon_np(a)), False),
            ("reduce128_lazy", REDUCE128_LAZY, a, b, R.add(R.mul(_canon_np(b), R._EPS), _canon_np(a)), True),
            ("canon", CANON, a, b, _canon_np(a), False)):
        got = _bulk(gh, op, x, y)
        if lazy:
            got = _canon_np(got)
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, (name, int(x[bad[0]]), int(y[bad[0]]), int(got[bad[0]]))
