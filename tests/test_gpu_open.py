"""Pcs::open kernel by kernel (multi_stark_b200/csrc/fri.cu) against a big-int reference kept in this file.

Every column is a polynomial f_c whose coefficients the test chooses. Its opened value at z is f_c(z) by Horner in the
extension field (not the barycentric formula the kernels use), stored LDE row i is f_c(7 * w_N^rev(i)), the reduced inputs
follow p3 `TwoAdicFriPcs::open` (rounds, then matrices, then points; alpha offset alpha^num_reduced[h]) and a fold is
`fold_row` of the restated verifier plus beta^2 times the next-height input. The device must match bit for bit:
  * opened values (msgpu_open_begin / msgpu_open_values): every chunk width of k_bary_partial, 1 to 9 points per matrix
    (all four template instances and the groups of more than four), points shared between heights, base-field points,
    several rounds, the one-row low coset, and large heights where k_bary_partial loops over its grid;
  * reduced inputs (msgpu_open_reduce / msgpu_open_read_input): contiguous and strided tiles, every tile height of
    k_reduce_openings, and the widest matrix it accepts;
  * the commit phase with host betas (every length from 2 to 2^14, across the k_fri_fold / k_fri_fold_commit boundary, with
    and without a rolled-in input) against the Python Merkle tree, and with the transcript on the device against PyChallenger;
  * a row-sharded opening on one GPU against the unsharded one, the refused calls, and whole proofs of wide circuits."""
import ctypes as C
import random

import numpy as np
import pytest

from tests import _oracle as orc
from tests import _proof
from tests import _pyverifier as pv
from tests.test_oracle_hash import py_mmcs_commit

P = pv.P
E = pv.E
G = pv.GENERATOR


@pytest.fixture(scope="module")
def gpu():
    import multi_stark_b200 as ms
    ctx = ms.GpuContext(0)
    yield ms, ctx
    ctx.close()


# ---- the reference ----------------------------------------------------------------------------------------------------
def col_values(F, xs):
    """(len(xs), w) uint64: f_c(x) for every x, where F[k][c] is the coefficient of x^k in f_c."""
    X = np.array([x % P for x in xs], dtype=object)[:, None]
    acc = np.zeros((len(xs), len(F[0])), dtype=object)
    for row in reversed(F):
        acc = (acc * X + np.array(row, dtype=object)[None, :]) % P
    return acc.astype(np.uint64)


def eval_at(F, z):
    """[f_c(z)] in the extension field, by Horner."""
    out = []
    for c in range(len(F[0])):
        acc = E(0)
        for row in reversed(F):
            acc = acc * z + row[c]
        out.append(acc)
    return out


def lde_x(i, log_h):
    """the point of stored LDE row i: GENERATOR * w_N^rev(i)"""
    return G * pow(pv.two_adic_generator(log_h), pv.rev_bits(i, log_h), P) % P


class Mat:
    """A committed matrix: columns f_c of degree < len(F), trace height 2^log_n, LDE height 2^(log_n + log_blowup)."""

    def __init__(self, F, log_n, log_blowup, points=()):
        self.F, self.log_n, self.log_h = F, log_n, log_n + log_blowup
        self.w = len(F[0])
        self.points = list(points)
        self._rows = {}

    def natural(self):
        n = 1 << self.log_n
        w = pv.two_adic_generator(self.log_n)
        xs = [1] * n
        for i in range(1, n):
            xs[i] = xs[i - 1] * w % P
        return col_values(self.F, xs)

    def lde_rows(self, idx):
        missing = [i for i in idx if i not in self._rows]
        if missing:
            for i, r in zip(missing, col_values(self.F, [lde_x(i, self.log_h) for i in missing])):
                self._rows[i] = [int(v) for v in r]
        return [self._rows[i] for i in idx]

    def values(self):
        return [eval_at(self.F, z) for z in self.points]


def rand_coeffs(rnd, deg, w):
    return [[rnd.randrange(P) for _ in range(w)] for _ in range(deg)]


def rand_ext(rnd):
    return E(rnd.randrange(P), rnd.randrange(P))


def reduce_ref(rounds, alpha, rows_of):
    """p3 TwoAdicFriPcs::open's reduced inputs: {log_h: {row: value}} for the rows rows_of(log_h) of every committed height."""
    max_w = max(m.w for r in rounds for m in r)
    apow = [E(1)]
    for _ in range(max_w):
        apow.append(apow[-1] * alpha)
    num_reduced, out = {}, {}
    for rnd in rounds:
        for m in rnd:
            lh = m.log_h
            vec = out.setdefault(lh, {i: E(0) for i in rows_of(lh)})
            if not m.points:
                continue
            terms = []  # (alpha offset, sum_c alpha^c y_c, z) per point
            for z, ys in zip(m.points, m.values()):
                yred = E(0)
                for c in range(m.w):
                    yred = yred + apow[c] * ys[c]
                terms.append((alpha.pow(num_reduced.get(lh, 0)), yred, z))
                num_reduced[lh] = num_reduced.get(lh, 0) + m.w
            idx = sorted(vec)
            for i, row in zip(idx, m.lde_rows(idx)):
                mred = E(sum(apow[c].a * row[c] for c in range(m.w)), sum(apow[c].b * row[c] for c in range(m.w)))
                x = lde_x(i, lh)
                for aoff, yred, z in terms:
                    vec[i] = vec[i] + aoff * (yred - mred) * (z - x).inverse()
    return out


def fold_ref(vec, beta, roll=None):
    """out[i] = fold_row(i, log_half, beta, in[2i], in[2i + 1]) + beta^2 roll[i]"""
    half = len(vec) // 2
    lh = half.bit_length() - 1
    bb = beta * beta
    return [pv.fold_row(i, lh, beta, vec[2 * i], vec[2 * i + 1]) + (bb * roll[i] if roll is not None else E(0))
            for i in range(half)]


def idft_coset(vals, log_h):
    """coefficients of the polynomial whose values at GENERATOR * w^rev(i) are vals[i] (O(N^2), small N only)"""
    n = 1 << log_h
    winv, ginv, ninv = pv.inv(pv.two_adic_generator(log_h)), pv.inv(G), pv.inv(n)
    nat = [vals[pv.rev_bits(j, log_h)] for j in range(n)]  # value at GENERATOR * w^j
    coeffs = []
    for k in range(n):
        acc = E(0)
        for j in range(n):
            acc = acc + nat[j] * pow(winv, j * k, P)
        coeffs.append(acc * (ninv * pow(ginv, k, P) % P))
    return coeffs


def test_reference_self_check():
    """CPU check of the reference: a reduced input built from the right opened values is the evaluation of a polynomial of
    degree below the trace height (a wrong value makes it full degree), and folding the evaluations of p(x) = pe(x^2) +
    x po(x^2) gives pe(y) + beta po(y) on the folded domain."""
    rnd = random.Random(1)
    log_n, lb = 3, 2
    m = Mat(rand_coeffs(rnd, 1 << log_n, 3), log_n, lb, [rand_ext(rnd), rand_ext(rnd)])
    alpha = rand_ext(rnd)
    N = 1 << m.log_h
    vec = reduce_ref([[m]], alpha, lambda lh: range(1 << lh))[m.log_h]
    coeffs = idft_coset([vec[i] for i in range(N)], m.log_h)
    assert all(c.is_zero() for c in coeffs[1 << log_n:])
    assert not all(c.is_zero() for c in coeffs[:1 << log_n])
    bad = Mat(m.F, log_n, lb, m.points)
    good_values = m.values()
    bad.values = lambda: [good_values[0][:1] + [good_values[0][1] + 1] + good_values[0][2:], good_values[1]]
    bvec = reduce_ref([[bad]], alpha, lambda lh: range(1 << lh))[m.log_h]
    assert not idft_coset([bvec[i] for i in range(N)], m.log_h)[-1].is_zero()
    # fold
    lh = 4
    pe, po = [rand_ext(rnd) for _ in range(8)], [rand_ext(rnd) for _ in range(8)]
    ev = lambda cs, x: sum((c * pow(x, k, P) for k, c in enumerate(cs)), E(0))
    g = pv.two_adic_generator(lh + 1)
    vals = []
    for j in range(2 << lh):
        x = pow(g, pv.rev_bits(j, lh + 1), P)
        vals.append(ev(pe, x * x % P) + ev(po, x * x % P) * x)
    beta = rand_ext(rnd)
    roll = [rand_ext(rnd) for _ in range(1 << lh)]
    got = fold_ref(vals, beta, roll)
    for i in range(1 << lh):
        y = pow(pv.two_adic_generator(lh), pv.rev_bits(i, lh), P)
        assert got[i] == ev(pe, y) + beta * ev(po, y) + beta * beta * roll[i]


# ---- the device --------------------------------------------------------------------------------------------------------
def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _u64p(a):
    from multi_stark_b200._ffi import c_u64p
    return a.ctypes.data_as(c_u64p)


class Opening:
    """msgpu_open over rounds of committed Mats (one ProverData per round)."""

    def __init__(self, ctx, pds, rounds, log_blowup, shard=None):
        from multi_stark_b200._ffi import check
        self.ctx, self.L, self.check, self.rounds = ctx, ctx.L, check, rounds
        npts = np.array([len(m.points) for r in rounds for m in r] or [0], dtype=np.uint64)
        pts = np.array([v for r in rounds for m in r for z in m.points for v in (z.a, z.b)] or [0], dtype=np.uint64)
        arr = (C.c_void_p * len(pds))(*[pd.h for pd in pds])
        self.h = C.c_void_p()
        nv = C.c_uint64()
        if shard is None:
            check(self.L.msgpu_open_begin(ctx.h, len(pds), arr, _u64p(npts), _u64p(pts), log_blowup, C.byref(self.h), C.byref(nv)))
        else:
            index, n_shards, owner = shard
            modes = np.ones(len(pds), dtype=np.uint32)
            ns = C.c_uint64()
            check(self.L.msgpu_open_begin_shard(ctx.h, len(pds), arr, _ptr(modes), index, n_shards, owner, _ptr(npts), _ptr(pts),
                                                log_blowup, C.byref(self.h), C.byref(nv), C.byref(ns)))
            self.n_sums = int(ns.value)
        self.n_values = int(nv.value)
        assert self.n_values == sum(len(m.points) * m.w for r in rounds for m in r)

    def values(self):
        raw = np.zeros(2 * max(self.n_values, 1), dtype=np.uint64)
        self.check(self.L.msgpu_open_values(self.h, _ptr(raw)))
        out, o = [], 0
        for r in self.rounds:
            for m in r:
                mv = []
                for _ in m.points:
                    mv.append([E(int(raw[o + 2 * c]), int(raw[o + 2 * c + 1])) for c in range(m.w)])
                    o += 2 * m.w
                out.append(mv)
        return out

    def reduce(self, alpha):
        a = np.array([alpha.a, alpha.b], dtype=np.uint64)
        n, lmh = C.c_uint64(), C.c_uint32()
        self.check(self.L.msgpu_open_reduce(self.h, _ptr(a), C.byref(n), C.byref(lmh)))
        return int(n.value), int(lmh.value)

    def read_input(self, k):
        ln = C.c_uint64()
        self.check(self.L.msgpu_open_read_input(self.h, k, None, C.byref(ln)))
        raw = np.zeros(2 * int(ln.value), dtype=np.uint64)
        self.check(self.L.msgpu_open_read_input(self.h, k, _ptr(raw), C.byref(ln)))
        return raw

    def commit_round(self):
        root = np.zeros(32, dtype=np.uint8)
        self.check(self.L.msgpu_fri_commit_round(self.h, _ptr(root)))
        return bytes(root)

    def fold(self, beta):
        self.check(self.L.msgpu_fri_fold(self.h, _ptr(np.array([beta.a, beta.b], dtype=np.uint64))))

    def current(self):
        ln = C.c_uint64()
        self.check(self.L.msgpu_fri_current_len(self.h, C.byref(ln)))
        raw = np.zeros(2 * int(ln.value), dtype=np.uint64)
        self.check(self.L.msgpu_fri_read_current(self.h, _ptr(raw)))
        return as_ext(raw)

    def commit_phase(self, buf, stop_len, max_rounds, input_len=None):
        b = np.frombuffer(bytes(buf), dtype=np.uint8).copy() if len(buf) else np.zeros(1, dtype=np.uint8)
        roots = np.zeros((max(max_rounds, 1), 32), dtype=np.uint8)
        betas = np.zeros(2 * max(max_rounds, 1), dtype=np.uint64)
        n = C.c_uint64()
        rc = self.L.msgpu_fri_commit_phase(self.h, _ptr(b), len(buf) if input_len is None else input_len, stop_len, max_rounds,
                                           _ptr(roots), _ptr(betas), C.byref(n))
        if rc:
            return rc, None, None
        k = int(n.value)
        return 0, [bytes(r) for r in roots[:k]], [E(int(betas[2 * i]), int(betas[2 * i + 1])) for i in range(k)]

    def free(self):
        if self.h:
            self.L.msgpu_open_free(self.h)
            self.h = None


def as_ext(raw):
    return [E(int(raw[2 * i]), int(raw[2 * i + 1])) for i in range(len(raw) // 2)]


def commit_rounds(ms, ctx, rounds, lb):
    pcs = ms.GpuPcs(ctx, lb)
    return [pcs.commit([m.natural() for m in r])[1] for r in rounds]


def open_rounds(ms, ctx, rounds, lb):
    pds = commit_rounds(ms, ctx, rounds, lb)
    return Opening(ctx, pds, rounds, lb), pds


def check_values(op, rounds):
    got = op.values()
    want = [m.values() for r in rounds for m in r]
    for k, (g, w) in enumerate(zip(got, want)):
        assert g == w, "opened values of matrix %d" % k


def check_inputs(op, rounds, alpha, sample=None):
    """reduce, then compare every input (or the rows sample(log_h) of it) with the reference"""
    heights = sorted({m.log_h for r in rounds for m in r}, reverse=True)
    n, lmh = op.reduce(alpha)
    assert (n, lmh) == (len(heights), heights[0])
    rows_of = (lambda lh: range(1 << lh)) if sample is None else sample
    want = reduce_ref(rounds, alpha, rows_of)
    for k, lh in enumerate(heights):
        raw = op.read_input(k)
        assert len(raw) == 2 << lh
        for i, v in want[lh].items():
            assert E(int(raw[2 * i]), int(raw[2 * i + 1])) == v, "input %d (height 2^%d), row %d" % (k, lh, i)


def free_all(op, pds):
    op.free()
    for pd in pds:
        pd.free()


def odd_tile_widths():
    return [wc for wc in range(1, 257) if min(256, max(8, 4096 // wc)) * wc % 2]


# ---- opened values -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_values_width_sweep(gpu):
    """Every width 1..260 and 275, 385, 495, 700, 2625: every chunk width of k_bary_partial, among them the 67 whose
    tile_rows * wc is odd, and the strided path of matrices wider than 256 columns. The columns of width w are the first
    w of one pool, so the reference evaluates each polynomial once."""
    ms, ctx = gpu
    assert len(odd_tile_widths()) == 67
    rnd = random.Random(2)
    log_n, lb = 7, 1
    pool = rand_coeffs(rnd, 4, 2625)
    z = [rand_ext(rnd), rand_ext(rnd)]
    nat = Mat(pool, log_n, lb).natural()
    ys = [eval_at(pool, zz) for zz in z]
    pcs = ms.GpuPcs(ctx, lb)
    for w in list(range(1, 261)) + [275, 385, 495, 700, 2625]:
        m = Mat([row[:w] for row in pool], log_n, lb, z)
        _, pd = pcs.commit([nat[:, :w]])
        op = Opening(ctx, [pd], [[m]], lb)
        got = op.values()[0]
        assert got == [y[:w] for y in ys], "width %d" % w
        free_all(op, [pd])


@pytest.mark.gpu
@pytest.mark.parametrize("npts", [1, 2, 3, 4, 5, 8, 9])
def test_points_per_matrix(gpu, npts):
    """k_bary_partial<1..4>, points taken in groups of four, and the alpha offsets of the groups in k_reduce_openings."""
    ms, ctx = gpu
    rnd = random.Random(10 + npts)
    lb = 1
    rounds = [[Mat(rand_coeffs(rnd, 32, 19), 5, lb, [rand_ext(rnd) for _ in range(npts)]),
               Mat(rand_coeffs(rnd, 8, 6), 3, lb, [rand_ext(rnd) for _ in range(npts)])]]
    op, pds = open_rounds(ms, ctx, rounds, lb)
    check_values(op, rounds)
    check_inputs(op, rounds, rand_ext(rnd))
    free_all(op, pds)


@pytest.mark.gpu
def test_shared_point_and_base_field_point(gpu):
    """One point on matrices of three heights (the inverse denominators of the tallest serve the others), a second point
    shared by two of them, and a base-field point off the coset."""
    ms, ctx = gpu
    rnd = random.Random(3)
    lb = 2
    z, z2, zb = rand_ext(rnd), rand_ext(rnd), E(rnd.randrange(P), 0)
    rounds = [[Mat(rand_coeffs(rnd, 16, 5), 4, lb, [z]), Mat(rand_coeffs(rnd, 64, 3), 6, lb, [z, z2]),
               Mat(rand_coeffs(rnd, 8, 4), 3, lb, [z2, zb, z])]]
    op, pds = open_rounds(ms, ctx, rounds, lb)
    check_values(op, rounds)
    check_inputs(op, rounds, rand_ext(rnd))
    free_all(op, pds)


@pytest.mark.gpu
def test_multiple_rounds(gpu):
    """Three rounds; one matrix, alone at its height, has no points and still gets a (zero) input."""
    ms, ctx = gpu
    rnd = random.Random(4)
    lb = 1
    z, zn = rand_ext(rnd), rand_ext(rnd)
    rounds = [[Mat(rand_coeffs(rnd, 32, 7), 5, lb, [z, zn]), Mat(rand_coeffs(rnd, 4, 2), 2, lb, [z])],
              [Mat(rand_coeffs(rnd, 8, 3), 3, lb, [])],
              [Mat(rand_coeffs(rnd, 32, 4), 5, lb, [z]), Mat(rand_coeffs(rnd, 4, 9), 2, lb, [z, zn])]]
    op, pds = open_rounds(ms, ctx, rounds, lb)
    check_values(op, rounds)
    check_inputs(op, rounds, rand_ext(rnd))
    assert all(v == 0 for v in op.read_input(1))  # heights 2^6, 2^4 (no points), 2^3
    free_all(op, pds)


@pytest.mark.gpu
@pytest.mark.parametrize("lb", [1, 2, 3])
def test_smallest_matrix(gpu, lb):
    """Height 2^log_blowup: the low coset is one row, and the opened value is that row at any point."""
    ms, ctx = gpu
    rnd = random.Random(20 + lb)
    rounds = [[Mat(rand_coeffs(rnd, 1, 5), 0, lb, [rand_ext(rnd), rand_ext(rnd), E(rnd.randrange(P), 0)])]]
    op, pds = open_rounds(ms, ctx, rounds, lb)
    check_values(op, rounds)
    assert op.values()[0][0] == [E(v) for v in rounds[0][0].F[0]]
    check_inputs(op, rounds, rand_ext(rnd))
    free_all(op, pds)


def sample_rows(lh, tile_rows, rnd, k=24):
    n = 1 << lh
    rows = {0, 1, n - 1, n - 2, n // 2 - 1, n // 2}
    for t in (tile_rows, 2 * tile_rows, 215, 256, 888 * 256):
        rows |= {t - 1, t, t + 1}
    rows |= {rnd.randrange(n) for _ in range(k)}
    return sorted(r for r in rows if 0 <= r < n)


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,w,lb", [(18, 4, 1), (16, 19, 2)])
def test_large(gpu, log_n, w, lb):
    """Heights where k_bary_partial loops over its grid (2^18 rows of 4 columns need 1024 tiles of 256 rows, more than its
    6 CTAs per SM) and k_bary_sum adds the most partials; the reduced input is checked on a sample of rows."""
    ms, ctx = gpu
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if w == 4:
        assert (1 << log_n) // 256 > 6 * sms
    rnd = random.Random(log_n)
    rounds = [[Mat(rand_coeffs(rnd, 3, w), log_n, lb, [rand_ext(rnd), rand_ext(rnd)])]]
    op, pds = open_rounds(ms, ctx, rounds, lb)
    check_values(op, rounds)
    srnd = random.Random(5)
    check_inputs(op, rounds, rand_ext(rnd), sample=lambda lh: sample_rows(lh, 128, srnd))
    free_all(op, pds)


# ---- reduced inputs ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("w", [1, 2, 19, 63, 64, 65, 700, 2625, 4266])
def test_reduce_widths(gpu, w):
    """Odd widths take the contiguous tile copy, even ones the strided one (pitch w | 1); 63 .. 4266 columns shrink
    tile_rows from 128 to 4. 4266 is the widest matrix k_reduce_openings takes."""
    ms, ctx = gpu
    rnd = random.Random(30 + w)
    lb = 1
    log_n = 6 if w < 700 else 3
    rounds = [[Mat(rand_coeffs(rnd, 4, w), log_n, lb, [rand_ext(rnd), rand_ext(rnd)])]]
    op, pds = open_rounds(ms, ctx, rounds, lb)
    check_values(op, rounds)
    check_inputs(op, rounds, rand_ext(rnd))
    free_all(op, pds)


@pytest.mark.gpu
def test_reduce_rejects_4267_columns_and_context_survives(gpu):
    from multi_stark_b200._ffi import MsgpuError
    ms, ctx = gpu
    rnd = random.Random(6)
    lb = 1
    rounds = [[Mat(rand_coeffs(rnd, 2, 4267), 2, lb, [rand_ext(rnd)])]]
    op, pds = open_rounds(ms, ctx, rounds, lb)
    with pytest.raises(MsgpuError, match="4266 columns"):
        op.reduce(rand_ext(rnd))
    free_all(op, pds)
    rounds = [[Mat(rand_coeffs(rnd, 16, 21), 4, lb, [rand_ext(rnd), rand_ext(rnd)])]]
    op, pds = open_rounds(ms, ctx, rounds, lb)
    check_values(op, rounds)
    check_inputs(op, rounds, rand_ext(rnd))
    free_all(op, pds)


@pytest.mark.gpu
def test_point_on_the_coset_is_refused(gpu):
    """z = GENERATOR * w_N^j would make 1 / (z - x) undefined for one row and zero for every row of its inversion batch."""
    from multi_stark_b200._ffi import MsgpuError
    ms, ctx = gpu
    rnd = random.Random(7)
    lb = 1
    low = Mat(rand_coeffs(rnd, 4, 3), 2, lb, [])
    tall = Mat(rand_coeffs(rnd, 16, 3), 4, lb, [])
    pds = commit_rounds(ms, ctx, [[low, tall]], lb)
    for j in (0, 3, 31):
        tall.points = [E(lde_x(j, tall.log_h))]
        with pytest.raises(MsgpuError, match="coset"):
            Opening(ctx, pds, [[low, tall]], lb)
    # a point of the tall coset that the short matrix does not have is only refused where the tall matrix opens it
    tall.points = []
    low.points = [E(lde_x(16, tall.log_h))]
    assert pow(low.points[0].a * pv.inv(G), 1 << low.log_h, P) != 1
    op = Opening(ctx, pds, [[low, tall]], lb)
    check_values(op, [[low, tall]])
    op.free()
    for pd in pds:
        pd.free()


# ---- the commit phase --------------------------------------------------------------------------------------------------
def check_layer(op, k, vec):
    """root and openings of commit-phase layer k against the Python Merkle tree over len/2 rows of 4 base columns"""
    rows = np.array([[v.a, v.b, w.a, w.b] for v, w in zip(vec[0::2], vec[1::2])], dtype=np.uint64)
    layers = py_mmcs_commit([rows])
    pd = op.L.msgpu_fri_layer_pdata(op.h, k)  # borrowed: the opening frees it
    assert pd
    n = len(rows)
    idx = np.array(sorted({0, n - 1, n // 2, (n * 5) // 7}), dtype=np.uint64)
    depth = n.bit_length() - 1
    opened = np.zeros((len(idx), 4), dtype=np.uint64)
    proofs = np.zeros((len(idx), max(depth, 1), 32), dtype=np.uint8)
    op.check(op.L.msgpu_open_batch(op.ctx.h, C.c_void_p(pd), _ptr(idx), len(idx), _ptr(opened), _ptr(proofs)))
    for q, i in enumerate(int(v) for v in idx):
        assert np.array_equal(opened[q], rows[i])
        j = i
        for l in range(depth):
            assert bytes(proofs[q, l]) == layers[l][j ^ 1], "layer %d, index %d, level %d" % (k, i, l)
            j >>= 1
    return layers[-1][0]


@pytest.mark.gpu
@pytest.mark.parametrize("roll", [False, True])
@pytest.mark.parametrize("log_len", list(range(1, 15)))
def test_commit_phase_host_beta(gpu, log_len, roll):
    """fri_commit_round / fri_fold from 2^log_len down to one element: k_fri_fold while the folded length is above 4096,
    k_fri_fold_commit from 4096 down to 2, k_fri_fold for the last fold; with roll, inputs of half and an eighth of the
    length are rolled in (an eighth in a fused fold when the lengths allow)."""
    ms, ctx = gpu
    rnd = random.Random(100 * log_len + roll)
    lb = 1
    heights = [log_len] + ([h for h in (log_len - 1, log_len - 3) if h >= lb] if roll else [])
    rounds = [[Mat(rand_coeffs(rnd, min(2, 1 << (h - lb)), 2), h - lb, lb, [rand_ext(rnd)]) for h in heights]]
    op, pds = open_rounds(ms, ctx, rounds, lb)
    n, _ = op.reduce(rand_ext(rnd))
    inputs = [as_ext(op.read_input(k)) for k in range(n)]
    vec, nxt = inputs[0], 1
    k = 0
    while len(vec) > 1:
        root = op.commit_round()
        assert root == check_layer(op, k, vec), "root of layer %d" % k
        beta = rand_ext(rnd)
        op.fold(beta)
        roll_in = None
        if nxt < len(inputs) and len(inputs[nxt]) == len(vec) // 2:
            roll_in, nxt = inputs[nxt], nxt + 1
        vec = fold_ref(vec, beta, roll_in)
        assert op.current() == vec, "fold %d" % k
        k += 1
    assert nxt == len(inputs) and k == log_len
    assert int(op.L.msgpu_fri_num_layers(op.h)) == log_len
    free_all(op, pds)


def transcript_opening(ms, ctx, seed):
    rnd = random.Random(seed)
    lb = 1
    rounds = [[Mat(rand_coeffs(rnd, 2, 3), 9, lb, [rand_ext(rnd)]), Mat(rand_coeffs(rnd, 2, 2), 6, lb, [rand_ext(rnd)])]]
    op, pds = open_rounds(ms, ctx, rounds, lb)
    op.reduce(rand_ext(rnd))
    return op, pds


@pytest.mark.gpu
@pytest.mark.parametrize("stop_len", [1, 2, 8])
@pytest.mark.parametrize("input_len", [1, 31, 32, 33, 95, 96, 97, 960])
def test_device_transcript(gpu, input_len, stop_len):
    """msgpu_fri_commit_phase: prefix + root on both sides of every 64-byte BLAKE3 block edge up to 992 bytes; betas equal
    PyChallenger's, roots and the last vector equal the host-beta path on an identical opening."""
    ms, ctx = gpu
    buf = bytes(random.Random(input_len).randrange(256) for _ in range(input_len))
    op, pds = transcript_opening(ms, ctx, 8)
    rc, roots, betas = op.commit_phase(buf, stop_len, 16)
    assert rc == 0 and len(roots) == 10 - (stop_len.bit_length() - 1)
    final = op.current()
    ch = pv.PyChallenger(buf)
    for r, b in zip(roots, betas):
        ch.observe(r)
        assert ch.sample_ext() == b
    op2, pds2 = transcript_opening(ms, ctx, 8)
    for r, b in zip(roots, betas):
        assert op2.commit_round() == r
        op2.fold(b)
    assert op2.current() == final and len(final) == stop_len
    free_all(op, pds)
    free_all(op2, pds2)


@pytest.mark.gpu
def test_device_transcript_zero_rounds_and_refusals(gpu):
    ms, ctx = gpu
    op, pds = transcript_opening(ms, ctx, 9)
    for stop in (1024, 2048):
        rc, roots, betas = op.commit_phase(b"x" * 32, stop, 0)
        assert rc == 0 and roots == [] and betas == []
    for buf, n in ((b"x", 0), (b"x" * 961, None)):
        assert op.commit_phase(buf, 1, 16, input_len=n)[0] == -1  # MSGPU_ERR_INVALID
    assert op.commit_phase(b"x" * 32, 1, 9)[0] == -1  # 10 rounds do not fit
    rc, roots, _ = op.commit_phase(b"x" * 32, 1, 10)
    assert rc == 0 and len(roots) == 10
    free_all(op, pds)


# ---- a row-sharded opening on one GPU ----------------------------------------------------------------------------------
@pytest.mark.gpu
def test_sharded_opening_matches_unsharded(gpu):
    """Two row shards of a 19-column matrix (msgpu_open_begin_shard): the summed barycentric sums give the unsharded values,
    and the non-owner's reduced rows added into the owner's give the unsharded input."""
    ms, ctx = gpu
    from multi_stark_b200._ffi import check
    rnd = random.Random(11)
    lb = 1
    m = Mat(rand_coeffs(rnd, 64, 19), 6, lb, [rand_ext(rnd), rand_ext(rnd)])
    alpha = rand_ext(rnd)
    op, pds = open_rounds(ms, ctx, [[m]], lb)
    want_values = op.values()
    op.reduce(alpha)
    want_input = op.read_input(0)
    lde = pds[0].read_rows(0)
    free_all(op, pds)
    N = len(lde)
    pcs = ms.GpuPcs(ctx, lb)
    bufs, spds, ops = [], [], []
    for s in range(2):
        half = np.ascontiguousarray(lde[s * N // 2:(s + 1) * N // 2])
        bufs.append(ctx.upload(half))
        spds.append(pcs.commit_ldes([(bufs[-1], N // 2, m.w)])[1])
        ops.append(Opening(ctx, [spds[-1]], [[m]], lb, shard=(s, 2, 1 if s == 0 else 0)))
    sums = []
    for o in ops:
        raw = np.zeros(max(o.n_sums, 1), dtype=np.uint64)
        check(o.L.msgpu_open_sums(o.h, _ptr(raw)))
        sums.append([int(v) for v in raw[:o.n_sums]])
    total = np.array([(a + b) % P for a, b in zip(*sums)], dtype=np.uint64)
    for s, o in enumerate(ops):
        check(o.L.msgpu_open_finish_values(o.h, _ptr(total)))
        assert o.values() == want_values
        assert o.reduce(alpha) == (1, m.log_h - s)  # the other rank keeps only the rows it holds
    dst, src = C.c_void_p(), C.c_void_p()
    ln = C.c_uint64()
    check(ctx.L.msgpu_open_input_dev(ops[0].h, 0, C.byref(dst), C.byref(ln)))
    assert int(ln.value) == N
    check(ctx.L.msgpu_open_input_dev(ops[1].h, 0, C.byref(src), C.byref(ln)))
    assert int(ln.value) == N // 2
    check(ctx.L.msgpu_ext_add_dev(ctx.h, C.c_void_p(dst.value + (N // 2) * 16), src, N // 2))
    assert np.array_equal(ops[0].read_input(0), want_input)
    for o, pd, b in zip(ops, spds, bufs):
        o.free()
        pd.free()
        ctx.free(b)


# ---- calls out of order ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_calls_out_of_order_are_refused(gpu):
    from multi_stark_b200._ffi import MsgpuError
    ms, ctx = gpu
    rnd = random.Random(12)
    lb = 1
    rounds = [[Mat(rand_coeffs(rnd, 8, 3), 3, lb, [rand_ext(rnd)]), Mat(rand_coeffs(rnd, 4, 2), 2, lb, [rand_ext(rnd)])]]
    op, pds = open_rounds(ms, ctx, rounds, lb)
    alpha = rand_ext(rnd)
    op.reduce(alpha)
    with pytest.raises(MsgpuError, match="already reduced"):
        op.reduce(alpha)
    with pytest.raises(MsgpuError, match="commit the current vector first"):
        op.fold(rand_ext(rnd))
    op.commit_round()
    op.fold(rand_ext(rnd))  # 16 -> 8 rolls in the input of height 8
    with pytest.raises(MsgpuError, match="already consumed"):
        op.read_input(1)
    free_all(op, pds)


# ---- whole proofs of wide circuits -------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("w", [19, 131])
def test_wide_circuit_proof(gpu, oracle, w):
    """A circuit with w main columns (chunk widths with an odd tile in k_bary_partial) proves through msh_prove with the
    oracle's bytes, and the restated verifier accepts the proof."""
    ms, ctx = gpu
    Ex = pv.Expr
    m = Ex.main
    cons = [m(2) - m(0) * m(1)] + [m(j) - m(j - 1) - Ex.const(j) for j in range(3, w)]
    circ = pv.Circuit(w, [], cons)
    n = 1 << 6
    rng = np.random.default_rng(w)
    t = np.zeros((n, w), dtype=object)
    t[:, 0] = [int(v) for v in rng.integers(0, P, size=n, dtype=np.uint64)]
    t[:, 1] = [int(v) for v in rng.integers(0, P, size=n, dtype=np.uint64)]
    t[:, 2] = t[:, 0] * t[:, 1] % P
    for j in range(3, w):
        t[:, j] = (t[:, j - 1] + j) % P
    trace = t.astype(np.uint64)
    kw = dict(log_blowup=1, num_queries=20)
    g = pv.graph_dict(circ)
    system = ms.System.from_graphs([g], **kw)
    pr = ms.Prover(ctx, system)
    proof = pr.prove([trace], [])
    S = orc.OracleSystem(oracle, None, graphs=[g], **kw)
    want, _ = S.prove([trace], [])
    assert proof == want
    prm = dict(kw, log_final_poly_len=0, max_log_arity=1, commit_pow_bits=0, query_pow_bits=0)
    assert pv.verify([circ], prm, None, [], _proof.parse(proof)) == "Ok"
    pr.close()
    S.close()
    system.close()
