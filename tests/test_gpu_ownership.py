"""Device memory ownership of libmsgpu's handles (multi_stark_b200/csrc). Every refused call leaves the context's arena
exactly as it found it (msgpu_arena_in_use), buffers a refused call was asked to adopt stay the caller's, and each handle's
whole lifecycle ends with nothing left behind. The context keeps working after the refusals."""
import contextlib
import ctypes as C
import random

import numpy as np
import pytest

from tests import _oracle as orc
from tests import _pyverifier as pv
from tests.test_gpu_arena import _upload_begin
from tests.test_gpu_constraints import ext, fingerprint, lookup_rows, neg, rnd_ext
from tests.test_gpu_open import E, Mat, Opening, _ptr, commit_rounds, free_all, lde_x, open_rounds, rand_coeffs, rand_ext, \
    transcript_opening
from tests.test_oracle_hash import py_mmcs_commit

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    import multi_stark_b200 as ms
    ctx = ms.GpuContext(0)
    yield ms, ctx
    ctx.close()


def in_use(ctx):
    n = C.c_uint64()
    assert ctx.L.msgpu_arena_in_use(ctx.h, C.byref(n)) == 0
    return int(n.value)


@contextlib.contextmanager
def arena_unchanged(ctx):
    before = in_use(ctx)
    yield
    assert in_use(ctx) == before


# ---- refused calls ----------------------------------------------------------------------------------------------------------
def test_reduce_refusing_mixed_shard_rows_frees_its_vectors(gpu):
    """fri_owner = 0 with a whole (mode 0) and a row-sharded (mode 1) round of one global height: the reduced-openings vector
    of that height is allocated for the first matrix, then the second is refused."""
    ms, ctx = gpu
    from multi_stark_b200._ffi import check
    rnd = random.Random(41)
    lb = 1
    whole = Mat(rand_coeffs(rnd, 8, 3), 3, lb, [rand_ext(rnd)])   # LDE height 16, all rows here
    shard = Mat(rand_coeffs(rnd, 4, 2), 2, lb, [rand_ext(rnd)])   # 8 rows: shard 0 of 2 of a height-16 matrix
    start = in_use(ctx)
    pds = commit_rounds(ms, ctx, [[whole], [shard]], lb)
    npts = np.array([1, 1], dtype=np.uint64)
    pts = np.array([v for m in (whole, shard) for z in m.points for v in (z.a, z.b)], dtype=np.uint64)
    modes = np.array([0, 1], dtype=np.uint32)
    arr = (C.c_void_p * 2)(*[pd.h for pd in pds])
    op, nv, ns = C.c_void_p(), C.c_uint64(), C.c_uint64()
    check(ctx.L.msgpu_open_begin_shard(ctx.h, 2, arr, _ptr(modes), 0, 2, 0, _ptr(npts), _ptr(pts), lb, C.byref(op), C.byref(nv),
                                       C.byref(ns)))
    alpha = np.array([5, 7], dtype=np.uint64)
    n, lmh = C.c_uint64(), C.c_uint32()
    with arena_unchanged(ctx):
        assert ctx.L.msgpu_open_reduce(op, _ptr(alpha), C.byref(n), C.byref(lmh)) != 0
        assert b"cover the same rows" in ctx.L.msgpu_last_error()
    ctx.L.msgpu_open_free(op)
    for pd in pds:
        pd.free()
    assert in_use(ctx) == start


def test_reduce_refusing_4267_columns(gpu):
    ms, ctx = gpu
    from multi_stark_b200._ffi import MsgpuError
    rnd = random.Random(6)
    rounds = [[Mat(rand_coeffs(rnd, 2, 4267), 2, 1, [rand_ext(rnd)])]]
    op, pds = open_rounds(ms, ctx, rounds, 1)
    with arena_unchanged(ctx):
        with pytest.raises(MsgpuError, match="4266 columns"):
            op.reduce(rand_ext(rnd))
    free_all(op, pds)


def test_open_refusing_a_point_on_the_coset(gpu):
    ms, ctx = gpu
    from multi_stark_b200._ffi import MsgpuError
    rnd = random.Random(7)
    tall = Mat(rand_coeffs(rnd, 16, 3), 4, 1, [])
    pds = commit_rounds(ms, ctx, [[tall]], 1)
    tall.points = [rand_ext(rnd), E(lde_x(3, tall.log_h))]
    with arena_unchanged(ctx):
        with pytest.raises(MsgpuError, match="coset"):
            Opening(ctx, pds, [[tall]], 1)
    for pd in pds:
        pd.free()


def test_commit_upload_refusing_non_canonical_values(gpu):
    ms, ctx = gpu
    bad = np.zeros((64, 2), dtype=np.uint64)
    bad[17, 1] = ms.P
    with arena_unchanged(ctx):
        rc, up = _upload_begin(ms, ctx, [np.ones((64, 3), dtype=np.uint64), bad])
        assert rc == 0
        kept = (C.c_void_p * 2)()
        pd, root = C.c_void_p(), np.zeros(32, dtype=np.uint8)
        assert ctx.L.msgpu_commit_upload(up, 1, 1, kept, 0, C.byref(pd), _ptr(root)) != 0
        assert b"canonical" in ctx.L.msgpu_last_error()


def test_stage2_and_claims_refusing_a_zero_message(gpu):
    ms, ctx = gpu
    from multi_stark_b200._ffi import MsgpuError
    circ = pv.Circuit(4, [pv.push(pv.Expr.main(k), [pv.Expr.main(k + 1), pv.Expr.main(0) * pv.Expr.main(3)]) for k in range(3)], [])
    rng = np.random.default_rng(5)
    main = orc.rand_matrix(rng, 256, 4)
    gamma = rnd_ext(rng)
    _, args = lookup_rows(circ.graph, main)[33][2]
    beta = neg(fingerprint(ext(gamma), args))
    system = ms.System.from_graphs([pv.graph_dict(circ)])
    prog = ms.Program(ctx, system, 0)
    d_main = ctx.upload(main)
    d_out = ctx.malloc(256 * prog.info["stage2_width"] * 8)
    ls = np.zeros(2, dtype=np.uint64)
    with arena_unchanged(ctx):
        assert ctx.L.msgpu_stage2_trace(ctx.h, prog.h, None, C.c_void_p(d_main), 256, _ptr(beta), _ptr(gamma), C.c_void_p(d_out),
                                        _ptr(ls)) != 0
        assert b"logUp message" in ctx.L.msgpu_last_error()
    for p in (d_main, d_out):
        ctx.free(p)
    prog.free()
    system.close()
    claims = orc.rand_matrix(rng, 100, 4)
    beta = neg(fingerprint(ext(gamma), [int(v) for v in claims[52]]))
    with arena_unchanged(ctx):
        with pytest.raises(MsgpuError, match="logUp message"):
            ms.claims_accumulator(ctx, claims, beta, gamma)


def test_fri_commit_phase_refusals(gpu):
    ms, ctx = gpu
    op, pds = transcript_opening(ms, ctx, 9)
    with arena_unchanged(ctx):
        for buf, n in ((b"x", 0), (b"x" * 961, None)):
            assert op.commit_phase(buf, 1, 16, input_len=n)[0] == -1
        assert op.commit_phase(b"x" * 32, 1, 9)[0] == -1  # 10 rounds do not fit
        assert op.commit_phase(b"x" * 32, 3, 16)[0] == -1  # stop length not a power of two
    free_all(op, pds)


@pytest.mark.parametrize("entry", ["commit_local_dev", "commit_ldes_dev"])
def test_refused_adopting_commit_leaves_the_buffers_to_the_caller(gpu, entry):
    """inputs_are_ldes = 1 / take_ownership = 1 adopt the buffers only when the call succeeds. Here the height-64 class is hashed
    and the row of the height-1 matrix is refused as too wide: both buffers still free exactly once with msgpu_free."""
    ms, ctx = gpu
    from multi_stark_b200._ffi import MsgpuError
    good = ctx.upload(np.arange(128, dtype=np.uint64).reshape(64, 2))
    wide = ctx.malloc(64)
    ptrs = (C.c_void_p * 2)(good, wide)
    hs = (C.c_uint64 * 2)(64, 1)
    ws = (C.c_uint64 * 2)(2, 1 << 29)
    pd, root = C.c_void_p(), np.zeros(32, dtype=np.uint8)
    with arena_unchanged(ctx):
        if entry == "commit_local_dev":
            rc = ctx.L.msgpu_commit_local_dev(ctx.h, ptrs, hs, ws, 2, 1, 1, C.byref(pd))
        else:
            rc = ctx.L.msgpu_commit_ldes_dev(ctx.h, ptrs, hs, ws, 2, 1, C.byref(pd), _ptr(root))
        assert rc != 0
        assert b"row too wide" in ctx.L.msgpu_last_error()
    for p in (good, wide):
        ctx.free(p)
        with pytest.raises(MsgpuError):
            ctx.free(p)


# ---- whole lifecycles -------------------------------------------------------------------------------------------------------
def test_commit_open_reduce_commit_phase_then_free(gpu):
    ms, ctx = gpu
    with arena_unchanged(ctx):
        op, pds = transcript_opening(ms, ctx, 8)
        rc, roots, _ = op.commit_phase(b"y" * 40, 1, 16)
        assert rc == 0 and len(roots) == 10
        free_all(op, pds)


def test_program_create_and_free(gpu):
    ms, ctx = gpu
    circ = pv.Circuit(4, [pv.push(pv.Expr.main(0), [pv.Expr.main(1)])], [])
    system = ms.System.from_graphs([pv.graph_dict(circ)])
    with arena_unchanged(ctx):
        ms.Program(ctx, system, 0).free()
    system.close()


def test_claims_prefetch_and_free(gpu):
    ms, ctx = gpu
    claims = orc.rand_matrix(np.random.default_rng(2), 300, 3)
    with arena_unchanged(ctx):
        cl = C.c_void_p()
        assert ctx.L.msgpu_claims_prefetch(ctx.h, _ptr(claims), 300, 3, C.byref(cl)) == 0
        ctx.L.msgpu_claims_free(cl)


def test_upload_begin_and_free(gpu):
    ms, ctx = gpu
    mats = [np.ones((256, 3), dtype=np.uint64), np.ones((64, 5), dtype=np.uint64)]
    with arena_unchanged(ctx):
        rc, up = _upload_begin(ms, ctx, mats)
        assert rc == 0
        ctx.L.msgpu_upload_free(up)


def test_context_still_commits_after_the_refusals(gpu):
    ms, ctx = gpu
    rows = orc.rand_matrix(np.random.default_rng(9), 64, 5)
    with arena_unchanged(ctx):
        root, pd = ms.GpuMmcs(ctx).commit([rows])
        assert bytes(root) == py_mmcs_commit([rows])[-1][0]
        pd.free()
