"""The commitment side of libmsgpu (ntt.cu, merkle.cu, mmcs.cu) against the exact CPU reference of tests/_commit_ref.py,
shape by shape, comparing whole outputs bit for bit.

NTT: a Python mirror of `plan_passes` and of the LDE's pass structure names the kernel instantiations each shape runs. The
CPU test `test_shapes_reach_every_instantiation` checks that the shapes below reach `k_ntt_strided<TB, fwd>` and
`<TB, inv>`, `k_lde_mid<TB>` and (through MSGPU_LDE_UNFUSED=1 in a subprocess) `k_ntt_block<TB>` for every TB = 1..10, and
every entry point with 1-, 2- and 3-pass plans; each GPU test checks its launch counts against the mirror with the
context's profile. Four-pass plans (2^31 rows and more) are out of reach of a test and not covered.

Merkle: the same for the leaf-kernel choice of `b3_hash_rows` (staged / stream / direct / gather), node layers with a class
injected at every level of every `k_merkle_subtree` launch, `msgpu_open_batch_multi` over trees at different shifts, and
the column-block kernels.

These tests supersede, as checks of the kernels, the oracle comparisons of test_gpu_ntt.py, test_ntt_tiles.py and
test_gpu_merkle.py, which stay as a second, independent pin."""
import ctypes as C
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import _commit_ref as R

P = R.P
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RAND_SHIFT = 0x1234567890ABCDEF % P
SHIFTS = [7, 1, P - 1, RAND_SHIFT]
WIDTHS = [1, 2, 3, 4, 5, 6, 7, 8, 9, 17, 64]


# ---- mirror of the host drivers of ntt.cu ------------------------------------------------------------------------------
def plan_passes(log_n):
    """ntt.cu plan_passes: the fewest passes of at most 10 bits, the larger ones first."""
    if log_n == 0:
        return []
    n_passes = (log_n + 9) // 10
    base, rem = divmod(log_n, n_passes)
    return [base + (1 if i < rem else 0) for i in range(n_passes)]


def dft_kernels(log_n, inverse=False):
    return [("k_ntt_strided", tb, "inv" if inverse else "fwd") for tb in plan_passes(log_n)]


def lde_kernels(log_n, fused=True):
    """ntt_coset_lde: inverse passes over the upper bits, the last inverse pass fused with the first forward pass of every
    coset (k_lde_mid) or the whole inverse then k_ntt_block, then the remaining forward passes of size n / 2^tb."""
    if log_n == 0:
        return []
    plan = plan_passes(log_n)
    tb = plan[-1]
    inv = plan[:-1] if fused else plan
    first = ("k_lde_mid", tb) if fused else ("k_ntt_block", tb)
    return [("k_ntt_strided", t, "inv") for t in inv] + [first] + dft_kernels(log_n - tb)


def launch_counts(kernels):
    out = {}
    for k in kernels:
        out[k[0]] = out.get(k[0], 0) + 1
    return out


# ---- shapes ---------------------------------------------------------------------------------------------------------------
# (log_n, w): dft_batch, dft_batch_bitrev and idft_batch of one matrix
DFT_SHAPES = [(l, WIDTHS[l % len(WIDTHS)]) for l in range(0, 11)] + [(11, 3), (13, 17), (15, 2), (20, 1), (21, 2), (22, 1)]
# (log_n, added_bits, w, shift): coset_lde_batch_bitrev; 2^21 rows at added_bits 3 is a 2^24-row LDE
LDE_SHAPES = [(l, l % 5, WIDTHS[(l + 3) % len(WIDTHS)], SHIFTS[l % 4]) for l in range(0, 11)] + [
    (3, 4, 64, 7), (4, 3, 17, P - 1), (5, 0, 9, RAND_SHIFT), (11, 0, 3, 7), (14, 4, 1, 1), (17, 2, 2, RAND_SHIFT),
    (20, 1, 1, P - 1), (21, 0, 2, 7), (21, 3, 1, RAND_SHIFT), (22, 1, 1, 7)]
# (log_n, added_bits, w): lde_from_shifted_coefficients, a batch of 2^added_bits transforms of size n
LFC_SHAPES = [(0, 2, 3), (3, 0, 2), (6, 1, 5), (9, 2, 1), (10, 3, 17), (12, 3, 2), (16, 1, 1), (21, 1, 1), (21, 2, 1)]
# (log_nq, q, d): shifted_quotient_slices
SLICE_SHAPES = [(4, 2, 3), (12, 4, 2), (15, 1, 1), (21, 1, 2), (22, 2, 1), (23, 4, 1)]
# the three device-pointer forms: (log_n, w)
DEV_SHAPES = [(7, 5), (15, 2), (21, 1)]
# (log_n, added_bits, w): the unfused LDE, k_ntt_block at every tile size
UNFUSED_SHAPES = [(l, l % 4, 1 + l % 5) for l in range(1, 11)] + [(13, 1, 2), (21, 1, 1)]


def _matrix(seed, rows, cols):
    """Random canonical values with a column of p - 1, a column alternating 0 and p - 1, and edge values in the last column."""
    rng = np.random.default_rng(seed)
    m = rng.integers(0, P, size=(rows, cols), dtype=np.uint64)
    if cols >= 2:
        m[:, 0] = P - 1
    if cols >= 3:
        m[:, 1] = np.where(np.arange(rows) % 2 == 0, 0, P - 1).astype(np.uint64)
    edge = np.array([P - 1, 0, 1, P - 2**32, 2**32 - 1, 2**32], dtype=np.uint64)[:rows]
    m[:len(edge), -1] = edge
    return m


@functools.lru_cache(maxsize=None)
def _dft_case(log_n, w):
    m = _matrix(log_n * 100 + w, 1 << log_n, w)
    return m, R.dft(m)


# ---- CPU: the shapes reach every instantiation ----------------------------------------------------------------------
def test_plan_mirror_matches_source():
    """The mirror's constants are the ones in ntt.cu (a change there must be mirrored here)."""
    src = open(os.path.join(ROOT, "multi_stark_b200", "csrc", "ntt.cu")).read()
    assert "constexpr int kMaxLogT = 10;" in src
    assert "u32 np = (log_n + kMaxLogT - 1) / kMaxLogT;" in src
    assert "u32 base = log_n / np, rem = log_n % np;" in src
    assert [plan_passes(l) for l in (1, 10, 11, 20, 21, 24, 30)] == [[1], [10], [6, 5], [10, 10], [7, 7, 7], [8, 8, 8],
                                                                    [10, 10, 10]]


def test_shapes_reach_every_instantiation():
    reached = set()
    for l, _ in DFT_SHAPES:
        reached |= set(dft_kernels(l)) | set(dft_kernels(l, inverse=True))
    for l, _, _, _ in LDE_SHAPES:
        reached |= set(lde_kernels(l))
    for l, _, _ in LFC_SHAPES:
        reached |= set(dft_kernels(l))
    for l, _, _ in SLICE_SHAPES:
        reached |= set(dft_kernels(l))
    for l, _, _ in UNFUSED_SHAPES:
        reached |= set(lde_kernels(l, fused=False))
    want = {("k_ntt_strided", tb, d) for tb in range(1, 11) for d in ("fwd", "inv")}
    want |= {("k_lde_mid", tb) for tb in range(1, 11)} | {("k_ntt_block", tb) for tb in range(1, 11)}
    assert want <= reached, sorted(want - reached)
    for logs in ([l for l, _ in DFT_SHAPES], [s[0] for s in LDE_SHAPES], [s[0] for s in LFC_SHAPES],
                 [s[0] for s in SLICE_SHAPES], [s[0] for s in DEV_SHAPES], [s[0] for s in UNFUSED_SHAPES]):
        assert {1, 2, 3} <= {len(plan_passes(l)) for l in logs}
    assert set(range(5)) == {s[1] for s in LDE_SHAPES} and set(range(4)) <= {s[1] for s in LFC_SHAPES}
    assert set(SHIFTS) <= {s[3] for s in LDE_SHAPES} and set(WIDTHS) <= {s[1] for s in DFT_SHAPES} | {s[2] for s in LDE_SHAPES}
    assert {1, 2, 4} == {s[1] for s in SLICE_SHAPES if s[0] >= 21}


# ---- GPU fixtures and helpers -----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu():
    import multi_stark_b200 as ms
    ctx = ms.GpuContext(0)
    yield ms, ctx
    ctx.close()


def _profiled(ctx, fn):
    """(fn(), {kernel: launches}) over the launches of fn; the per-context table fills are dropped."""
    ctx.profile_begin()
    try:
        out = fn()
    finally:
        prof = ctx.profile_end()
    counts = {}
    for e in prof:
        if not e["kernel"].startswith("k_fill_"):
            counts[e["kernel"]] = counts.get(e["kernel"], 0) + e["launches"]
    return out, counts


def _u64p(a):
    return a.ctypes.data_as(C.c_void_p)


# ---- NTT ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("log_n,w", DFT_SHAPES)
def test_dft_idft(gpu, log_n, w):
    ms, ctx = gpu
    m, y = _dft_case(log_n, w)
    dft = ms.GpuDft(ctx)
    got, counts = _profiled(ctx, lambda: dft.dft_batch_bitrev(m))
    assert np.array_equal(got, y[R.rev_perm(log_n)])
    assert counts.get("k_ntt_strided", 0) == len(plan_passes(log_n))
    assert np.array_equal(dft.dft_batch(m), y)
    got, counts = _profiled(ctx, lambda: dft.idft_batch(y))
    assert np.array_equal(got, m)
    assert counts.get("k_ntt_strided", 0) == len(plan_passes(log_n))


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,added_bits,w,shift", LDE_SHAPES)
def test_coset_lde(gpu, log_n, added_bits, w, shift):
    ms, ctx = gpu
    m = _matrix(7 * log_n + added_bits, 1 << log_n, w)
    got, counts = _profiled(ctx, lambda: ms.GpuDft(ctx).coset_lde_batch_bitrev(m, added_bits, shift))
    assert np.array_equal(got, R.coset_lde_bitrev(m, added_bits, shift))
    want = launch_counts(lde_kernels(log_n))
    assert {k: counts.get(k, 0) for k in ("k_ntt_strided", "k_lde_mid", "k_ntt_block")} == \
        {k: want.get(k, 0) for k in ("k_ntt_strided", "k_lde_mid", "k_ntt_block")}


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,added_bits,w", LFC_SHAPES)
def test_lde_from_shifted_coefficients(gpu, log_n, added_bits, w):
    ms, ctx = gpu
    m = _matrix(11 * log_n + added_bits, 1 << log_n, w)
    got, counts = _profiled(ctx, lambda: ms.GpuDft(ctx).lde_from_shifted_coefficients(m, added_bits))
    assert np.array_equal(got, R.lde_from_shifted_coefficients(m, added_bits))
    assert counts.get("k_ntt_strided", 0) == len(plan_passes(log_n))


@pytest.mark.gpu
@pytest.mark.parametrize("log_nq,q,d", SLICE_SHAPES)
def test_shifted_quotient_slices(gpu, log_nq, q, d):
    ms, ctx = gpu
    m = _matrix(13 * log_nq + q, 1 << log_nq, d)
    got, counts = _profiled(ctx, lambda: ms.shifted_quotient_slices(ctx, m, q))
    assert np.array_equal(got, R.shifted_quotient_slices(m, q))
    assert counts.get("k_ntt_strided", 0) == len(plan_passes(log_nq))


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,w", DEV_SHAPES)
def test_device_pointer_forms(gpu, log_n, w):
    """msgpu_dft_batch_bitrev_dev, msgpu_coset_lde_batch_bitrev_dev and msgpu_lde_from_shifted_coefficients_dev."""
    ms, ctx = gpu
    L = ctx.L
    m, y = _dft_case(log_n, w)
    n = 1 << log_n
    din = ctx.upload(m)
    dout = ctx.malloc(n * 4 * w * 8)
    try:
        assert L.msgpu_dft_batch_bitrev_dev(ctx.h, C.c_void_p(din), n, w, C.c_void_p(dout)) == 0
        assert np.array_equal(ctx.download(dout, (n, w)), y[R.rev_perm(log_n)])
        assert L.msgpu_coset_lde_batch_bitrev_dev(ctx.h, C.c_void_p(din), n, w, 2, RAND_SHIFT, C.c_void_p(dout)) == 0
        assert np.array_equal(ctx.download(dout, (4 * n, w)), R.coset_lde_bitrev(m, 2, RAND_SHIFT))
        assert L.msgpu_lde_from_shifted_coefficients_dev(ctx.h, C.c_void_p(din), n, w, 1, C.c_void_p(dout)) == 0
        assert np.array_equal(ctx.download(dout, (2 * n, w)), R.lde_from_shifted_coefficients(m, 1))
    finally:
        ctx.free(din)
        ctx.free(dout)


_UNFUSED = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import multi_stark_b200 as ms
from tests import _commit_ref as R
from tests.test_gpu_commit_ref import UNFUSED_SHAPES, _matrix, _profiled
ctx = ms.GpuContext(0)
dft = ms.GpuDft(ctx)
for log_n, lb, w in UNFUSED_SHAPES:
    m = _matrix(log_n, 1 << log_n, w)
    got, counts = _profiled(ctx, lambda: dft.coset_lde_batch_bitrev(m, lb, 7))
    assert np.array_equal(got, R.coset_lde_bitrev(m, lb, 7)), (log_n, lb, w)
    assert counts.get("k_ntt_block") == 1 and "k_lde_mid" not in counts, (log_n, counts)
ctx.close()
print("ok")
"""


@pytest.mark.gpu
def test_unfused_coset_lde_every_tile():
    """MSGPU_LDE_UNFUSED=1 (read once per process): the whole inverse, then k_ntt_block per coset, at TB = 1..10."""
    env = dict(os.environ, MSGPU_LDE_UNFUSED="1")
    r = subprocess.run([sys.executable, "-c", _UNFUSED, ROOT], env=env, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr


# ---- leaf kernels -----------------------------------------------------------------------------------------------------
def leaf_kernel(widths, height):
    """merkle.cu b3_hash_rows: staged rows while 128 of them fit 96 KB (< 96 columns) or the row is one chunk, streamed
    segments for wider rows from 32 rows up, direct global reads when neither fits."""
    words = 2 * sum(widths)
    pitch = words | 1
    rows = min(128, 96 * 1024 // (pitch * 4))
    if rows < 128 and words * 4 > 1024 and height >= 32:
        return "k_hash_rows_stream"
    if rows >= 32 or rows >= height:
        return "k_hash_rows_staged"
    return "k_hash_rows_direct"


def leaf_rows_per_cta(widths, height):
    kernel = leaf_kernel(widths, height)
    if kernel != "k_hash_rows_staged":
        return 128
    rows = min(128, 96 * 1024 // ((2 * sum(widths) | 1) * 4))
    return max(1, rows // 32 * 32 if rows > 32 else rows)


# (widths of one height class, height); heights are powers of two (the ABI refuses others), so a partial last CTA comes from
# a staged tile of 96 rows or from fewer rows than one CTA
LEAF_SHAPES = [([95], 256), ([96], 128), ([128], 32), ([129], 32), ([129], 16), ([1], 1), ([3] * 12 + [0, 0], 128),
               ([10] * 10 + [0], 256), ([129], 64), ([400], 32), ([400], 256), ([7] * 9 + [0] + [50] * 5, 512), ([1000], 128),
               ([400], 16), ([1000], 16), ([1000], 8), ([45] * 19 + [0], 16), ([0, 2000, 0], 8), ([0, 2000, 0], 4)]
LEAF_SHAPES += [([5, 0, 3], 1 << k) for k in range(0, 10)] + [([500] * 2, h) for h in (8, 16, 32)]


def test_leaf_shapes_reach_every_branch():
    by = {}
    for ws, h in LEAF_SHAPES:
        by.setdefault(leaf_kernel(ws, h), []).append((ws, h))
    assert set(by) == {"k_hash_rows_staged", "k_hash_rows_stream", "k_hash_rows_direct"}
    for k, shapes in by.items():
        assert any(len([w for w in ws if w]) > 8 for ws, _ in shapes), k     # the uploaded (non-inline) matrix list
        assert any(0 in ws for ws, _ in shapes), k                            # zero-width matrices
        assert any(h % leaf_rows_per_cta(ws, h) for ws, h in shapes), k       # a partial last CTA
        assert any(h > leaf_rows_per_cta(ws, h) for ws, h in shapes) or k == "k_hash_rows_direct", k  # several CTAs
    assert leaf_rows_per_cta([96], 128) == 96 and leaf_rows_per_cta([95], 256) == 128
    assert leaf_kernel([95], 256) == "k_hash_rows_staged" and leaf_kernel([96], 128) == "k_hash_rows_staged"
    assert leaf_kernel([128], 32) == "k_hash_rows_staged" and leaf_kernel([129], 32) == "k_hash_rows_stream"
    assert leaf_kernel([129], 16) == "k_hash_rows_staged"
    assert [leaf_kernel([500] * 2, h) for h in (8, 16, 32)] == ["k_hash_rows_staged", "k_hash_rows_direct", "k_hash_rows_stream"]


@pytest.mark.gpu
@pytest.mark.parametrize("widths,height", LEAF_SHAPES)
def test_leaf_dispatch(gpu, widths, height):
    ms, ctx = gpu
    rng = np.random.default_rng(height * 7 + len(widths))
    mats = [rng.integers(0, P, size=(height, w), dtype=np.uint64) for w in widths]
    (root, pd), counts = _profiled(ctx, lambda: ms.GpuMmcs(ctx).commit(mats))
    want = R.mmcs_commit(mats)
    got = pd.layers()
    assert len(got) == len(want)
    for g, e in zip(got, want):
        assert np.array_equal(g, e)
    assert bytes(root) == want[-1][0].tobytes()
    leaf = {k: v for k, v in counts.items() if k.startswith("k_hash_rows")}
    assert leaf == {leaf_kernel(widths, height): 1}
    pd.free()


@pytest.mark.gpu
@pytest.mark.parametrize("n_asm,width,height", [(5, 6, 256), (1, 3000, 8), (2, 150, 64)])
def test_assembled_blocks(gpu, n_asm, width, height):
    """Column-block matrices assembled while hashed (msgpu_commit_ldes_blocks_dev): more than 4 in a class, or rows the
    direct kernel hashes, go through k_gather_blocks first."""
    ms, ctx = gpu
    rng = np.random.default_rng(n_asm * width)
    mats = [rng.integers(0, P, size=(height, width), dtype=np.uint64) for _ in range(n_asm)]
    cuts = [0, 1, width // 2, width]
    dsts, blocks, args = [], [], []
    for m in mats:
        dst = ctx.malloc(m.nbytes)
        bl = [(ctx.upload(np.ascontiguousarray(m[:, a:b])), b - a) for a, b in zip(cuts, cuts[1:])]
        dsts.append(dst)
        blocks += [p for p, _ in bl]
        args.append((dst, height, width, bl))
    try:
        (root, pd), counts = _profiled(ctx, lambda: ms.GpuPcs(ctx, 1).commit_ldes_blocks(args))
        want = R.mmcs_commit(mats)
        assert bytes(root) == want[-1][0].tobytes()
        assert np.array_equal(pd.layers()[0], want[0])
        for i, m in enumerate(mats):
            assert np.array_equal(ctx.download(dsts[i], m.shape), m)
        direct = leaf_kernel([width] * n_asm, height) == "k_hash_rows_direct"
        assert (counts.get("k_gather_blocks", 0) > 0) == (n_asm > 4 or direct)
        pd.free()
    finally:
        for p in dsts + blocks:
            ctx.free(p)


# ---- trees ------------------------------------------------------------------------------------------------------------
def subtree_launches(log_max):
    """mmcs.cu build_nodes: 10 levels per k_merkle_subtree launch while the layer is longer than 4096, then the rest."""
    out, l = [], 0
    while l < log_max:
        levels = 10 if (1 << (log_max - l)) > 4096 else log_max - l
        out.append(list(range(l + 1, l + levels + 1)))
        l += levels
    return out


def test_tree_shapes_reach_every_launch_position():
    assert subtree_launches(14) == [list(range(1, 11)), [11, 12, 13, 14]]
    assert subtree_launches(22) == [list(range(1, 11)), list(range(11, 23))]
    assert subtree_launches(23) == [list(range(1, 11)), list(range(11, 21)), [21, 22, 23]]


@pytest.mark.gpu
@pytest.mark.parametrize("log_max", range(0, 15))
def test_tree_injection_every_level(gpu, log_max):
    """One injected class at each level in turn (the first, middle and last level of every launch), then all at once."""
    ms, ctx = gpu
    rng = np.random.default_rng(log_max)
    top = rng.integers(0, P, size=(1 << log_max, 2), dtype=np.uint64)
    cases = [[top]] + [[top, rng.integers(0, P, size=(1 << (log_max - l), 1 + l % 3), dtype=np.uint64)]
                       for l in range(1, log_max + 1)]
    cases.append([top] + [rng.integers(0, P, size=(1 << (log_max - l), 1), dtype=np.uint64) for l in range(1, log_max + 1)])
    for mats in cases:
        (root, pd), counts = _profiled(ctx, lambda: ms.GpuMmcs(ctx).commit(mats))
        want = R.mmcs_commit(mats)
        got = pd.layers()
        assert len(got) == log_max + 1
        for l, (g, e) in enumerate(zip(got, want)):
            assert np.array_equal(g, e), (len(mats), l)
        assert counts.get("k_merkle_subtree", 0) == len(subtree_launches(log_max))
        pd.free()


def _tree_from_digests(ctx, classes):
    """msgpu_tree_from_digests over {height: (height, 32) uint8 digests} -> (pdata handle, root, device buffers)."""
    hs = sorted(classes, reverse=True)
    bufs = [ctx.upload(classes[h]) for h in hs]
    out, root = C.c_void_p(), np.zeros(32, dtype=np.uint8)
    assert ctx.L.msgpu_tree_from_digests(ctx.h, len(hs), (C.c_uint64 * len(hs))(*hs), (C.c_void_p * len(hs))(*bufs),
                                         C.byref(out), _u64p(root)) == 0
    return out, root, bufs


def _read_layers(ctx, h):
    out = []
    for i in range(int(ctx.L.msgpu_pdata_num_layers(h))):
        buf = np.empty((int(ctx.L.msgpu_pdata_layer_len(h, i)), 32), dtype=np.uint8)
        assert ctx.L.msgpu_pdata_read_layer(ctx.h, h, i, _u64p(buf)) == 0
        out.append(buf)
    return out


@pytest.mark.gpu
def test_tree_2_22_every_class(gpu):
    """Leaves of height 2^22 with a class injected at every level: two k_merkle_subtree launches, the second starting at the
    level of height 2^11."""
    ms, ctx = gpu
    rng = np.random.default_rng(22)
    classes = {1 << k: rng.integers(0, 256, size=(1 << k, 32), dtype=np.uint8) for k in range(0, 23)}
    (h, root, bufs), counts = _profiled(ctx, lambda: _tree_from_digests(ctx, classes))
    try:
        want = R.node_layers(classes[1 << 22], {k: v for k, v in classes.items() if k != 1 << 22})
        got = _read_layers(ctx, h)
        assert len(got) == 23
        for l, (g, e) in enumerate(zip(got, want)):
            assert np.array_equal(g, e), l
        assert bytes(root) == want[-1][0].tobytes()
        assert counts.get("k_merkle_subtree", 0) == 2
    finally:
        ctx.L.msgpu_pdata_free(h)
        for b in bufs:
            ctx.free(b)


# ---- openings -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_idx", [1, 7, 1000])
def test_open_batch_multi(gpu, n_idx):
    """k_open_multi over: an input round (rows of 1, 129, 128 and 1000 columns at three heights), FRI-layer-shaped trees at
    shifts 1 and 7, the rows-only local part of a sharded commitment (depth 0) and a paths-only tree from class digests."""
    ms, ctx = gpu
    L = ctx.L
    rng = np.random.default_rng(n_idx)
    mats_a = [rng.integers(0, P, size=s, dtype=np.uint64) for s in [(4096, 1), (4096, 129), (1024, 128), (128, 1000)]]
    mats_b = [rng.integers(0, P, size=(2048, 4), dtype=np.uint64)]
    mats_c = [rng.integers(0, P, size=(32, 4), dtype=np.uint64)]
    mats_d = [rng.integers(0, P, size=s, dtype=np.uint64) for s in [(4096, 3), (512, 2)]]
    cls_e = {4096: rng.integers(0, 256, size=(4096, 32), dtype=np.uint8), 8: rng.integers(0, 256, size=(8, 32), dtype=np.uint8)}
    _, pa = ms.GpuMmcs(ctx).commit(mats_a)
    _, pb = ms.GpuMmcs(ctx).commit(mats_b)
    _, pc = ms.GpuMmcs(ctx).commit(mats_c)
    dev_d = [ctx.upload(m) for m in mats_d]  # adopted by the local part
    loc = C.c_void_p()
    assert L.msgpu_commit_local_dev(ctx.h, (C.c_void_p * 2)(*dev_d), (C.c_uint64 * 2)(4096, 512), (C.c_uint64 * 2)(3, 2), 2, 1, 1,
                                    C.byref(loc)) == 0
    te, _, bufs = _tree_from_digests(ctx, cls_e)
    try:
        idx = rng.integers(0, 4096, size=n_idx, dtype=np.uint64)
        idx[:min(n_idx, 4)] = [0, 4095, 4095, 0][:min(n_idx, 4)]
        if n_idx > 10:
            idx[10:20] = idx[5]
        handles = [pa.h, pb.h, pc.h, loc, te]
        shifts = [0, 1, 7, 0, 0]
        want_o, want_p = R.open_batch_multi(
            [(mats_a, R.mmcs_commit(mats_a)), (mats_b, R.mmcs_commit(mats_b)), (mats_c, R.mmcs_commit(mats_c)), (mats_d, None),
             ([], R.node_layers(cls_e[4096], {8: cls_e[8]}))], shifts, idx)
        opened = np.zeros(max(want_o.size, 1), dtype=np.uint64)
        proofs = np.zeros((max(want_p.shape[0], 1), 32), dtype=np.uint8)
        got, counts = _profiled(ctx, lambda: L.msgpu_open_batch_multi(ctx.h, (C.c_void_p * 5)(*handles), (C.c_uint32 * 5)(*shifts), 5,
                                                                      _u64p(idx), n_idx, _u64p(opened), _u64p(proofs)))
        assert got == 0
        assert counts == {"k_open_multi": 1}
        assert np.array_equal(opened[:want_o.size], want_o)
        assert np.array_equal(proofs[:want_p.shape[0]], want_p)
        bad = np.array([4096 << 1], dtype=np.uint64)  # out of range for tree b at shift 1
        assert L.msgpu_open_batch_multi(ctx.h, (C.c_void_p * 1)(pb.h), (C.c_uint32 * 1)(1), 1, _u64p(bad), 1, _u64p(opened),
                                        _u64p(proofs)) != 0
    finally:
        L.msgpu_pdata_free(loc)
        L.msgpu_pdata_free(te)
        for b in bufs:
            ctx.free(b)
        pa.free()
        pb.free()
        pc.free()


# ---- column blocks -------------------------------------------------------------------------------------------------------
BLOCK_CASES = [[5], [0, 5], [2, 0, 3], [1] * 16, [0] * 15 + [7], [3, 0, 0, 4, 1, 0, 9, 2], [4] * 8, [0], [1, 2, 3, 4, 5, 6, 7, 8, 9, 10]]


@pytest.mark.gpu
@pytest.mark.parametrize("widths", BLOCK_CASES)
@pytest.mark.parametrize("rows", [1, 37, 1024])
def test_pack_interleave_round_trip(gpu, widths, rows):
    ms, ctx = gpu
    L = ctx.L
    W = sum(widths)
    m = np.random.default_rng(rows + W).integers(0, P, size=(rows, W), dtype=np.uint64)
    c1 = np.cumsum(widths).astype(np.uint64)
    c0 = np.concatenate([[0], c1[:-1]]).astype(np.uint64)
    want = np.concatenate([m[:, int(a):int(b)].ravel() for a, b in zip(c0, c1)])
    src, packed, back = ctx.upload(m), ctx.malloc(max(m.nbytes, 8)), ctx.malloc(max(m.nbytes, 8))
    try:
        assert L.msgpu_pack_column_blocks_dev(ctx.h, C.c_void_p(src), rows, W, len(widths), _u64p(c0), _u64p(c1), C.c_void_p(packed)) == 0
        assert np.array_equal(ctx.download(packed, (rows * W,)), want)
        wv = np.array(widths, dtype=np.uint64)
        assert L.msgpu_interleave_column_blocks_dev(ctx.h, C.c_void_p(packed), rows, len(widths), _u64p(wv), C.c_void_p(back)) == 0
        assert np.array_equal(ctx.download(back, (rows, W)), m)
    finally:
        for p in (src, packed, back):
            ctx.free(p)


@pytest.mark.gpu
def test_column_blocks_refusals(gpu):
    ms, ctx = gpu
    L = ctx.L
    buf = ctx.malloc(64 * 17 * 8)
    try:
        def pack(c0, c1, width):
            a, b = np.array(c0, dtype=np.uint64), np.array(c1, dtype=np.uint64)
            return L.msgpu_pack_column_blocks_dev(ctx.h, C.c_void_p(buf), 4, width, len(c0), _u64p(a), _u64p(b), C.c_void_p(buf))
        assert pack(list(range(17)), list(range(1, 18)), 17) != 0          # 17 blocks
        assert pack([0, 2], [2, 5], 4) != 0                                 # does not end at the width
        assert pack([0, 3], [2, 5], 5) != 0                                 # a gap
        assert pack([0, 1], [2, 5], 5) != 0                                 # an overlap
        assert pack([1], [5], 5) != 0                                       # does not start at 0
        assert pack([0, 2], [2, 5], 5) == 0
        w17 = np.ones(17, dtype=np.uint64)
        assert L.msgpu_interleave_column_blocks_dev(ctx.h, C.c_void_p(buf), 4, 17, _u64p(w17), C.c_void_p(buf)) != 0
        assert L.msgpu_interleave_column_blocks_dev(ctx.h, C.c_void_p(buf), 4, 0, _u64p(w17), C.c_void_p(buf)) != 0
    finally:
        ctx.free(buf)
