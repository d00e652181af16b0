"""The constraint-program kernels of csrc/quotient.cu against a plain big-int reference kept in this file (Python ints and
tests/_pyverifier.py's extension arithmetic and graph sweep; no oracle, no numpy uint64 arithmetic), bit for bit:

  * the stage-2 (logUp) trace: k_lookup_messages (the lookup-prefix interpreter), k_terms_and_block_sums, k_scan_block_sums,
    k_scan_write -- at every interpreter size launch_by_slots instantiates (both sides of each bucket edge, found with the
    lowering itself), at row counts that are not powers of two, at the edges of one scan block and past 1024 scan blocks;
  * the claims accumulator (k_claims), host-array and device-resident;
  * the quotient values (k_quotient_eval) on the quotient coset, whole and through the row-shard ABI
    (msgpu_quotient_values_shard with whole or column-extracted next shards, msgpu_quotient_finish);
  * the refusals: lookup expressions that read stage 2 or a public value, zero logUp messages, and row-sharded stage 2 of
    lookups that read a selector.
Selectors inside lookups follow the single-GPU convention: first = (r == 0), last = (r == rows - 1), trans = 1 - last; the
next row wraps around."""
import ctypes as C
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

from tests import _oracle as orc
from tests import _pyverifier as pv

P = pv.P
E = pv.E
X = pv.Expr
m, mn = X.main, X.main_next
FIRST, LAST, TRANS = X("first"), X("last"), X("trans")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INTERP_EDGES = [32, 64, 128, 256, 1024]   # launch_by_slots: <= 32, 64, 128, 256, 1024 slots, else the 4096-slot build


@pytest.fixture(scope="module")
def gpu():
    import multi_stark_b200 as ms
    ctx = ms.GpuContext(0)
    yield ms, ctx
    ctx.close()


# ---- reference ------------------------------------------------------------------------------------------------------------
def ext(v):
    return E(int(v[0]), int(v[1]))


def fingerprint(gamma, args):
    """sum_k args[k] * gamma^k (Horner over the reversed arguments)."""
    f = E(0)
    for a in reversed(args):
        f = f * gamma + a
    return f


def lookup_rows(graph, main, pre=None):
    """Per row r: [(multiplicity, [arguments])] of every lookup, from a sweep of the lookup prefix over the natural-order
    traces with first = (r == 0), last = (r == rows - 1), trans = 1 - last and the next row wrapping around."""
    rows = main.shape[0]
    prefix = types.SimpleNamespace(nodes=graph.nodes[:graph.lookup_prefix_len])
    out = []
    for r in range(rows):
        rn = (r + 1) % rows
        vals = lambda t, i: [E(int(v)) for v in t[i]] if t is not None else []  # noqa: E731
        first, last = E(int(r == 0)), E(int(r == rows - 1))
        buf = pv.sweep(prefix, [vals(pre, r), vals(pre, rn)], [vals(main, r), vals(main, rn)], None, None, first, last,
                       E(1) - last)
        out.append([(buf[mu].a, [buf[a].a for a in args]) for mu, args in graph.lookups])
    return out


def stage2_reference(graph, main, beta, gamma, pre=None):
    """(rows x 2L trace as Python ints, local sum): the exclusive running sum, row-major over (row, lookup), of
    multiplicity / (beta + fingerprint), each term inverted on its own."""
    s, flat = E(0), []
    for row in lookup_rows(graph, main, pre):
        for mult, args in row:
            msg = beta + fingerprint(gamma, args)
            assert not msg.is_zero(), "zero logUp message: the reference has no inverse for it"
            flat += [s.a, s.b]
            s = s + msg.inverse() * mult
    L = len(graph.lookups)
    return np.array(flat, dtype=object).reshape(main.shape[0], 2 * L), s


def claims_reference(claims, beta, gamma):
    acc = E(0)
    for c in claims:
        acc = acc + (beta + fingerprint(gamma, [int(v) for v in c])).inverse()
    return acc


def quotient_reference(circ, log_n, log_q, s1_lde, s2_lde, publics8, alpha, pre_lde=None):
    """Quotient values on the coset GENERATOR * H_{n q} from the first n q stored (bit-reversed) rows of the committed LDEs:
    the graph sweep, the logUp constraint values, the reversed-alpha fold and the division by Z_H. Returns (natural order,
    stored order), each nq x 2 of Python ints."""
    log_nq = log_n + log_q
    n, nq, q = 1 << log_n, 1 << log_nq, 1 << log_q
    w, ginv = pv.two_adic_generator(log_nq), pv.inv(pv.two_adic_generator(log_n))
    inj_norm = pv.inv(n * pv.two_adic_generator(log_n))
    publics = [E(int(v)) for v in publics8]
    delta = [(publics[6] - publics[4]) * inj_norm, (publics[7] - publics[5]) * inj_norm]
    a = ext(alpha)
    rows = lambda t, s: [E(int(v)) for v in t[s]] if t is not None else []  # noqa: E731
    nat = np.zeros((nq, 2), dtype=object)
    for i in range(nq):
        x = pv.GENERATOR * pow(w, i, P) % P
        zh = (pow(x, n, P) - 1) % P
        first, last = E(zh * pv.inv(x - 1)), E(zh * pv.inv(x - ginv))
        cur, nxt = pv.rev_bits(i, log_nq), pv.rev_bits((i + q) % nq, log_nq)
        s2c, s2n = rows(s2_lde, cur), rows(s2_lde, nxt)
        buf = pv.sweep(circ.graph, [rows(pre_lde, cur), rows(pre_lde, nxt)], [rows(s1_lde, cur), rows(s1_lde, nxt)],
                       [s2c, s2n], publics, first, last, E(x - ginv))
        cv = [buf[z] for z in circ.graph.zeros]
        pv.logup_constraint_values(circ.graph.lookups, buf, s2c, s2n, publics, delta, last, cv)
        assert len(cv) == circ.constraint_count
        comp = E(0)
        for v in cv:
            comp = comp * a + v
        val = comp * pv.inv(zh)
        nat[i] = (val.a, val.b)
    stored = nat[[pv.rev_bits(s, log_nq) for s in range(nq)]]
    return nat, stored


def u64(a):
    return np.asarray(a, dtype=object).astype(np.uint64)


# ---- circuits -------------------------------------------------------------------------------------------------------------
def slot_circuit(a, extra=0, width=24, n_lookups=2):
    """n_lookups lookups of `a` distinct non-leaf arguments each, all pinned until the end of the lookup prefix: the lowered
    slot count grows with `a` (by 1 to 4 per step); `extra` distinct constant arguments of lookup 0 add one slot each.
    Degree-3 logUp (quotient degree 2), plus one constraint that reads the selectors."""
    lookups = []
    for t in range(n_lookups):
        args = [m((i + t) % width) * m((3 * i + 1) % width) + X.const(t * a + i + 1) for i in range(a)]
        args += [X.const(P - 1 - i) for i in range(extra if t == 0 else 0)]
        lookups.append(pv.push(m(width - 1 - t), args) if t % 2 == 0 else pv.pull(m(width - 1 - t), args))
    return pv.Circuit(width, lookups, [FIRST * (m(0) - m(1)) + LAST * m(2) * m(3) + TRANS * (mn(4) - m(5))])


def slot_counts(circ, oracle, pre=None):
    """(full program slots, lookup-prefix slots) of the device lowering, checked against a node-by-node evaluation."""
    S = orc.OracleSystem(oracle, None, graphs=[pv.graph_dict(circ)], preprocessed=pre, log_blowup=1, num_queries=4)
    out = np.zeros(4, dtype=np.uint32)
    bad = int(oracle.orc_check_lowering(S.h, 0, 2, 5, out))
    S.close()
    assert bad == 0
    return int(out[0]), int(out[2])


_SLOTS = {}


def slots_of(a, oracle, extra=0):
    if (a, extra) not in _SLOTS:
        _SLOTS[a, extra] = slot_counts(slot_circuit(a, extra), oracle)
    return _SLOTS[a, extra]


def a_with_slots(kind, want, oracle):
    """(a, extra) whose full program (kind 0) or lookup prefix (kind 1) lowers to exactly `want` slots: the largest `a` that
    needs at most `want` (binary search: the count does not decrease with a), then constant arguments for the rest."""
    lo, hi = 1, 2
    while slots_of(hi, oracle)[kind] <= want:
        lo, hi = hi, hi * 2
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if slots_of(mid, oracle)[kind] <= want:
            lo = mid
        else:
            hi = mid
    extra = want - slots_of(lo, oracle)[kind]
    assert 0 <= extra <= 8
    assert slots_of(lo, oracle, extra)[kind] == want, "(%d, %d) lowers the %s to %d slots, not %d" % (
        lo, extra, ("full program", "prefix")[kind], slots_of(lo, oracle, extra)[kind], want)
    return lo, extra


SLOT_CASES = [(kind, t + d) for kind in ("full", "prefix") for t in INTERP_EDGES for d in (0, 1)]


def shape_circuits():
    """Lookup shapes next to the slot sweep: (name, circuit, preprocessed column or None)."""
    c = X.const
    pre = X.preprocessed
    return [
        ("preprocessed", pv.Circuit(3, [pv.pull(m(0), [c(0), pre(0)]), pv.push(m(1), [pre(1) * m(2), X.var(pv.PRE, 1, 0)])],
                                    [m(2) * pre(0) - m(1)], pre_width=2, pre_height=32), True),
        ("no_arguments", pv.Circuit(3, [pv.push(m(0), []), pv.pull(m(1) * m(2), [m(2)])], [m(0) * m(1) - m(2)]), None),
        ("single_pull", pv.Circuit(2, [pv.pull(m(1), [m(0)])], []), None),
        ("no_lookups", pv.Circuit(3, [], [m(0) * m(1) - m(2), FIRST * m(0), LAST * (mn(1) - m(2))]), None),
        ("selectors", pv.Circuit(4, [pv.push(FIRST * m(0), [m(1), LAST]), pv.pull(LAST + m(2), [TRANS * m(3), mn(0)]),
                                     pv.push(TRANS, [mn(3) * m(1), FIRST + c(5)]), pv.pull(m(3), [mn(2)])], [m(0) - mn(1) * TRANS]),
         None),
    ]


# ---- device helpers -------------------------------------------------------------------------------------------------------
def run_stage2(ms, ctx, system, main, beta, gamma, pre=None):
    prog = ms.Program(ctx, system, 0)
    d_main = ctx.upload(main)
    d_pre = ctx.upload(pre) if pre is not None else None
    try:
        out, local = prog.stage2_trace(d_main, main.shape[0], beta, gamma, d_pre)
        got = ctx.download(out, (main.shape[0], system.circuits[0]["stage2_width"]))
        ctx.free(out)
    finally:
        ctx.free(d_main)
        if d_pre:
            ctx.free(d_pre)
        prog.free()
    return got, local


def check_stage2(ms, ctx, circ, main, beta2, gamma2, pre=None, system=None):
    own = system is None
    if own:
        system = ms.System.from_graphs([pv.graph_dict(circ)], preprocessed=[pre] if pre is not None else None)
    got, local = run_stage2(ms, ctx, system, main, beta2, gamma2, pre)
    if own:
        system.close()
    if circ.num_lookups == 0:  # the pass-through accumulator column is zero
        assert not got.any() and not local.any()
        return
    want, total = stage2_reference(circ.graph, main, ext(beta2), ext(gamma2), pre)
    assert np.array_equal(got, u64(want)), "stage-2 trace differs from the reference"
    assert (int(local[0]), int(local[1])) == (total.a, total.b), "local sum differs from the reference"


def check_quotient(ms, ctx, oracle, circ, log_n, lb, rng, pre=None):
    g = pv.graph_dict(circ)
    system = ms.System.from_graphs([g], preprocessed=[pre] if pre is not None else None, log_blowup=lb)
    info = system.circuits[0]
    log_q = info["quotient_degree"].bit_length() - 1
    assert (1 << log_q) == circ.quotient_degree()
    n, nq = 1 << log_n, 1 << (log_n + log_q)
    main = orc.rand_matrix(rng, n, circ.main_width)
    s2 = orc.rand_matrix(rng, n, circ.stage2_width)   # the evaluation is pointwise: any stage-2 values exercise it
    pcs = ms.GpuPcs(ctx, lb)
    _, pd1 = pcs.commit([main])
    _, pd2 = pcs.commit([s2])
    pd0 = pcs.commit([pre])[1] if pre is not None else None
    alpha = rng.integers(0, P, size=2, dtype=np.uint64)
    publics = rng.integers(0, P, size=8, dtype=np.uint64)
    prog = ms.Program(ctx, system, 0)
    lde, rows, cols, vals = prog.quotient(pd0, 0, pd1, 0, pd2, 0, log_n, log_q, lb, publics, alpha, want_values=True)
    s1_lde, s2_lde = pd1.read_rows(0, 0, nq), pd2.read_rows(0, 0, nq)
    pre_lde = pd0.read_rows(0, 0, nq) if pd0 is not None else None
    want, _ = quotient_reference(circ, log_n, log_q, s1_lde, s2_lde, publics, alpha, pre_lde)
    assert np.array_equal(vals, u64(want)), "quotient values differ from the reference"
    # slices + LDE of the reference values through the oracle's path
    q = 1 << log_q
    sl = np.zeros((n, 2 * q), dtype=np.uint64)
    oracle.orc_shifted_quotient_slices(u64(want), nq, 2, q, sl)
    want_lde = np.zeros((rows, cols), dtype=np.uint64)
    oracle.orc_lde_from_shifted_coefficients(sl, n, 2 * q, lb, want_lde)
    assert np.array_equal(ctx.download(lde, (rows, cols)), want_lde), "quotient LDE differs"
    ctx.free(lde)
    prog.free()
    for pd in (pd0, pd1, pd2):
        if pd is not None:
            pd.free()
    system.close()


def rnd_ext(rng):
    return rng.integers(0, P, size=2, dtype=np.uint64)


# ---- CPU: the reference itself --------------------------------------------------------------------------------------------
def test_reference_stage2_recurrence_and_balance(oracle):
    """On a valid U32-add witness the local sums of the byte table and the adds plus the claims accumulator vanish; each
    trace step adds multiplicity / message; and the reference agrees with the oracle on the same inputs."""
    import multi_stark_b200 as ms
    byte, add, claims = ms.u32_add_workload(16)
    table, adds = pv.byte_table(), pv.u32_add()
    pre = np.arange(256, dtype=np.uint64).reshape(256, 1)
    rng = np.random.default_rng(3)
    b2, g2 = rnd_ext(rng), rnd_ext(rng)
    beta, gamma = ext(b2), ext(g2)
    t0, s0 = stage2_reference(table.graph, byte, beta, gamma, pre)
    t1, s1 = stage2_reference(adds.graph, add, beta, gamma)
    acc = claims_reference(claims, beta, gamma)
    assert (s0 + s1 + acc).is_zero(), "lookups of a valid witness do not balance"
    flat = t1.reshape(-1, 2)
    k = 0
    for mult, args in [t for row in lookup_rows(adds.graph, add) for t in row][:-1]:
        step = E(*flat[k + 1]) - E(*flat[k])
        assert step * (beta + fingerprint(gamma, args)) == E(mult)
        k += 1
    osy = oracle.orc_system_create(b"u32_add", 1, 0, 1, 100, 0, 0)
    for ci, (tr, want) in enumerate([(byte, t0), (add, t1)]):
        got = np.zeros(want.shape, dtype=np.uint64)
        wl = np.zeros(2, dtype=np.uint64)
        oracle.orc_stage2_trace(osy, ci, np.ascontiguousarray(tr), tr.shape[0], b2, g2, got, wl)
        assert np.array_equal(got, u64(want))
    oracle.orc_system_free(osy)
    want_acc = np.zeros(2, dtype=np.uint64)
    oracle.orc_claims_accumulator(claims, claims.shape[0], claims.shape[1], b2, g2, want_acc)
    assert (int(want_acc[0]), int(want_acc[1])) == (acc.a, acc.b)


def test_reference_quotient_matches_oracle(oracle):
    """The quotient reference against the oracle's quotient_values on arbitrary rows (the evaluation is pointwise)."""
    circ = shape_circuits()[4][1]
    rng = np.random.default_rng(11)
    log_n, log_q = 3, circ.quotient_degree().bit_length() - 1
    nq = 1 << (log_n + log_q)
    s1, s2 = orc.rand_matrix(rng, nq, circ.main_width), orc.rand_matrix(rng, nq, circ.stage2_width)
    publics, alpha = rng.integers(0, P, size=8, dtype=np.uint64), rnd_ext(rng)
    want, stored = quotient_reference(circ, log_n, log_q, s1, s2, publics, alpha)
    S = orc.OracleSystem(oracle, None, graphs=[pv.graph_dict(circ)], log_blowup=log_q)
    got = np.zeros((nq, 2), dtype=np.uint64)
    oracle.orc_quotient_values(S.h, 0, log_n, log_q, None, s1, s2, publics, alpha, got)
    S.close()
    assert np.array_equal(got, u64(want))
    assert np.array_equal(stored[[pv.rev_bits(i, 3 + log_q) for i in range(nq)]], want)


@pytest.mark.parametrize("kind,want", SLOT_CASES)
def test_slot_cases_hit_every_interpreter_size(oracle, kind, want):
    """The slot sweep lands on both sides of every launch_by_slots edge, for the full program (k_quotient_eval) and the lookup
    prefix (k_lookup_messages): want - 1 <= 1024 runs the 4096-slot build."""
    a, extra = a_with_slots(("full", "prefix").index(kind), want, oracle)
    assert slots_of(a, oracle, extra)[("full", "prefix").index(kind)] == want


# ---- fix 1: lookups that read stage 2 or a public value are refused when the program is made ----------------------------
def bad_lookup_graphs():
    # lookup 0 reads node 0 (a stage-2 column / a public value) as its argument: multiplicity = const 1 (node 1)
    base = dict(zeros=[], lookups=[(1, [0])], lookup_prefix_len=2, main_width=1)
    return [dict(base, nodes=[("var", pv.STAGE2, 0, 0), ("const", 1)]), dict(base, nodes=[("public", 0), ("const", 1)]),
            dict(base, nodes=[("var", pv.MAIN, 0, 0), ("public", 2), ("mul", 0, 1)], lookups=[(2, [0])], lookup_prefix_len=3)]


@pytest.mark.parametrize("which", [0, 1, 2])
def test_system_refuses_lookup_reading_stage2_or_public(which):
    import multi_stark_b200 as ms
    with pytest.raises(ValueError, match="lookup expression reads"):
        ms.System.from_graphs([bad_lookup_graphs()[which]])


@pytest.mark.gpu
@pytest.mark.parametrize("which", [0, 1, 2])
def test_program_create_refuses_lookup_reading_stage2_or_public(gpu, which):
    """msgpu_program_create takes descriptors directly. Only creation is tried: a kernel run of such a program would read a
    null stage-2 / publics pointer."""
    ms, ctx = gpu
    from multi_stark_b200.system import graph_descs
    arr, keep = graph_descs([bad_lookup_graphs()[which]])
    h = C.c_void_p()
    rc = ctx.L.msgpu_program_create(ctx.h, C.cast(arr, C.c_void_p), C.byref(h))
    if rc == 0:
        ctx.L.msgpu_program_free(h)
    assert rc != 0, "a lookup that reads stage 2 or a public value was accepted"
    assert b"lookup expression reads" in ctx.L.msgpu_last_error()


# ---- interpreter sizes ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind,want", SLOT_CASES)
def test_interpreter_sizes_match_reference(gpu, oracle, kind, want):
    ms, ctx = gpu
    a, extra = a_with_slots(("full", "prefix").index(kind), want, oracle)
    circ = slot_circuit(a, extra)
    rng = np.random.default_rng(want * 2 + len(kind))
    log_n = 5 + want % 3
    main = orc.rand_matrix(rng, 1 << log_n, circ.main_width)
    check_stage2(ms, ctx, circ, main, rnd_ext(rng), rnd_ext(rng))
    check_quotient(ms, ctx, oracle, circ, 5, 1 + want % 2, rng)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [s[0] for s in shape_circuits()])
@pytest.mark.parametrize("log_n,lb", [(5, 1), (6, 2)])
def test_lookup_shapes_match_reference(gpu, oracle, name, log_n, lb):
    ms, ctx = gpu
    _, circ, has_pre = [s for s in shape_circuits() if s[0] == name][0]
    rng = np.random.default_rng(log_n * 7 + lb)
    n = 1 << log_n
    pre = orc.rand_matrix(rng, n, circ.pre_width) if has_pre else None
    if has_pre:
        circ.pre_height = n
    main = orc.rand_matrix(rng, n, circ.main_width)
    check_stage2(ms, ctx, circ, main, rnd_ext(rng), rnd_ext(rng), pre)
    check_quotient(ms, ctx, oracle, circ, log_n, lb, rng, pre)


# ---- scan shapes ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("rows,L", [(1, 1), (1, 3), (3, 2), (7, 1), (7, 4), (2047, 1), (2048, 1), (2049, 1), (683, 3), (1023, 2),
                                    (1025, 2)])
def test_stage2_scan_edges_match_reference(gpu, rows, L):
    """Row counts that are not powers of two, and rows x L = 2047 / 2048 / 2049 (the edges of one 2048-term scan block)."""
    ms, ctx = gpu
    lookups = [(pv.push if j % 2 else pv.pull)(m(j) + FIRST, [m(j + 1) * mn(0), TRANS + m(0)]) for j in range(L)]
    circ = pv.Circuit(L + 1, lookups, [])
    rng = np.random.default_rng(rows * 10 + L)
    check_stage2(ms, ctx, circ, orc.rand_matrix(rng, rows, L + 1), rnd_ext(rng), rnd_ext(rng))


@pytest.mark.gpu
@pytest.mark.parametrize("rows,L", [(1 << 21, 1), ((1 << 21) + 8, 1), (1 << 20, 3), ((1 << 19) + 3, 5)])
def test_stage2_many_scan_blocks(gpu, rows, L):
    """2^21 terms = exactly 1024 scan blocks, and more (k_scan_block_sums' per-thread chunk loop). Lookups without arguments:
    every message is beta, so trace entry i is beta^-1 times the exclusive prefix sum of the multiplicities."""
    ms, ctx = gpu
    circ = pv.Circuit(L, [(pv.push if j % 2 else pv.pull)(m(j), []) for j in range(L)], [])
    rng = np.random.default_rng(rows + L)
    main = orc.rand_matrix(rng, rows, L)
    beta, gamma = rnd_ext(rng), rnd_ext(rng)
    system = ms.System.from_graphs([pv.graph_dict(circ)])
    got, local = run_stage2(ms, ctx, system, main, beta, gamma)
    system.close()
    mult = main.astype(object)
    mult[:, 0::2] = (P - mult[:, 0::2]) % P   # pulls: the multiplicity enters negated
    flat = mult.reshape(-1)
    excl = np.concatenate([[0], np.cumsum(flat)[:-1]]) % P
    bi = ext(beta).inverse()
    want = np.empty((flat.size, 2), dtype=object)
    want[:, 0] = excl * bi.a % P
    want[:, 1] = excl * bi.b % P
    assert np.array_equal(got.reshape(-1, 2), u64(want))
    total = int(flat.sum()) % P
    assert (int(local[0]), int(local[1])) == (total * bi.a % P, total * bi.b % P)


# ---- claims ---------------------------------------------------------------------------------------------------------------
def claims_upload_accumulate(ctx, claims, beta, gamma):
    from multi_stark_b200._ffi import check
    cl = C.c_void_p()
    digest = np.zeros(32, dtype=np.uint8)
    check(ctx.L.msgpu_claims_upload(ctx.h, claims.ctypes.data_as(C.c_void_p), claims.shape[0], claims.shape[1], None, 0,
                                    C.byref(cl), digest.ctypes.data_as(C.c_void_p)))
    out = np.zeros(2, dtype=np.uint64)
    try:
        b, g = np.asarray(beta, dtype=np.uint64), np.asarray(gamma, dtype=np.uint64)
        check(ctx.L.msgpu_claims_accumulate(cl, b.ctypes.data_as(C.c_void_p), g.ctypes.data_as(C.c_void_p),
                                            out.ctypes.data_as(C.c_void_p)))
    finally:
        ctx.L.msgpu_claims_free(cl)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("length", [0, 1, 4, 33])
@pytest.mark.parametrize("n", [1, 7, 8, 9, 2047, 2048, 2049, 3 * 2048 + 5])
def test_claims_match_reference(gpu, n, length):
    ms, ctx = gpu
    rng = np.random.default_rng(n * 41 + length)
    claims = orc.rand_matrix(rng, n, length)
    beta, gamma = rnd_ext(rng), rnd_ext(rng)
    want = claims_reference(claims, ext(beta), ext(gamma))
    got = ms.claims_accumulator(ctx, claims, beta, gamma)
    assert (int(got[0]), int(got[1])) == (want.a, want.b)
    if length:  # the device-resident path (msgpu_claims_upload takes claims of at least one value)
        got = claims_upload_accumulate(ctx, claims, beta, gamma)
        assert (int(got[0]), int(got[1])) == (want.a, want.b)


# ---- fix 3: a zero logUp message is refused ---------------------------------------------------------------------------------
def neg(e):
    return np.array([(-e.a) % P, (-e.b) % P], dtype=np.uint64)


@pytest.mark.gpu
@pytest.mark.parametrize("r,j", [(1, 1), (33, 2), (100, 2)])
def test_stage2_refuses_zero_message(gpu, r, j):
    """beta = -fingerprint(gamma, arguments of row r, lookup j), a term in the middle of a batch of 8: refused; beta + 1 is
    not, and matches the reference."""
    ms, ctx = gpu
    from multi_stark_b200._ffi import MsgpuError
    L = 3
    circ = pv.Circuit(4, [pv.push(m(k), [m(k + 1), m(0) * m(3)]) for k in range(L)], [])
    rng = np.random.default_rng(r + j)
    main = orc.rand_matrix(rng, 256, 4)
    assert (r * L + j) % 8 in (3, 4, 5, 6)
    gamma = rnd_ext(rng)
    _, args = lookup_rows(circ.graph, main)[r][j]
    beta = neg(fingerprint(ext(gamma), args))
    system = ms.System.from_graphs([pv.graph_dict(circ)])
    with pytest.raises(MsgpuError, match="logUp message"):
        run_stage2(ms, ctx, system, main, beta, gamma)
    beta[0] = (int(beta[0]) + 1) % P
    check_stage2(ms, ctx, circ, main, beta, gamma, system=system)
    system.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n,i", [(7, 3), (2049, 2045), (100, 52)])
def test_claims_refuse_zero_message(gpu, n, i):
    ms, ctx = gpu
    from multi_stark_b200._ffi import MsgpuError
    rng = np.random.default_rng(n + i)
    claims = orc.rand_matrix(rng, n, 4)
    gamma = rnd_ext(rng)
    beta = neg(fingerprint(ext(gamma), [int(v) for v in claims[i]]))
    with pytest.raises(MsgpuError, match="logUp message"):
        ms.claims_accumulator(ctx, claims, beta, gamma)
    with pytest.raises(MsgpuError, match="logUp message"):
        claims_upload_accumulate(ctx, claims, beta, gamma)
    beta[0] = (int(beta[0]) + 1) % P
    want = claims_reference(claims, ext(beta), ext(gamma))
    for got in (ms.claims_accumulator(ctx, claims, beta, gamma), claims_upload_accumulate(ctx, claims, beta, gamma)):
        assert (int(got[0]), int(got[1])) == (want.a, want.b)


# ---- row-shard quotient ABI on one GPU --------------------------------------------------------------------------------------
def shard_circuit(q):
    """A circuit with preprocessed, main and stage-2 reads at the next row (main columns 2..4 only: a narrow halo) and quotient
    degree q."""
    pre = X.preprocessed
    deg = {1: 2, 2: 3, 4: 5}[q]
    prod = m(2)
    for k in range(deg - 1):
        prod = prod * m(k % 5)
    cons = [prod - mn(3), FIRST * (X.var(pv.PRE, 1, 1) - m(0)), LAST * mn(2), TRANS * (mn(4) - pre(0))]
    return pv.Circuit(6, [pv.push(m(5), [m(1), pre(1)]), pv.pull(m(0), [m(4)])], cons, pre_width=2, pre_height=0)


def next_of(e, q, n_shards):
    """The shard holding the next trace rows of shard e (as RowShardBackend::commit_quotient computes it)."""
    lnp = n_shards.bit_length() - 1
    return pv.rev_bits((pv.rev_bits(e, lnp) + q) % n_shards, lnp)


@pytest.mark.gpu
@pytest.mark.parametrize("n_shards", [2, 4, 8])
@pytest.mark.parametrize("q,lb", [(1, 1), (1, 2), (2, 1), (2, 2), (4, 2)])
def test_quotient_shards_match_reference(gpu, oracle, n_shards, q, lb):
    ms, ctx = gpu
    from multi_stark_b200._ffi import check
    L = ctx.L
    circ = shard_circuit(q)
    log_n = 5
    n = 1 << log_n
    circ.pre_height = n
    rng = np.random.default_rng(q * 100 + lb * 10 + n_shards)
    pre = orc.rand_matrix(rng, n, 2)
    system = ms.System.from_graphs([pv.graph_dict(circ)], preprocessed=[pre], log_blowup=lb)
    log_q = system.circuits[0]["quotient_degree"].bit_length() - 1
    assert 1 << log_q == q
    nq = n * q
    main, s2 = orc.rand_matrix(rng, n, 6), orc.rand_matrix(rng, n, circ.stage2_width)
    pcs = ms.GpuPcs(ctx, lb)
    pds = [pcs.commit([t])[1] for t in (pre, main, s2)]
    widths = [2, 6, circ.stage2_width]
    alpha, publics = rnd_ext(rng), rng.integers(0, P, size=8, dtype=np.uint64)
    prog = ms.Program(ctx, system, 0)
    lde_whole, rows, cols, vals = prog.quotient(pds[0], 0, pds[1], 0, pds[2], 0, log_n, log_q, lb, publics, alpha, want_values=True)
    ldes = [pd.read_rows(0, 0, nq) for pd in pds]
    want_nat, want_stored = quotient_reference(circ, log_n, log_q, ldes[1], ldes[2], publics, alpha, ldes[0])
    assert np.array_equal(vals, u64(want_nat))
    # the columns read at the next row, per source (the stage-2 accumulator pair always)
    lo_hi = [(1, 2), (2, 5), (0, 2)]
    Ls = nq // n_shards
    bufs = [[ctx.upload(np.ascontiguousarray(t[e * Ls:(e + 1) * Ls])) for t in ldes] for e in range(n_shards)]
    pub_p, al_p = publics.ctypes.data_as(C.c_void_p), alpha.ctypes.data_as(C.c_void_p)
    assert any(next_of(e, q, n_shards) != e for e in range(n_shards)) == (q % n_shards != 0)
    for extract in (False, True):
        out = ctx.malloc(nq * 16)
        tmp = []
        for e in range(n_shards):
            dn = next_of(e, q, n_shards)
            nxt, nw, nc0 = list(bufs[dn]), list(widths), [0, 0, 0]
            if extract:
                for k, (lo, hi) in enumerate(lo_hi):
                    d = ctx.malloc(Ls * (hi - lo) * 8)
                    tmp.append(d)
                    check(L.msgpu_extract_columns_dev(ctx.h, C.c_void_p(bufs[dn][k]), Ls, widths[k], lo, hi, C.c_void_p(d)))
                    nxt[k], nw[k], nc0[k] = d, hi - lo, lo
            check(L.msgpu_quotient_values_shard(ctx.h, prog.h, (C.c_void_p * 3)(*bufs[e]), (C.c_void_p * 3)(*nxt),
                                                (C.c_uint32 * 3)(*nw), (C.c_uint32 * 3)(*nc0), e * Ls, Ls, dn * Ls, log_n, log_q,
                                                pub_p, al_p, C.c_void_p(out + e * Ls * 16)))
        got = ctx.download(out, (nq, 2))
        assert np.array_equal(got, u64(want_stored)), "sharded quotient values differ (extract=%s)" % extract
        assert np.array_equal(got, vals[[pv.rev_bits(s, log_n + log_q) for s in range(nq)]])
        lde = C.c_void_p()
        check(L.msgpu_quotient_finish(ctx.h, C.c_void_p(out), log_n, log_q, lb, C.byref(lde)))
        assert ctx.download(lde.value, (rows, cols)).tobytes() == ctx.download(lde_whole, (rows, cols)).tobytes()
        ctx.free(lde.value)
        for d in tmp + [out]:
            ctx.free(d)
    # refusals (argument checks, nothing is launched)
    dummy = ctx.malloc(Ls * 16)
    cur = (C.c_void_p * 3)(*bufs[0])
    rc = L.msgpu_quotient_values_shard(ctx.h, prog.h, cur, cur, None, None, nq - Ls + 1, Ls, 0, log_n, log_q, pub_p, al_p,
                                       C.c_void_p(dummy))
    assert rc != 0 and b"outside the quotient domain" in L.msgpu_last_error()
    missing = (C.c_void_p * 3)(bufs[0][0], None, bufs[0][2])
    rc = L.msgpu_quotient_values_shard(ctx.h, prog.h, missing, cur, None, None, 0, Ls, 0, log_n, log_q, pub_p, al_p, C.c_void_p(dummy))
    assert rc != 0 and b"missing matrix" in L.msgpu_last_error()
    no_pre = (C.c_void_p * 3)(None, bufs[0][1], bufs[0][2])
    rc = L.msgpu_quotient_values_shard(ctx.h, prog.h, no_pre, no_pre, None, None, 0, Ls, 0, log_n, log_q, pub_p, al_p,
                                       C.c_void_p(dummy))
    assert rc != 0 and b"missing matrix" in L.msgpu_last_error()
    ctx.free(dummy)
    for bl in bufs:
        for d in bl:
            ctx.free(d)
    ctx.free(lde_whole)
    prog.free()
    for pd in pds:
        pd.free()
    system.close()


# ---- fix 2: row-sharded stage 2 refuses selectors inside lookups ------------------------------------------------------------
def free_port():
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def run_rowshard_cases(tmp_path, world, cases):
    spec = tmp_path / "cases.json"
    spec.write_text(json.dumps(cases))
    prefix = str(tmp_path / "rs")
    port = free_port()
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "_rowshard_lookup_worker.py"), str(spec), prefix],
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = []
    for p in procs:
        try:
            out, _ = p.communicate(timeout=600)
        except subprocess.TimeoutExpired:
            for x in procs:
                x.kill()
            raise
        outs.append(out)
    if any(p.returncode != 0 for p in procs):
        raise AssertionError("\n".join("---- rank %d rc %s ----\n%s" % (r, p.returncode, outs[r][-2500:]) for r, p in enumerate(procs)))
    return [json.load(open("%s.rank%d.json" % (prefix, r))) for r in range(world)]


@pytest.mark.gpu
def test_rowshard_refuses_selectors_in_lookups(tmp_path):
    """push(first, [m(0)]) and pull(first, [m(0)]) cancel on every trace, so the witness is valid. On a trace split into row
    blocks every block's row 0 would see first = 1: the row-sharded prover refuses it on every rank. On traces that are not
    split (width < ranks, or fewer than 64 rows per rank) it proves, with the single-GPU proof's bytes."""
    rng = np.random.default_rng(9)
    cases, want_error = [], []
    for width, height, refused in [(2, 128, True), (1, 128, False), (2, 64, False)]:
        circ = pv.Circuit(width, [pv.push(FIRST, [m(0)]), pv.pull(FIRST, [m(0)])], [])
        g = pv.graph_dict(circ)
        cases.append(dict(graph=g, trace=orc.rand_matrix(rng, height, width).tolist()))
        want_error.append(refused)
    results = run_rowshard_cases(tmp_path, 2, cases)
    for k, refused in enumerate(want_error):
        for r in range(2):
            res = results[r][k]
            if refused:
                assert res["error"] is not None and "is_first_row" in res["error"], "case %d rank %d: %s" % (k, r, res)
            else:
                assert res["error"] is None, res["error"]
                assert res["proof"] == results[0][k]["single"], "case %d rank %d: proof differs from the single-GPU proof" % (k, r)
