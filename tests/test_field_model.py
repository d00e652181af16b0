"""The Goldilocks primitives of csrc/gl.cuh, run through tests/_gl_model.py (which interprets gl.cuh's own inline PTX), against
Python ints, with a record of every carry and borrow outcome.

The operand table (tests/_gl_model.py) holds the edge classes, the non-canonical values that "any u64" operands may take,
targeted pairs and Acc160 limb states. Together with 10^5 seeded random operands it must (a) give the exact result of every
primitive, inside the range its comment promises, and (b) drive every carry / borrow of every asm block both ways, except
the ones listed in CLAIMED_NEVER: those are the comments of gl.cuh saying a carry cannot happen, and they must stay 0 on
every operand. The GPU test (test_gpu_field.py) runs the same table through the compiled code, so this coverage is the
coverage of the device test too."""
import os
import re

import numpy as np
import pytest

from tests import _gl_model as G
from tests import _naive as nv

P = G.P
N_RANDOM = 100_000

# (block, instruction index, instruction): why its carry / borrow can never be 1. The comments are quoted from gl.cuh.
CLAIMED_NEVER = {
    ("add_lazy", 6, "addc.u32 %1, %1, 0"): "cannot wrap again since b < p",
    ("sub_lazy", 5, "subc.u32 %1, %1, 0"): "cannot borrow again since b < p (and b = p, which gl::add passes)",
    ("reduce128_lazy", 5, "subc.u32 %1, %1, 0"): "t = lo - hh (+p on borrow): lo - hh + p >= 0 since hh < 2^32",
    ("reduce128_lazy", 7, "subc.u32 t1, %4, 0"): "u = hl * (2^32 - 1) = (hl << 32) - hl is not negative",
    ("reduce128_lazy", 13, "addc.u32 %1, %1, 0"): "cannot carry twice, u <= (2^32-1)^2",
    ("reduce128", 6, "subc.u32 t1, t1, 0"): "t = lo - h1 (- eps on borrow): the - eps cannot borrow again",
    ("reduce128", 11, "mad.wide.u32 rr, k, 0xffffffff, rr"): "r = t + h0 * eps (+ eps on carry): the + eps cannot carry "
                                                               "again, since h0 * eps <= (2^32-1)^2",
    ("acc_mac", 4, "addc.u32 %4, %4, 0"): "Exact for up to 2^32 terms: l4 never overflows",
    ("acc_mac", 8, "addc.u32 %4, %4, 0"): "Exact for up to 2^32 terms: l4 never overflows",
    ("acc_mac", 12, "addc.u32 %4, %4, 0"): "Exact for up to 2^32 terms: l4 never overflows",
}

POW_EXPONENTS = [0, 1, P - 2, P - 1, 2**64 - 1]


def _pairs(xs, ys):
    return [x for x in xs for y in ys], [y for x in xs for y in ys]


def random_operands(n, seed=11):
    rng = np.random.default_rng(seed)
    a = [int(v) for v in rng.integers(0, 2**64, size=n, dtype=np.uint64)]
    b = [int(v) for v in rng.integers(0, 2**64, size=n, dtype=np.uint64)]
    return a, b


def check_all(m, n_random):
    """Run every primitive of model `m` over the table (and n_random random operands); returns the failures found."""
    fails = []

    def expect(name, got, want, args, canonical=True):
        got = [int(v) for v in got]
        for i, (g, w) in enumerate(zip(got, want)):
            if (g != w) if canonical else (g % P != w % P or not 0 <= g < 2**64):
                fails.append("%s%r = %d, want %d" % (name, tuple(a[i] for a in args), g, w))
                return

    ra, rb = random_operands(n_random)
    rca, rcb = [x % P for x in ra], [x % P for x in rb]
    any_a, any_b = _pairs(G.ANY_U64, G.ANY_U64)
    any_a, any_b = any_a + ra, any_b + rb
    can_a, can_b = _pairs(G.CLASSES, G.CLASSES)
    can_a, can_b = can_a + rca, can_b + rcb
    t_a = [a for a, b, _ in G.TARGETED.values()]
    t_b = [b for a, b, _ in G.TARGETED.values()]

    xs = G.ANY_U64 + ra
    expect("canon", m.canon(xs), [x % P for x in xs], (xs,))
    # add_lazy: a any u64, b canonical; sub_lazy: a any u64, b in [0, p] (gl::add passes p - b, which is p when b = 0)
    la, lb = _pairs(G.ANY_U64, G.CLASSES + [P])
    la, lb = la + ra, lb + rcb
    lb_c = [b % P for b in lb]
    expect("add_lazy", m.add_lazy(la, lb_c), [(a + b) % P for a, b in zip(la, lb_c)], (la, lb_c), canonical=False)
    expect("sub_lazy", m.sub_lazy(la, lb), [(a - b) % P for a, b in zip(la, lb)], (la, lb), canonical=False)
    # canonical a, b: gl::add / gl::sub (= gf::add / gf::sub, the same code) are canonical
    expect("add", m.add(can_a, can_b), [(a + b) % P for a, b in zip(can_a, can_b)], (can_a, can_b))
    expect("sub", m.sub(can_a, can_b), [(a - b) % P for a, b in zip(can_a, can_b)], (can_a, can_b))
    cs = G.CLASSES + rca
    expect("neg", m.neg(cs), [-x % P for x in cs], (cs,))
    expect("halve", m.halve(cs), [x * (P + 1) // 2 % P for x in cs], (cs,))
    expect("mul7", m.mul7(cs), [7 * x % P for x in cs], (cs,))
    # 128-bit operands: lo and hi any u64
    expect("reduce128_lazy", m.reduce128_lazy(any_a, any_b), [(lo + (hi << 64)) % P for lo, hi in zip(any_a, any_b)],
           (any_a, any_b), canonical=False)
    expect("gf::reduce128", m.reduce128(any_a, any_b), [(lo + (hi << 64)) % P for lo, hi in zip(any_a, any_b)],
           (any_a, any_b))
    ma, mb = any_a + t_a, any_b + t_b
    expect("mul", m.mul(ma, mb), [a * b % P for a, b in zip(ma, mb)], (ma, mb))
    expect("mul_lazy", m.mul_lazy(ma, mb), [a * b % P for a, b in zip(ma, mb)], (ma, mb), canonical=False)
    expect("sqr", m.sqr(xs), [x * x % P for x in xs], (xs,))
    for e in POW_EXPONENTS:
        expect("pow(., %d)" % e, m.pow(G.ANY_U64, e), [pow(x, e, P) for x in G.ANY_U64], (G.ANY_U64,))
    expect("inv", m.inv(G.CLASSES), [pow(x, P - 2, P) for x in G.CLASSES], (G.CLASSES,))  # inv(0) = 0
    mp = G.ANY_U64 + ra[:2000]
    for e in range(1, 96):
        expect("mul_pow2(., %d)" % e, m.mul_pow2(mp, e), [(x << e) % P for x in mp], (mp,))
    for e in range(96):
        if m.pow2_mod_p(e) != pow(2, e, P):
            fails.append("pow2_mod_p(%d) = %d" % (e, m.pow2_mod_p(e)))

    # Acc160: one acc_mac on every limb state and operand pair whose exact sum fits 160 bits, then acc_reduce
    sa, sb = _pairs(G.CLASSES, G.CLASSES)
    lanes = [(s, a, b) for s in G.acc_states() for a, b in zip(sa, sb) if G.limbs_value(s) + a * b < 2**160]
    st = [[s[i] for s, _, _ in lanes] for i in range(5)]
    aa, bb = [a for _, a, _ in lanes], [b for _, _, b in lanes]
    out = m.acc_mac(st, aa, bb)
    want = [G.limbs_value(s) + a * b for s, a, b in lanes]
    got = [sum(int(out[i][k]) << (32 * i) for i in range(5)) for k in range(len(lanes))]
    for k in range(len(lanes)):
        if got[k] != want[k]:
            fails.append("acc_mac(%r, %d, %d) = %d, want %d" % (lanes[k] + (got[k], want[k])))
            break
    states = G.acc_states()
    expect("acc_reduce", m.acc_reduce([[s[i] for s in states] for i in range(5)]), [G.limbs_value(s) % P for s in states],
           (states,))

    # extension field
    ea, eb = _pairs(G.E2_TABLE, G.E2_TABLE)
    xa, ya = [x[0] for x in ea], [y[0] for y in eb]
    xb, yb = [x[1] for x in ea], [y[1] for y in eb]
    for name, ref in (("e2_add", nv.e_add), ("e2_sub", nv.e_sub), ("e2_mul", nv.e_mul)):
        r = getattr(m, name)((xa, xb), (ya, yb))
        want = [ref(x, y) for x, y in zip(ea, eb)]
        expect(name + "[0]", r[0], [w[0] for w in want], (ea, eb))
        expect(name + "[1]", r[1], [w[1] for w in want], (ea, eb))
    r = m.e2_mul_base((xa, xb), ya)
    expect("e2_mul_base[0]", r[0], [x[0] * y[0] % P for x, y in zip(ea, eb)], (ea, eb))
    expect("e2_mul_base[1]", r[1], [x[1] * y[0] % P for x, y in zip(ea, eb)], (ea, eb))
    r = m.e2_inv(([x[0] for x in G.E2_TABLE], [x[1] for x in G.E2_TABLE]))
    want = [nv.e_inv(x) for x in G.E2_TABLE]  # (0, 0) -> (0, 0), as inv(0) = 0
    expect("e2_inv[0]", r[0], [w[0] for w in want], (G.E2_TABLE,))
    expect("e2_inv[1]", r[1], [w[1] for w in want], (G.E2_TABLE,))
    return fails


@pytest.fixture(scope="module")
def model():
    m = G.GlModel()
    m.failures = check_all(m, N_RANDOM)
    return m


def test_asm_blocks_are_read_from_gl_cuh():
    m = G.GlModel()
    assert sorted(m.blocks) == sorted(["canon", "add_lazy", "sub_lazy", "reduce128_lazy", "reduce128", "acc_mac"])
    # gl.cuh holds all inline asm of the proving path: the model covers every asm block a proof runs. peaks.cu's asm is
    # the integer-pipe peak microbenchmark, which computes nothing a proof uses.
    csrc = os.path.dirname(G.GL_CUH)
    for f in os.listdir(csrc):
        if f not in ("gl.cuh", "peaks.cu"):
            with open(os.path.join(csrc, f)) as fh:
                assert not re.search(r"\basm\s*(volatile\s*)?\(", fh.read()), f


def test_primitives_match_python_ints(model):
    assert not model.failures, "\n".join(model.failures[:20])


def test_targeted_pairs_reach_their_outcome():
    for name, (a, b, (blk, idx, val)) in G.TARGETED.items():
        assert a < P and b < P
        m = G.GlModel()
        m.mul([a], [b])
        assert m.coverage[(blk, idx)] == {val}, name


def test_every_carry_is_driven_both_ways(model, capsys):
    rows, bad = [], []
    for blk, idx, text in model.chain_insns():
        seen = model.coverage.get((blk, idx), set())
        claim = CLAIMED_NEVER.get((blk, idx, text))
        if seen == {0, 1} and claim is None:
            state = "both"
        elif seen == {0} and claim is not None:
            state = "never (claimed by comment)"
        else:
            state = "FAIL: seen %s%s" % (sorted(seen), ", claimed never" if claim else "")
            bad.append((blk, idx, text))
        rows.append("%-15s %3d  %-40s %s" % (blk, idx, text, state))
    with capsys.disabled():
        print("\ncarry / borrow coverage of gl.cuh's asm blocks:\n" + "\n".join(rows))
    assert not bad, bad
    # every claim names an instruction that exists
    assert set(CLAIMED_NEVER) <= set(model.chain_insns())


def test_acc160_bound():
    """2^32 terms of at most (p - 1)^2 fit the 160-bit accumulator."""
    assert 2**32 * (P - 1)**2 < 2**160
    # and the limb states used above with l4 = 0xffffffff include ones every product still fits
    assert any(G.limbs_value(s) + (P - 1)**2 < 2**160 for s in G.acc_states() if s[4] == G.M32)


def test_unknown_opcode_is_an_error():
    with open(G.GL_CUH) as f:
        src = f.read()
    m = G.GlModel(src.replace("neg.s32 k, k;", "neg.s64 k, k;", 1))
    with pytest.raises(ValueError, match="not modelled"):
        m.canon([5])


def _insn_lines(src):
    """the lines of `src` and the indices of those holding one instruction of an asm template (`.reg` lines excluded)"""
    lines = src.split("\n")
    return lines, [i for i, ln in enumerate(lines) if re.match(r'\s*"[a-z]', ln)]


def _in_place(line):
    """An instruction that updates a register in place (its destination is also a source): running it twice is a change."""
    op, _, rest = re.search(r'"([^"]*);', line).group(1).strip().partition(" ")
    ops = G._split_operands(rest)
    return ops[0] in ops[1:]


# Deleting this instruction gives an equivalent program: gf::reduce128's `r >= p` test then reads r before the "+ eps on
# carry" fix-up, and the two differ only when that carry is 1, where r < p before and after the fix-up.
EQUIVALENT_DELETIONS = {"mov.b64 {r0, r1}, rr"}


def _fails(src):
    try:
        return bool(check_all(G.GlModel(src), 0))
    except ValueError:
        return True


def test_model_follows_the_source():
    """Deleting any instruction of gl.cuh's asm, or repeating any that updates a register in place, makes the check above
    fail: the model reads gl.cuh and is not a copy of it."""
    with open(G.GL_CUH) as f:
        src = f.read()
    lines, idx = _insn_lines(src)
    assert len(idx) == sum(len([op for op, _, _ in b.insns if op != ".reg"]) for b in G.parse_blocks(src).values())
    survivors = []
    for i in idx:
        equivalent = re.search(r'"([^"]*);', lines[i]).group(1).strip() in EQUIVALENT_DELETIONS
        if _fails("\n".join(lines[:i] + lines[i + 1:])) == equivalent:
            survivors.append(("deleted", lines[i].strip(), "equivalent" if equivalent else ""))
        if _in_place(lines[i]) and not _fails("\n".join(lines[:i + 1] + [lines[i]] + lines[i + 1:])):
            survivors.append(("repeated", lines[i].strip()))
    assert not survivors, survivors
