"""A model of multi_stark_b200/csrc/gl.cuh that runs the file's own inline PTX.

Every `asm("...")` block of gl.cuh is read from the source text and interpreted instruction by instruction over Python
ints, vectorised as numpy object arrays (one lane per operand). Operands are bound by name through each block's
constraint list, so the model follows the source: an instruction added, removed or edited in gl.cuh changes what the
model computes. An opcode the interpreter does not know is an error.

For every instruction that computes a carry or borrow the model records which values it took, per block and instruction
index: the flag written by a `.cc` instruction, and the carry-out that a chain's last `addc` / `subc` (or a 64-bit
`mad.wide`) drops. The C++ around the asm (mul_pow2, add = sub_lazy(a, p - b), halve, neg, mul7, the e2 functions,
acc_reduce, ...) is transcribed below as plain Python over the interpreted blocks."""
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GL_CUH = os.path.join(ROOT, "multi_stark_b200", "csrc", "gl.cuh")

P = 2**64 - 2**32 + 1
EPS = 2**32 - 1
M32 = 2**32 - 1
M64 = 2**64 - 1


class AsmBlock:
    """One asm statement: its function, instruction list and operand constraints."""

    def __init__(self, func, text, outputs, inputs):
        self.func = func
        self.outputs = outputs  # [(constraint, C expression)], operands %0 .. in order
        self.inputs = inputs
        self.operands = outputs + inputs
        self.insns = []  # (opcode, [operand tokens], source text), `.reg` declarations included
        for stmt in re.split(r"[;\n]", text):
            stmt = stmt.strip().strip("{}").strip()
            if not stmt:
                continue
            op, _, rest = stmt.partition(" ")
            self.insns.append((op, _split_operands(rest), stmt))


def _split_operands(s):
    out, depth, cur = [], 0, ""
    for ch in s:
        if ch == "," and depth == 0:
            out.append(cur.strip())
            cur = ""
            continue
        depth += ch == "{"
        depth -= ch == "}"
        cur += ch
    if cur.strip():
        out.append(cur.strip())
    return out


def _string_literal(src, i):
    """Decode the C string literal starting at src[i] == '"'; returns (text, index after the closing quote)."""
    out, i = [], i + 1
    esc = {"n": "\n", "t": "\t", '"': '"', "\\": "\\"}
    while src[i] != '"':
        if src[i] == "\\":
            out.append(esc[src[i + 1]])
            i += 2
        else:
            out.append(src[i])
            i += 1
    return "".join(out), i + 1


def parse_blocks(src):
    """{function name: AsmBlock} for every asm statement of `src` (the text of gl.cuh)."""
    funcs = [(m.start(), m.group(1)) for m in re.finditer(r"__device__\s+__forceinline__\s+[\w:]+\s+(\w+)\s*\(", src)]
    blocks = {}
    for m in re.finditer(r"\basm\s*(?:volatile\s*)?\(", src):
        i = m.end()
        parts = []
        while True:  # the template: string literals, whitespace and // comments up to the first ':'
            while src[i].isspace():
                i += 1
            if src.startswith("//", i):
                i = src.index("\n", i)
            elif src[i] == '"':
                s, i = _string_literal(src, i)
                parts.append(s)
            elif src[i] == ":":
                break
            else:
                raise ValueError("unexpected %r in asm template at offset %d" % (src[i], i))
        depth, j = 1, i
        while depth:
            if src[j] == '"':
                j = _string_literal(src, j)[1]
                continue
            depth += src[j] == "("
            depth -= src[j] == ")"
            j += 1
        sections = src[i + 1:j - 1].split(":")
        cons = [re.findall(r'"([^"]*)"\s*\(([^()]*)\)', s) for s in sections[:2]]
        func = [name for pos, name in funcs if pos < m.start()][-1]
        if func in blocks:
            raise ValueError("two asm blocks in %s" % func)
        outputs, inputs = ([(c, e.strip()) for c, e in sec] for sec in cons)
        blocks[func] = AsmBlock(func, "".join(parts), outputs, inputs)
    return blocks


def _arr(x):
    """Python int or sequence -> 1-D numpy object array of Python ints."""
    if isinstance(x, np.ndarray) and x.dtype == object and x.ndim == 1:
        return x
    a = np.empty(np.size(x) if np.ndim(x) else 1, dtype=object)
    a[:] = [int(v) for v in np.ravel(np.asarray(x, dtype=object))]
    return a


def _lit(tok):
    return int(tok, 16) if tok.lower().startswith("0x") else int(tok)


class GlModel:
    """The primitives of gl.cuh, with their asm interpreted from `src` (default: the text of gl.cuh)."""

    def __init__(self, src=None):
        if src is None:
            with open(GL_CUH) as f:
                src = f.read()
        self.blocks = parse_blocks(src)
        self.coverage = {}  # (block, instruction index) -> set of carry / borrow values seen

    # ---- the interpreter -------------------------------------------------------------------------------------------------
    def run(self, name, env):
        """Run block `name` with C variables from `env` (name -> int array), return {C expression: array} of its outputs."""
        blk = self.blocks[name]
        regs, width = {}, {}
        n = max(len(v) for v in env.values())
        for k, (con, expr) in enumerate(blk.operands):
            w = 64 if "l" in con else 32
            width["%%%d" % k] = w
            if not con.startswith("="):  # "+r" and inputs are read
                v = _arr(env[expr]) if np.ndim(env[expr]) else _arr([env[expr]] * n)
                if any(x >> w for x in v):
                    raise ValueError("%s: operand %s = %r does not fit %d bits" % (name, expr, v, w))
                regs["%%%d" % k] = v
        cf = None

        def get(tok):
            if tok in regs:
                return regs[tok]
            if tok in width:
                raise ValueError("%s: register %s read before it is written" % (name, tok))
            if re.fullmatch(r"0x[0-9a-fA-F]+|\d+", tok):
                return _arr([_lit(tok)] * n)
            raise ValueError("%s: unknown operand %r" % (name, tok))

        def put(tok, v):
            if tok not in width:
                raise ValueError("%s: undeclared register %r" % (name, tok))
            regs[tok] = v & ((1 << width[tok]) - 1)

        def record(idx, v):
            self.coverage.setdefault((name, idx), set()).update(int(x) for x in set(v))

        def carry_in():
            if cf is None:
                raise ValueError("%s: carry flag read before a .cc instruction set it" % name)
            return cf

        for idx, (op, ops, text) in enumerate(blk.insns):
            if op == ".reg":
                ty = ops[0].split()[0]
                names = [ops[0].split()[1]] + ops[1:]
                for r in names:
                    if r in width:
                        raise ValueError("%s: register %s declared twice" % (name, r))
                    width[r] = {".u32": 32, ".u64": 64}[ty]
                continue
            base = op.split(".")
            if op in ("add.cc.u32", "addc.cc.u32", "addc.u32", "sub.cc.u32", "subc.cc.u32", "subc.u32"):
                d, a, b = ops
                cin = carry_in() if base[0] in ("addc", "subc") else 0
                if base[0].startswith("add"):
                    s = get(a) + get(b) + cin
                    c = s >> 32
                else:
                    s = get(a) - get(b) - cin
                    c = -(s >> 32)  # s >= -2^32: 1 on borrow
                put(d, s)
                if (a, b) != ("0", "0"):  # `addc k, 0, 0` / `subc m, 0, 0` only read the flag
                    record(idx, c)
                if ".cc" in op:
                    cf = c
            elif op in ("mad.lo.cc.u32", "madc.lo.cc.u32", "madc.hi.cc.u32"):
                d, a, b, c_ = ops
                pr = get(a) * get(b)
                pr = pr & M32 if base[1] == "lo" else pr >> 32
                s = pr + get(c_) + (carry_in() if base[0] == "madc" else 0)
                put(d, s)
                record(idx, s >> 32)
                if ".cc" in op:
                    cf = s >> 32
            elif op == "mad.wide.u32":
                d, a, b, c_ = ops
                s = get(a) * get(b) + get(c_)
                put(d, s)
                record(idx, s >> 64)
            elif op == "neg.s32":
                d, a = ops
                put(d, -get(a))
            elif op == "mov.b64":
                d, a = ops
                if a.startswith("{"):
                    lo, hi = [t.strip() for t in a.strip("{}").split(",")]
                    put(d, get(lo) | (get(hi) << 32))
                elif d.startswith("{"):
                    lo, hi = [t.strip() for t in d.strip("{}").split(",")]
                    v = get(a)
                    put(lo, v & M32)
                    put(hi, v >> 32)
                else:
                    raise ValueError("%s: mov.b64 %r is neither a pack nor an unpack" % (name, text))
            else:
                raise ValueError("%s: opcode %r (in %r) is not modelled" % (name, op, text))
        out = {}
        for k, (con, expr) in enumerate(blk.outputs):
            out[expr] = get("%%%d" % k)
        return out

    def chain_insns(self):
        """[(block, index, text)] of every instruction that computes a carry or borrow (the keys of `coverage`)."""
        return [(b.func, i, t) for b in self.blocks.values() for i, (op, ops, t) in enumerate(b.insns)
                if op.split(".")[0] in ("add", "addc", "sub", "subc", "mad", "madc") and ops[1:] != ["0", "0"]]

    # ---- the C++ around the asm, transcribed -----------------------------------------------------------------------------
    def canon(self, x):
        x = _arr(x)
        o = self.run("canon", {"x0": x & M32, "x1": x >> 32})
        return o["r0"] | (o["r1"] << 32)

    def add_lazy(self, a, b):
        a, b = _arr(a), _arr(b)
        o = self.run("add_lazy", {"a0": a & M32, "a1": a >> 32, "b0": b & M32, "b1": b >> 32})
        return o["r0"] | (o["r1"] << 32)

    def sub_lazy(self, a, b):
        a, b = _arr(a), _arr(b)
        o = self.run("sub_lazy", {"a0": a & M32, "a1": a >> 32, "b0": b & M32, "b1": b >> 32})
        return o["r0"] | (o["r1"] << 32)

    def add(self, a, b):
        return self.sub_lazy(a, (P - _arr(b)) & M64)

    def sub(self, a, b):
        return self.sub_lazy(a, b)

    @staticmethod
    def neg(a):
        a = _arr(a)
        return np.where(a != 0, (P - a) & M64, 0).astype(object)

    def reduce128_lazy(self, lo, hi):
        lo, hi = _arr(lo), _arr(hi)
        o = self.run("reduce128_lazy", {"l0": lo & M32, "l1": lo >> 32, "hl": hi & M32, "hh": hi >> 32})
        return o["r0"] | (o["r1"] << 32)

    def reduce128(self, lo, hi):
        """gf::reduce128"""
        lo, hi = _arr(lo), _arr(hi)
        return self.run("reduce128", {"l0": lo & M32, "l1": lo >> 32, "h0": hi & M32, "h1": hi >> 32})["r"]

    def mul(self, a, b):
        """gl::mul and gf::mul (the same code: the 128-bit product through gf::reduce128)"""
        pr = _arr(a) * _arr(b)
        return self.reduce128(pr & M64, pr >> 64)

    def mul_lazy(self, a, b):
        pr = _arr(a) * _arr(b)
        return self.reduce128_lazy(pr & M64, pr >> 64)

    def sqr(self, a):
        return self.mul(a, a)

    def pow(self, a, e):
        acc, a = _arr([1] * len(_arr(a))), _arr(a)
        while e:
            if e & 1:
                acc = self.mul(acc, a)
            a = self.sqr(a)
            e >>= 1
        return acc

    def inv(self, a):
        return self.pow(a, P - 2)

    @staticmethod
    def halve(a):
        a = _arr(a)
        return np.where((a & 1) == 1, (a >> 1) + (P >> 1) + 1, a >> 1).astype(object)

    @staticmethod
    def pow2_mod_p(e):
        return (1 << e) if e < 64 else ((1 << (e - 32)) - (1 << (e - 64)))

    def mul_pow2(self, x, e):
        """gf::mul_pow2 for 0 < e < 96"""
        assert 0 < e < 96
        x = _arr(x)
        q, r = e // 32, e % 32
        x0, x1 = x & M32, x >> 32
        if r == 0:
            y0, y1, y2 = x0, x1, x0 * 0
        else:
            y0 = (x0 << r) & M32
            y1 = ((x1 << r) | (x0 >> (32 - r))) & M32  # __funnelshift_l(x0, x1, r)
            y2 = x1 >> (32 - r)
        if q == 2:
            return self.sub_lazy(y0 * EPS, (y2 << 32) | y1)
        if q == 0:
            return self.sub_lazy((y1 << 32) | y0, P - y2 * EPS)
        return self.sub_lazy(self.sub_lazy(y0 << 32, y2), P - y1 * EPS)

    def acc_mac(self, s, a, b):
        """s: the five limbs (l0 .. l4) as arrays; returns the new limbs."""
        a, b = _arr(a), _arr(b)
        env = {"s.l%d" % i: _arr(s[i]) for i in range(5)}
        env.update({"a0": a & M32, "a1": a >> 32, "b0": b & M32, "b1": b >> 32})
        o = self.run("acc_mac", env)
        return tuple(o["s.l%d" % i] for i in range(5))

    def acc_reduce(self, s):
        s = [_arr(v) for v in s]
        r = self.reduce128(s[0] | (s[1] << 32), s[2] | (s[3] << 32))
        return self.sub_lazy(r, s[4] << 32)

    # extension field F_p[X]/(X^2 - 7); an element is a pair of arrays (a, b) = a + b X
    def mul7(self, x):
        x2 = self.add(x, x)
        x4 = self.add(x2, x2)
        return self.sub(self.add(x4, x4), x)

    def e2_add(self, x, y):
        return self.add(x[0], y[0]), self.add(x[1], y[1])

    def e2_sub(self, x, y):
        return self.sub(x[0], y[0]), self.sub(x[1], y[1])

    def e2_mul(self, x, y):
        v0, v1 = self.mul(x[0], y[0]), self.mul(x[1], y[1])
        cross = self.sub(self.sub(self.mul(self.add(x[0], x[1]), self.add(y[0], y[1])), v0), v1)
        return self.add(v0, self.mul7(v1)), cross

    def e2_mul_base(self, x, s):
        return self.mul(x[0], s), self.mul(x[1], s)

    def e2_inv(self, x):
        norm = self.sub(self.sqr(x[0]), self.mul7(self.sqr(x[1])))
        ni = self.inv(norm)
        return self.mul(x[0], ni), self.mul(self.neg(x[1]), ni)


# ---- the operand table shared by the field tests ---------------------------------------------------------------------------
# Canonical edge classes, then the non-canonical values that only "any u64" operands may take.
CLASSES = sorted({0, 1, 2, 7, 2**32 - 2, 2**32 - 1, 2**32, 2**32 + 1, 2**63 - 1, 2**63, (P - 1) // 2, (P + 1) // 2, P - 2,
                  P - 1, 0xFFFFFFFF << 32, 0xFFFFFFFF})
NONCANON = [P, P + 1, P + 2**32 - 2, 2**64 - 2, 2**64 - 1]
ANY_U64 = CLASSES + NONCANON
# Pairs the cross product of the table does not reach with canonical operands of gl::mul, each with the outcome it reaches
# (block, instruction index, carry): the products 2^64 - 1 and 2^65 - 2^32 reduce to r = 2^64 - 1 >= p before
# gf::reduce128's final fix-up.
TARGETED = {
    "mul (2^32 + 1)(2^32 - 1) = 2^64 - 1": (2**32 + 1, 2**32 - 1, ("reduce128", 14, 1)),
    "mul 2^32 (2^33 - 1) = 2^65 - 2^32": (2**32, 2**33 - 1, ("reduce128", 14, 1)),
}


def _sqrt(n):
    """a square root of n mod p (Tonelli-Shanks), or None"""
    n %= P
    if n == 0:
        return 0
    if pow(n, (P - 1) // 2, P) != 1:
        return None
    q, s = P - 1, 0
    while q % 2 == 0:
        q, s = q // 2, s + 1
    z = 7  # a non-residue
    m, c, t, r = s, pow(z, q, P), pow(n, q, P), pow(n, (q + 1) // 2, P)
    while t != 1:
        i, t2 = 0, t
        while t2 != 1:
            t2, i = t2 * t2 % P, i + 1
        b = pow(c, 1 << (m - i - 1), P)
        m, c, t, r = i, b * b % P, t * b * b % P, r * b % P
    return r


def _with_norm(n):
    """an element a + bX with a^2 - 7 b^2 = n, b != 0"""
    for b in range(1, 100):
        a = _sqrt(n + 7 * b * b)
        if a is not None:
            return (a, b)
    raise AssertionError(n)


# Extension-field operands: zero, (c, 0), (0, c) for every class, and elements whose norm a^2 - 7 b^2 is an edge value.
E2_NORMS = [1, 2, P - 1, P - 2, 2**32 - 1, 2**32, 2**63, (P - 1) // 2]
E2_TABLE = sorted({(0, 0)} | {(c, 0) for c in CLASSES} | {(0, c) for c in CLASSES} | {_with_norm(n) for n in E2_NORMS})


def acc_states(seed=5):
    """160-bit limb states (l0 .. l4) of an Acc160: every pattern of 0 / 0xffffffff in l0 .. l3 (so that each carry chain of
    acc_mac can run into l4) and seeded random low limbs, each with l4 = 0, 1 and 0xffffffff."""
    rng = np.random.default_rng(seed)
    lows = [tuple(M32 * ((k >> i) & 1) for i in range(4)) for k in range(16)]
    lows += [tuple(int(v) for v in rng.integers(0, 2**32, size=4)) for _ in range(4)]
    return [low + (l4,) for l4 in (0, 1, M32) for low in lows]


def limbs_value(s):
    return sum(int(v) << (32 * i) for i, v in enumerate(s))
