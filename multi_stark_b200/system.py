"""Host-side system objects: mirror of the reference's `System` / `Circuit` (src/system.rs:52-203) and of
the benchmark workload (benches/multi_stark.rs:171-238), over libmshost.so; plus the device programs
(`msgpu_program`) compiled from each circuit's ConstraintGraph."""
import ctypes as C

import numpy as np

from . import _ffi
from ._ffi import check

INFO_FIELDS = ["main_width", "pre_width", "pre_height", "num_lookups", "stage2_width", "constraint_count",
               "max_constraint_degree", "quotient_degree", "n_nodes", "n_zeros", "lookup_prefix_len", "preprocessed_index"]


class GraphDescC(C.Structure):
    """`msgpu_graph_desc` (include/msgpu.h)."""
    _fields_ = [("n_nodes", C.c_uint32), ("op", C.c_void_p), ("a", C.c_void_p), ("b", C.c_void_p), ("imm", C.c_void_p),
                ("n_zeros", C.c_uint32), ("zeros", C.c_void_p), ("n_lookups", C.c_uint32), ("lookup_mult", C.c_void_p),
                ("lookup_arg_off", C.c_void_p), ("lookup_args", C.c_void_p), ("lookup_prefix_len", C.c_uint32),
                ("pre_width", C.c_uint32), ("main_width", C.c_uint32), ("stage2_width", C.c_uint32)]


OPS = {"const": 0, "var": 1, "public": 2, "first": 3, "last": 4, "trans": 5, "add": 6, "sub": 7, "mul": 8, "neg": 9}


def graph_descs(graphs):
    """Compiled circuits -> (ctypes array of msgpu_graph_desc, keep-alive list). A graph is a dict with
    nodes: [("const", v) | ("var", source, offset, index) | ("public", i) | ("first",) | ("last",) | ("trans",) |
            ("add" | "sub" | "mul", a, b) | ("neg", a)]  (the reference's `Node`, src/graph.rs:35-46),
    zeros: sorted root ids, lookups: [(multiplicity id, [argument ids])], lookup_prefix_len, main_width, pre_width."""
    arr = (GraphDescC * len(graphs))()
    keep = []
    for i, g in enumerate(graphs):
        n = len(g["nodes"])
        op = np.zeros(max(n, 1), dtype=np.uint8)
        a = np.zeros(max(n, 1), dtype=np.uint32)
        b = np.zeros(max(n, 1), dtype=np.uint32)
        imm = np.zeros(max(n, 1), dtype=np.uint64)
        for k, nd in enumerate(g["nodes"]):
            op[k] = OPS[nd[0]]
            if nd[0] == "const":
                imm[k] = nd[1]
            elif nd[0] == "var":
                a[k], b[k] = nd[1] | (nd[2] << 2), nd[3]
            elif nd[0] in ("public", "neg"):
                a[k] = nd[1]
            elif nd[0] in ("add", "sub", "mul"):
                a[k], b[k] = nd[1], nd[2]
        zeros = np.array(list(g["zeros"]) or [0], dtype=np.uint32)
        lm = np.array([m for m, _ in g["lookups"]] or [0], dtype=np.uint32)
        off = np.zeros(len(g["lookups"]) + 1, dtype=np.uint32)
        args = []
        for j, (_, ar) in enumerate(g["lookups"]):
            args += list(ar)
            off[j + 1] = len(args)
        la = np.array(args or [0], dtype=np.uint32)
        keep += [op, a, b, imm, zeros, lm, off, la]
        d = arr[i]
        d.n_nodes, d.op, d.a, d.b, d.imm = n, op.ctypes.data, a.ctypes.data, b.ctypes.data, imm.ctypes.data
        d.n_zeros, d.zeros = len(g["zeros"]), zeros.ctypes.data
        d.n_lookups, d.lookup_mult, d.lookup_arg_off, d.lookup_args = len(g["lookups"]), lm.ctypes.data, off.ctypes.data, la.ctypes.data
        d.lookup_prefix_len = g["lookup_prefix_len"]
        d.pre_width, d.main_width = g.get("pre_width", 0), g["main_width"]
        d.stage2_width = max(len(g["lookups"]), 1) * 2
    return arr, keep


class System:
    """The reference's `System` (src/system.rs:52-203) on the host side: a named benchmark system (named_system_inputs in
    host/system.hpp: "u32_add", "mixed", "fib", "wide:W", "multi:K") or, with `System.from_graphs`, any circuits the caller
    compiled itself."""

    def __init__(self, kind, log_blowup=1, log_final_poly_len=0, max_log_arity=1, num_queries=100, commit_pow_bits=0,
                 query_pow_bits=0, _graphs=None, _preprocessed=None):
        self.H = _ffi.host_lib()
        self.kind = kind
        self.params = dict(log_blowup=log_blowup, log_final_poly_len=log_final_poly_len, max_log_arity=max_log_arity,
                           num_queries=num_queries, commit_pow_bits=commit_pow_bits, query_pow_bits=query_pow_bits)
        if _graphs is None:
            self.h = self.H.msh_system_create(kind.encode(), log_blowup, log_final_poly_len, max_log_arity, num_queries,
                                              commit_pow_bits, query_pow_bits)
        else:
            arr, keep = graph_descs(_graphs)
            pre = [None if p is None else np.ascontiguousarray(p, dtype=np.uint64) for p in (_preprocessed or [None] * len(_graphs))]
            ptrs = (C.c_void_p * len(_graphs))(*[p.ctypes.data if p is not None else None for p in pre])
            hs = (C.c_uint64 * len(_graphs))(*[p.shape[0] if p is not None else 0 for p in pre])
            self.h = self.H.msh_system_create_from_graphs(C.cast(arr, C.c_void_p), len(_graphs), C.cast(ptrs, C.c_void_p),
                                                          C.cast(hs, C.c_void_p), log_blowup, log_final_poly_len, max_log_arity,
                                                          num_queries, commit_pow_bits, query_pow_bits)
        if not self.h:
            raise ValueError(_ffi.host_error(-1).message)
        self.num_circuits = int(self.H.msh_system_num_circuits(self.h))
        self.circuits = []
        for i in range(self.num_circuits):
            buf = np.zeros(12, dtype=np.uint64)
            self.H.msh_circuit_info(self.h, i, buf.ctypes.data_as(C.c_void_p))
            info = {k: int(v) for k, v in zip(INFO_FIELDS, buf)}
            if info["preprocessed_index"] == 2**64 - 1:
                info["preprocessed_index"] = None
            self.circuits.append(info)

    @classmethod
    def from_graphs(cls, graphs, preprocessed=None, **params):
        """`msh_system_create_from_graphs`: graphs as described at graph_descs(); preprocessed[i] = (height x pre_width) array
        or None."""
        return cls("graphs", _graphs=graphs, _preprocessed=preprocessed, **params)

    def preprocessed(self, i):
        c = self.circuits[i]
        out = np.zeros((c["pre_height"], c["pre_width"]), dtype=np.uint64)
        if out.size:
            self.H.msh_circuit_preprocessed(self.h, i, out.ctypes.data_as(C.c_void_p))
        return out

    def graph_desc(self, i):
        return self.H.msh_circuit_graph(self.h, i)

    def close(self):
        if getattr(self, "h", None):
            self.H.msh_system_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def u32_add_workload(num_adds):
    """(byte_trace 256x1, add_trace next_pow2(num_adds)x14, claims num_adds x 4)."""
    H = _ffi.host_lib()
    h = 1
    while h < num_adds:
        h *= 2
    byte = np.zeros((256, 1), dtype=np.uint64)
    add = np.zeros((h, 14), dtype=np.uint64)
    claims = np.zeros((num_adds, 4), dtype=np.uint64)
    H.msh_u32add_workload(num_adds, byte.ctypes.data_as(C.c_void_p), add.ctypes.data_as(C.c_void_p),
                          claims.ctypes.data_as(C.c_void_p))
    return byte, add, claims


def multi_workload(log_heights):
    """Workload of the "multi:K" system (BASELINE configs[3]): circuit 0 = the byte table, circuit 1 + k = a U32-add circuit
    with 2^log_heights[k] additions from its own xorshift32 streams. Returns (traces [byte, add_0, ...], claims (n, 4));
    the byte multiplicities are summed over the K circuits."""
    H = _ffi.host_lib()
    byte_total = np.zeros((256, 1), dtype=np.uint64)
    traces, claims = [], []
    for k, lh in enumerate(log_heights):
        n = 1 << lh
        byte = np.zeros((256, 1), dtype=np.uint64)
        add = np.zeros((n, 14), dtype=np.uint64)
        cl = np.zeros((n, 4), dtype=np.uint64)
        H.msh_u32add_workload_seeded(n, (0xDEADBEEF + 0x9E3779B9 * k) & 0xFFFFFFFF or 1, (0xCAFEBABE + 0x85EBCA6B * k) & 0xFFFFFFFF or 1,
                                     byte.ctypes.data_as(C.c_void_p), add.ctypes.data_as(C.c_void_p), cl.ctypes.data_as(C.c_void_p))
        byte_total += byte
        traces.append(add)
        claims.append(cl)
    return [byte_total] + traces, np.concatenate(claims, axis=0)


def fib_trace(rows):
    H = _ffi.host_lib()
    out = np.zeros((rows, 3), dtype=np.uint64)
    H.msh_fib_trace(rows, out.ctypes.data_as(C.c_void_p))
    return out


def wide_trace(rows, width, row0=0, out=None):
    """Trace of the "wide:W" system (BASELINE configs[2]): column 2k = splitmix64(row * W + 2k) mod p, column 2k+1 its cube."""
    H = _ffi.host_lib()
    if out is None:
        out = np.zeros((rows, width), dtype=np.uint64)
    H.msh_wide_trace(row0, rows, width, out.ctypes.data_as(C.c_void_p))
    return out


class Program:
    """Device bytecode of one circuit (`msgpu_program`)."""

    def __init__(self, ctx, system, circuit_index):
        self.ctx = ctx
        self.L = ctx.L
        self.info = system.circuits[circuit_index]
        h = C.c_void_p()
        check(self.L.msgpu_program_create(ctx.h, system.graph_desc(circuit_index), C.byref(h)))
        self.h = h

    def free(self):
        if getattr(self, "h", None):
            self.L.msgpu_program_free(self.h)
            self.h = None

    def __del__(self):
        try:
            if self.ctx.h:
                self.free()
        except Exception:
            pass

    def stage2_trace(self, main_dev, rows, beta, gamma, pre_dev=None):
        """msgpu_stage2_trace: returns (device ptr of rows x stage2_width, local_sum[2])."""
        w = self.info["stage2_width"]
        out = self.ctx.malloc(max(rows * w * 8, 8))
        b = np.asarray(beta, dtype=np.uint64)
        g = np.asarray(gamma, dtype=np.uint64)
        ls = np.zeros(2, dtype=np.uint64)
        check(self.L.msgpu_stage2_trace(self.ctx.h, self.h, C.c_void_p(pre_dev) if pre_dev else None, C.c_void_p(main_dev), rows,
                                        b.ctypes.data_as(C.c_void_p), g.ctypes.data_as(C.c_void_p), C.c_void_p(out),
                                        ls.ctypes.data_as(C.c_void_p)))
        return out, ls

    def quotient(self, pd_pre, idx_pre, pd_s1, idx_s1, pd_s2, idx_s2, log_n, log_q, log_blowup, publics8, alpha,
                 want_values=False):
        """msgpu_quotient: returns (device ptr of the quotient LDE, rows, cols[, quotient values nq x 2])."""
        pub = np.asarray(publics8, dtype=np.uint64)
        al = np.asarray(alpha, dtype=np.uint64)
        lde = C.c_void_p()
        nq = 1 << (log_n + log_q)
        vals = np.zeros((nq, 2), dtype=np.uint64) if want_values else None
        check(self.L.msgpu_quotient(self.ctx.h, self.h, pd_pre.h if pd_pre is not None else None, idx_pre, pd_s1.h, idx_s1,
                                    pd_s2.h, idx_s2, log_n, log_q, log_blowup, pub.ctypes.data_as(C.c_void_p),
                                    al.ctypes.data_as(C.c_void_p), C.byref(lde),
                                    vals.ctypes.data_as(C.c_void_p) if want_values else None))
        rows, cols = 1 << (log_n + log_blowup), 2 << log_q
        return (lde.value, rows, cols, vals) if want_values else (lde.value, rows, cols)


def claims_accumulator(ctx, claims, beta, gamma):
    cl = np.ascontiguousarray(claims, dtype=np.uint64)
    b = np.asarray(beta, dtype=np.uint64)
    g = np.asarray(gamma, dtype=np.uint64)
    out = np.zeros(2, dtype=np.uint64)
    check(ctx.L.msgpu_claims_accumulator(ctx.h, cl.ctypes.data_as(C.c_void_p), cl.shape[0], cl.shape[1],
                                         b.ctypes.data_as(C.c_void_p), g.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)))
    return out


def shifted_quotient_slices(ctx, m, q):
    a = np.ascontiguousarray(m, dtype=np.uint64)
    out = np.zeros((a.shape[0] // q, a.shape[1] * q), dtype=np.uint64)
    check(ctx.L.msgpu_shifted_quotient_slices(ctx.h, a.ctypes.data_as(C.c_void_p), a.shape[0], a.shape[1], q,
                                              out.ctypes.data_as(C.c_void_p)))
    return out


STAGE_NAMES = ["stark/stage1_commit", "stark/claims", "stark/stage2_commit", "stark/quotient", "stark/fri_open", "stark/prove"]


def _claims_args(claims):
    """`claims` as msh_prove takes them: (flat uint64 buffer, offsets pointer or None, stride, n_claims). A 2-D uint64
    C-contiguous array is passed without a copy and without offsets (4M claims through the offsets form = 8 ms of numpy in the
    timed prove()); other 2-D arrays are converted once; a sequence of 1-D claims goes through offsets; None = no claims."""
    if isinstance(claims, np.ndarray) and claims.ndim == 2:
        flat = claims.reshape(-1) if (claims.dtype == np.uint64 and claims.flags.c_contiguous) else \
            np.ascontiguousarray(claims, dtype=np.uint64).ravel()
        (n_claims, stride), offs_p = claims.shape, None
    else:
        claims = [] if claims is None else claims
        n_claims, stride = len(claims), 0
        offs = np.zeros(n_claims + 1, dtype=np.uint64)
        for i, c in enumerate(claims):
            offs[i + 1] = offs[i] + len(c)
        flat = np.concatenate([np.asarray(c, dtype=np.uint64).ravel() for c in claims]) if n_claims else offs[:0]
        offs_p = offs.ctypes.data_as(_ffi.c_u64p)  # the pointer keeps `offs` alive
    if flat.size == 0:
        flat = np.zeros(1, dtype=np.uint64)
    return flat, offs_p, stride, n_claims


class ProverBase:
    """What the single-GPU and the sharded provers share: an `msh_prover` made by `create(system.h, ctx.h, *args)`, its
    verifier key, and the one msh_prove call."""

    def __init__(self, ctx, system, create, *args):
        self.H = _ffi.host_lib()
        self.ctx = ctx
        self.system = system
        self.last_stage_ms = None
        self.h = create(system.h, ctx.h, *args)
        if not self.h:
            raise self._error(-3)

    def _error(self, code):
        return _ffi.host_error(code)

    def preprocessed_commit(self):
        out = np.zeros(32, dtype=np.uint8)
        return bytes(out) if self.H.msh_prover_preprocessed_commit(self.h, out.ctypes.data_as(C.c_void_p)) else None

    def _prove(self, trace_ptrs, heights, claims):
        """msh_prove: trace_ptrs[i] = host pointer of circuit i's rows (None: no rows on this rank), heights[i] = its trace rows.
        Returns `Proof::to_bytes` and sets last_stage_ms."""
        n = self.system.num_circuits
        flat, offs_p, stride, n_claims = _claims_args(claims)
        out, ln = C.c_void_p(), C.c_uint64()
        ms = (C.c_double * 6)()
        rc = self.H.msh_prove(self.h, (C.c_void_p * n)(*trace_ptrs), (C.c_uint64 * n)(*[int(h) for h in heights]),
                              flat.ctypes.data_as(_ffi.c_u64p), offs_p, stride, n_claims, C.byref(out), C.byref(ln), ms)
        if rc != 0:
            raise self._error(rc)
        data = C.string_at(out.value, ln.value)
        self.H.msh_bytes_free(out)
        self.last_stage_ms = dict(zip(STAGE_NAMES, ms))
        return data

    def close(self):
        if getattr(self, "h", None):
            self.H.msh_prover_free(self.h)
            self.h = None


class Prover(ProverBase):
    """`System::prove_multiple_claims` (src/prover.rs:289-603) on the device: the host runs the Fiat-Shamir transcript
    (host/prover.hpp, host/pcs.hpp); every matrix stays in HBM between the LDE, Merkle, quotient and opening stages."""

    def __init__(self, ctx, system):
        super().__init__(ctx, system, _ffi.host_lib().msh_prover_create)

    def prove(self, traces, claims):
        """traces: one (h x main_width) uint64 array per circuit (h = 0 deactivates the circuit);
        claims: (n, len) uint64 array or sequence of 1-D uint64 arrays. Returns `Proof::to_bytes`."""
        mats = [np.ascontiguousarray(t, dtype=np.uint64) for t in traces]
        if len(mats) != self.system.num_circuits:
            raise _ffi.MsgpuError(-1, "expected one trace per circuit")
        for m, info in zip(mats, self.system.circuits):
            if m.ndim != 2 or (m.shape[0] and m.shape[1] != info["main_width"]):
                raise _ffi.MsgpuError(-1, "trace width does not match the circuit")
        return self._prove([m.ctypes.data if m.size else None for m in mats], [m.shape[0] for m in mats], claims)

    def last_transcript(self):
        """Test hook: (challenges [(c0, c1)...] = beta, gamma, alpha, zeta, alpha_pcs, FRI betas; query indices) of the last
        prove() on this thread."""
        ch = np.zeros(2 * 128, dtype=np.uint64)
        idx = np.zeros(4096, dtype=np.uint64)
        nidx = np.zeros(1, dtype=np.uint64)
        n = int(self.H.msh_last_transcript(ch.ctypes.data_as(C.c_void_p), 128, idx.ctypes.data_as(C.c_void_p), 4096,
                                           nidx.ctypes.data_as(C.c_void_p)))
        return [(int(ch[2 * i]), int(ch[2 * i + 1])) for i in range(n)], [int(v) for v in idx[:int(nidx[0])]]

    def __del__(self):
        try:
            if self.ctx.h:
                self.close()
        except Exception:
            pass
