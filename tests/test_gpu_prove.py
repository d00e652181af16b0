"""GPU parity of the whole prover: `Proof::to_bytes` of the device prover (libmsgpu behind host/prover.hpp) must equal the
CPU oracle's byte for byte -- commitments, accumulators, opened values, every FRI commitment, the final polynomial and all
query openings -- and the restated verifier (src/verifier.rs) must accept it."""
import numpy as np
import pytest

from tests import _oracle as orc
from tests import _proof

pytestmark = pytest.mark.gpu
P = orc.P


@pytest.fixture(scope="module")
def gpu():
    import multi_stark_b200 as ms
    ctx = ms.GpuContext(0)
    yield ms, ctx
    ctx.close()


def workload(ms, kind, log_rows):
    if kind == "fib":
        return [ms.fib_trace(1 << log_rows)], []
    if kind.startswith("wide:"):
        return [ms.wide_trace(1 << log_rows, int(kind[5:]))], []
    byte, add, claims = ms.u32_add_workload(1 << log_rows)
    if kind == "u32_add":
        return [byte, add], list(claims)
    return [ms.fib_trace(1 << max(log_rows - 1, 1)), byte, add], list(claims)


def first_difference(a, b, path=""):
    """where two parsed proofs differ (for the assertion message)"""
    if isinstance(a, dict):
        for k in a:
            d = first_difference(a[k], b[k], path + "." + k)
            if d:
                return d
        return None
    if isinstance(a, list):
        if len(a) != len(b):
            return "%s: length %d != %d" % (path, len(a), len(b))
        for i, (x, y) in enumerate(zip(a, b)):
            d = first_difference(x, y, "%s[%d]" % (path, i))
            if d:
                return d
        return None
    return None if a == b else "%s: %r != %r" % (path, a, b)


def assert_same_proof(got, want):
    if got == want:
        return
    try:
        diff = first_difference(_proof.parse(got), _proof.parse(want))
    except Exception as e:  # noqa: BLE001
        diff = "unparseable (%s); lengths %d vs %d" % (e, len(got), len(want))
    raise AssertionError("device proof differs from the oracle's at " + str(diff))


CASES = [
    # kind, log_rows, log_blowup, log_final_poly_len, num_queries, pow_bits
    ("fib", 3, 1, 0, 10, 0),
    ("fib", 6, 2, 1, 10, 0),
    ("u32_add", 4, 1, 0, 20, 0),
    ("u32_add", 8, 2, 0, 20, 0),
    ("u32_add", 12, 1, 0, 100, 0),   # BASELINE configs[0]
    ("u32_add", 12, 2, 0, 100, 4),   # the reference bench's own parameters with a smaller PoW (smallest witness)
    ("mixed", 7, 2, 0, 15, 0),
    ("mixed", 9, 3, 2, 15, 0),
    ("u32_add", 14, 1, 0, 30, 0),
    ("wide:8", 5, 1, 0, 10, 0),      # quotient degree 2 at the minimal blowup
    ("wide:256", 7, 2, 0, 10, 0),    # BASELINE configs[2] shape: 2048-byte rows = two BLAKE3 chunks per leaf
    ("wide:700", 4, 2, 1, 8, 0),     # 5600-byte rows, 350 constraints
]


@pytest.mark.parametrize("kind,log_rows,lb,fpl,nq,pow_bits", CASES)
def test_proof_bytes_match_oracle(gpu, oracle, kind, log_rows, lb, fpl, nq, pow_bits):
    ms, ctx = gpu
    kw = dict(log_blowup=lb, log_final_poly_len=fpl, num_queries=nq, commit_pow_bits=pow_bits, query_pow_bits=pow_bits)
    system = ms.System(kind, **kw)
    prover = ms.Prover(ctx, system)
    S = orc.OracleSystem(oracle, kind, **kw)
    assert prover.preprocessed_commit() == S.preprocessed_commit()
    traces, claims = workload(ms, kind, log_rows)
    launches0 = ctx.launches
    got = prover.prove(traces, claims)
    assert ctx.launches > launches0, "the device prover launched no kernels"
    want, _ = S.prove(traces, claims)
    assert_same_proof(got, want)
    assert S.verify(claims, got) == "Ok"
    # a second proof with the same prover object (pool reuse, per-proof state reset)
    assert prover.prove(traces, claims) == got
    prover.close()
    S.close()


def test_sparse_activation(gpu, oracle):
    ms, ctx = gpu
    kw = dict(log_blowup=2, num_queries=12)
    system = ms.System("mixed", **kw)
    prover = ms.Prover(ctx, system)
    S = orc.OracleSystem(oracle, "mixed", **kw)
    traces, claims = workload(ms, "mixed", 6)
    traces[0] = np.zeros((0, 3), dtype=np.uint64)  # fib circuit inactive (src/lookup.rs:1057)
    got = prover.prove(traces, claims)
    want, _ = S.prove(traces, claims)
    assert_same_proof(got, want)
    assert S.verify(claims, got) == "Ok"
    # every circuit inactive: the reference panics (src/prover.rs:323-326); here an error, not a crash
    with pytest.raises(ms.MsgpuError):
        prover.prove([np.zeros((0, 3), dtype=np.uint64), np.zeros((0, 1), dtype=np.uint64), np.zeros((0, 14), dtype=np.uint64)], [])
    prover.close()
    S.close()


def test_large_proof_verifies(gpu, oracle):
    """2^18 additions: too slow to prove twice on the CPU in a unit test, so the device proof is checked by the restated
    verifier (size-independent property: prove -> verify accepts, tamper -> rejects)."""
    ms, ctx = gpu
    kw = dict(log_blowup=1, num_queries=40)
    system = ms.System("u32_add", **kw)
    prover = ms.Prover(ctx, system)
    S = orc.OracleSystem(oracle, "u32_add", **kw)
    traces, claims = workload(ms, "u32_add", 18)
    got = prover.prove(traces, np.asarray(claims))
    assert S.verify(claims, got) == "Ok"
    bad = bytearray(got)
    bad[len(bad) // 2] ^= 0x40
    assert S.verify(claims, bytes(bad)) != "Ok"
    prover.close()
    S.close()


def test_invalid_witness_is_an_error_not_a_crash(gpu):
    ms, ctx = gpu
    system = ms.System("fib", log_blowup=2, num_queries=5)
    prover = ms.Prover(ctx, system)
    tr = ms.fib_trace(16)
    with pytest.raises(ms.MsgpuError):  # wrong width
        prover.prove([tr[:, :2]], [])
    bad = tr.copy()
    bad[3, 0] = P  # not canonical
    with pytest.raises(ms.MsgpuError):
        prover.prove([bad], [])
    # the refused proofs left no per-proof state behind: the same prover still proves the valid trace, byte for byte
    fresh = ms.Prover(ctx, system)
    assert prover.prove([tr], []) == fresh.prove([tr], [])
    fresh.close()
    prover.close()


@pytest.mark.parametrize("log_rows,lb,fpl,nq,pow_bits", [(4, 1, 0, 20, 0), (8, 2, 1, 25, 0), (10, 1, 0, 30, 3), (12, 1, 0, 100, 0)])
def test_independent_python_verifier_accepts_device_proofs(gpu, log_rows, lb, fpl, nq, pow_bits):
    """tests/_pyverifier.py shares nothing with the host layer or the oracle (own challenger, own graph compiler, own MMCS / FRI
    / STARK verifier from the reference text): it must accept the device proof, and every challenge the device prover's
    transcript produced must equal the one the Python transcript re-derives from the proof's commitments."""
    from tests import _pyverifier as pv
    ms, ctx = gpu
    kw = dict(log_blowup=lb, log_final_poly_len=fpl, num_queries=nq, commit_pow_bits=pow_bits, query_pow_bits=pow_bits)
    system = ms.System("u32_add", **kw)
    prover = ms.Prover(ctx, system)
    traces, claims = workload(ms, "u32_add", log_rows)
    proof = prover.prove(traces, claims)
    challenges, indices = prover.last_transcript()
    prm = dict(kw, max_log_arity=1)
    out = {}
    cl = [list(map(int, c)) for c in claims]
    assert pv.verify(pv.named_system("u32_add"), prm, prover.preprocessed_commit(), cl, _proof.parse(proof), out) == "Ok"
    mine = [out["beta"], out["gamma"], out["alpha"], out["zeta"], out["alpha_pcs"]] + out["fri_betas"]
    assert [(e.a, e.b) for e in mine] == challenges
    assert out["query_indices"] == indices
    prover.close()


def test_system_from_descriptors_proves_the_same_bytes(gpu):
    """msh_system_create_from_graphs: the U32-add system assembled from descriptors that the independent Python compiler made
    produces, through msh_prove, the proof bytes of the named system; and a circuit that exists only as a descriptor proves
    and is accepted by the Python verifier."""
    from tests import _pyverifier as pv
    ms, ctx = gpu
    kw = dict(log_blowup=1, num_queries=20)
    graphs = [pv.graph_dict(c) for c in pv.named_system("u32_add")]
    pre = [np.arange(256, dtype=np.uint64).reshape(256, 1), None]
    named, generic = ms.System("u32_add", **kw), ms.System.from_graphs(graphs, pre, **kw)
    traces, claims = workload(ms, "u32_add", 9)
    pa, pb = ms.Prover(ctx, named), ms.Prover(ctx, generic)
    assert pa.prove(traces, claims) == pb.prove(traces, claims)
    pa.close()
    pb.close()
    E = pv.Expr
    m = E.main
    circ = pv.Circuit(3, [], [m(2) - (m(0) * m(1) + E.const(3)), E("trans") * (E.main_next(0) - m(0) - E.const(1))])
    n = 1 << 10
    rng = np.random.default_rng(3)
    a = np.arange(5, 5 + n, dtype=np.uint64)
    b = rng.integers(0, P, size=n, dtype=np.uint64)
    c = np.array([(int(x) * int(y) + 3) % P for x, y in zip(a, b)], dtype=np.uint64)
    custom = ms.System.from_graphs([pv.graph_dict(circ)], **kw)
    pr = ms.Prover(ctx, custom)
    proof = pr.prove([np.stack([a, b, c], axis=1)], [])
    assert pv.verify([circ], dict(kw, log_final_poly_len=0, max_log_arity=1, commit_pow_bits=0, query_pow_bits=0), None, [],
                     _proof.parse(proof)) == "Ok"
    pr.close()
