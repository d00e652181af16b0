"""The Python layer shared by the provers: the claims marshaller every prove() goes through, the TorchComm callback wrapper,
and (on the GPU) the sharded provers taking every claims form the single-GPU prover takes."""
import json
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from multi_stark_b200.system import _claims_args

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_claims_array_is_passed_without_a_copy():
    claims = np.arange(12, dtype=np.uint64).reshape(3, 4)
    flat, offs, stride, n = _claims_args(claims)
    assert np.shares_memory(flat, claims)
    assert offs is None and (n, stride) == (3, 4)
    flat, offs, stride, n = _claims_args(claims.astype(np.int64))  # converted once, same stride form
    assert flat.tolist() == list(range(12)) and offs is None and (n, stride) == (3, 4)


def test_claims_list_goes_through_offsets():
    flat, offs, stride, n = _claims_args([np.array([1, 2], dtype=np.uint64), [3], np.array([4, 5, 6], dtype=np.uint64)])
    assert flat.tolist() == [1, 2, 3, 4, 5, 6] and n == 3 and stride == 0
    assert np.ctypeslib.as_array(offs, shape=(n + 1,)).tolist() == [0, 2, 3, 6]


@pytest.mark.parametrize("claims", [[], None, np.zeros((0, 4), dtype=np.uint64)], ids=["empty_list", "none", "zero_rows"])
def test_no_claims(claims):
    flat, _, _, n = _claims_args(claims)
    assert n == 0 and flat.size == 1 and flat.dtype == np.uint64


FAILING_CALLBACK_WORKER = textwrap.dedent("""
    import json, sys
    sys.path.insert(0, %r)
    import torch.distributed as dist
    from multi_stark_b200 import dist as msd
    dist.init_process_group("gloo", init_method=%r, rank=int(sys.argv[1]), world_size=2)
    comm = msd.TorchComm(ctx=None)     # host collectives only: a device collective has no context to stage through
    rc = comm.struct.allgather_dev(None, 0, 0, 8)
    print(json.dumps({"rc": rc, "errors": comm.errors, "seconds": sorted(comm.seconds)}))
    dist.destroy_process_group()
""")


def test_comm_callback_reports_a_failure_as_1(tmp_path):
    """a collective that raises comes back to C++ as 1, with the exception in `errors` and its time still counted"""
    script = tmp_path / "worker.py"
    script.write_text(FAILING_CALLBACK_WORKER % (ROOT, "file://" + str(tmp_path / "rendezvous")))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
             for r in range(2)]
    for p in procs:
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0, err[-2000:]
        res = json.loads(out.strip().splitlines()[-1])
        assert res["rc"] == 1
        assert len(res["errors"]) == 1 and "AttributeError" in res["errors"][0]
        assert res["seconds"] == ["allgather_dev"]


SHARDED_CLAIMS_WORKER = textwrap.dedent("""
    import json, sys
    sys.path.insert(0, %r)
    import numpy as np
    import torch.distributed as dist
    import multi_stark_b200 as ms
    from multi_stark_b200 import dist as msd
    dist.init_process_group("gloo", init_method=%r, rank=0, world_size=1)
    ctx = ms.GpuContext(0)
    byte, add, claims = ms.u32_add_workload(1 << 10)  # 4096 claim values: the claims are hashed on the device
    cases = [("u32_add", [byte, add], claims, {"array": claims, "list": list(claims)}),
             ("fib", [ms.fib_trace(1 << 7)], np.zeros((0, 1), dtype=np.uint64), {"empty": []})]
    checked = []
    for kind, traces, reference, forms in cases:
        system = ms.System(kind, log_blowup=1, num_queries=10)
        single = ms.Prover(ctx, system)
        want = single.prove(traces, reference)
        dp = msd.DistProver(ctx, system, [0] * system.num_circuits)
        rs = msd.RowShardProver(ctx, system)
        for name, cl in forms.items():
            assert single.prove(traces, cl) == want, (kind, name, "Prover")
            assert dp.prove(traces, [t.shape[0] for t in traces], cl) == want, (kind, name, "DistProver")
            assert rs.prove(traces, cl) == want, (kind, name, "RowShardProver")
            checked.append(f"{kind}/{name}")
        dp.close()
        rs.close()
        single.close()
    print(json.dumps(checked))
    ctx.close()
    dist.destroy_process_group()
""")


@pytest.mark.gpu
def test_sharded_provers_take_every_claims_form(tmp_path):
    """one-rank group: DistProver and RowShardProver prove with claims as an array, a list of 1-D arrays and [] and give the
    bytes of Prover"""
    script = tmp_path / "worker.py"
    script.write_text(SHARDED_CLAIMS_WORKER % (ROOT, "file://" + str(tmp_path / "rendezvous")))
    p = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, (p.stdout + p.stderr)[-3000:]
    assert json.loads(p.stdout.strip().splitlines()[-1]) == ["u32_add/array", "u32_add/list", "fib/empty"]
