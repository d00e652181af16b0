"""One proof over two ranks (SURVEY 8e partitioning A, BASELINE configs[3] shape): circuits are split over the ranks, class
digests / reduced openings / query rows are exchanged, and the proof must be byte-identical to the single-GPU proof and be
accepted by the restated verifier. On a single-GPU box both ranks share cuda:0 and exchange over gloo (device buffers staged
through the host); tools/dist_prove.py runs the same worker over NCCL with one GPU per rank."""
import json
import os
import socket
import subprocess
import sys

import pytest

from tests import _oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def run_world(tmp_path, world, kind, log_heights, owners, params, backend="gloo", extra_env=None):
    port = free_port()
    prefix = str(tmp_path / "dist")
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   **(extra_env or {}))
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "_dist_worker.py"), backend, kind,
                                       ",".join(map(str, log_heights)), owners, prefix, json.dumps(params)], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = []
    for p in procs:
        try:
            out, _ = p.communicate(timeout=600)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
        outs.append(out)
    if any(p.returncode != 0 for p in procs):
        raise AssertionError("\n".join("---- rank %d rc %s ----\n%s" % (r, p.returncode, outs[r][-2500:]) for r, p in enumerate(procs)))
    proofs = [open("%s.rank%d.proof" % (prefix, r), "rb").read() for r in range(world)]
    infos = [json.load(open("%s.rank%d.json" % (prefix, r))) for r in range(world)]
    single = open(prefix + ".single.proof", "rb").read()
    return proofs, single, infos


@pytest.mark.parametrize("log_heights,owners,params", [
    ([10, 12], "0,0,1", dict(log_blowup=1, num_queries=20)),          # byte table + small adds on rank 0, tall adds on rank 1
    ([12, 9], "1,0,1", dict(log_blowup=2, num_queries=15)),           # tree owner = rank 0, preprocessed table on rank 1
    ([11, 11, 8], "auto", dict(log_blowup=1, num_queries=10, log_final_poly_len=1)),  # two circuits of one height share a rank
])
def test_sharded_proof_is_byte_identical(tmp_path, oracle, log_heights, owners, params):
    kind = "multi:%d" % len(log_heights)
    proofs, single, infos = run_world(tmp_path, 2, kind, log_heights, owners, params)
    assert proofs[0] == proofs[1], "ranks disagree on the proof"
    assert proofs[0] == single, "sharded proof differs from the single-GPU proof"
    assert infos[0]["bytes_dev"] + infos[1]["bytes_dev"] > 0, "nothing was exchanged: the proof was not sharded"
    assert all(i["launches"] > 0 for i in infos)
    # acceptance by the restated verifier (oracle, test infrastructure)
    import multi_stark_b200 as ms
    traces, claims = ms.multi_workload(log_heights)
    S = orc.OracleSystem(oracle, kind, **params)
    assert S.verify(list(claims), proofs[0]) == "Ok"
    S.close()


def test_sharded_mixed_system_with_selectors(tmp_path, oracle):
    """fib_cubic (no lookups, quotient degree 2, selectors) on one rank, the lookup circuits on the other"""
    params = dict(log_blowup=1, num_queries=12)
    proofs, single, infos = run_world(tmp_path, 2, "mixed", [9, 7], "1,0,0", params)
    assert proofs[0] == proofs[1] == single


def test_same_height_on_two_ranks_is_refused(tmp_path):
    with pytest.raises(AssertionError) as e:
        run_world(tmp_path, 2, "multi:2", [10, 10], "0,0,1", dict(log_blowup=1, num_queries=5))
    assert "must live on one rank" in str(e.value)
