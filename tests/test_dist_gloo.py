"""N > 1 host logic on CPU: world_size 2 over gloo (the GPU box runs the same code over NCCL). Units are independent
proofs; ranks exchange proof digests and timing only. The prover here is the CPU oracle standing in for the device prover
(test infrastructure), so the sharding / gathering logic is exercised end to end without a GPU."""
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = textwrap.dedent("""
    import os, sys, json
    sys.path.insert(0, %r)
    import torch.distributed as dist
    from multi_stark_b200 import dist as msd
    import multi_stark_b200.system as mss
    from tests import _oracle as orc
    dist.init_process_group("gloo")
    r, w = dist.get_rank(), dist.get_world_size()
    assert msd.world() == w and msd.rank() == r
    # 1. partition
    units = [3, 4, 5, 6, 4]          # log2(#additions) of five independent proofs
    mine = list(msd.shard_units(len(units)))
    # 2. every rank proves its shard (oracle prover as the stand-in backend) and all digests are gathered
    L = orc.lib()
    S = orc.OracleSystem(L, "u32_add", log_blowup=1, num_queries=8)
    def prove(log_adds):
        byte, add, claims = mss.u32_add_workload(1 << log_adds)
        return S.prove([byte, add], list(claims))[0]
    proofs, digests = msd.prove_sharded(units, prove)
    assert sorted(proofs) == mine and len(digests) == len(units)
    for u in mine:
        assert digests[u] == msd.proof_digest(proofs[u])
    # 3. timing aggregation
    t = msd.max_over_ranks(10.0 + r)
    s = msd.sum_over_ranks(1.0 + r)
    msd.barrier()
    print(json.dumps({"rank": r, "mine": mine, "digests": [d.hex() for d in digests], "tmax": t, "sum": s}))
    dist.destroy_process_group()
""")


def test_shard_units_partition():
    from multi_stark_b200 import dist as msd
    for n in (0, 1, 5, 8, 13):
        for w in (1, 2, 3, 8):
            parts = [list(msd.shard_units(n, w, r)) for r in range(w)]
            assert sum(parts, []) == list(range(n))
            assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1


def test_two_ranks_over_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER % ROOT)
    port = 29500 + os.getpid() % 2000
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   OMP_NUM_THREADS="2")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = []
    for p in procs:
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0, err[-2000:]
        outs.append(out.strip().splitlines()[-1])
    import json
    res = sorted((json.loads(o) for o in outs), key=lambda d: d["rank"])
    assert res[0]["mine"] == [0, 1, 2] and res[1]["mine"] == [3, 4]
    assert res[0]["digests"] == res[1]["digests"] and len(set(res[0]["digests"])) == 4  # units 1 and 4 are the same proof
    assert res[0]["digests"][1] == res[0]["digests"][4]
    assert res[0]["tmax"] == res[1]["tmax"] == 11.0 and res[0]["sum"] == 3.0


COMM_WORKER = textwrap.dedent("""
    import ctypes as C, json, os, sys
    sys.path.insert(0, %r)
    import numpy as np
    import torch.distributed as dist
    from multi_stark_b200 import dist as msd
    dist.init_process_group("gloo")
    r, w = dist.get_rank(), dist.get_world_size()
    comm = msd.TorchComm(ctx=None)     # host collectives only: no device is touched
    st = comm.struct
    assert (st.rank, st.world) == (r, w)
    # all-gather of 24 bytes per rank through the C callback table (what host/dist_backend.hpp calls)
    send = np.arange(3, dtype=np.uint64) + 100 * r
    recv = np.zeros(3 * w, dtype=np.uint64)
    assert st.allgather_host(None, send.ctypes.data, recv.ctypes.data, 24) == 0
    # broadcast from rank 1
    buf = np.full(5, 7 + r, dtype=np.uint64)
    assert st.bcast_host(None, buf.ctypes.data, 40, 1) == 0
    # the staged device exchanges announce (sequence number, kind) first: ranks that make different sequences of device
    # collectives (a rank-dependent branch around one: a hang under NCCL) are told apart on every rank
    comm._same_call(1)
    comm._same_call(2)
    try:
        comm._same_call(1 if r == 0 else 2)
        mismatch = False
    except RuntimeError:
        mismatch = True
    print(json.dumps({"rank": r, "recv": recv.tolist(), "buf": buf.tolist(), "errors": comm.errors, "peer_memory": comm.peer_memory,
                      "mismatch_detected": mismatch}))
    dist.destroy_process_group()
""")


def test_comm_callbacks_over_gloo(tmp_path):
    """the collectives the sharded prover calls back into (multi_stark_b200/dist.py TorchComm), world_size 2 over gloo"""
    script = tmp_path / "comm_worker.py"
    script.write_text(COMM_WORKER % ROOT)
    port = 31500 + os.getpid() % 2000
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    import json
    res = []
    for p in procs:
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0, err[-2000:]
        res.append(json.loads(out.strip().splitlines()[-1]))
    for d in res:
        assert d["errors"] == []
        assert d["recv"] == [0, 1, 2, 100, 101, 102]
        assert d["buf"] == [8] * 5
        assert d["peer_memory"] == 0          # gloo ranks never map each other's device memory
        assert d["mismatch_detected"] is True


def test_assign_owners_keeps_height_classes_together():
    from multi_stark_b200 import dist as msd
    heights = [256, 1 << 20, 1 << 19, 1 << 20, 0, 1 << 18, 256]
    for w in (1, 2, 3, 8):
        own = msd.assign_owners(heights, w)
        assert len(own) == len(heights) and all(0 <= o < w for o in own)
        by_h = {}
        for h, o in zip(heights, own):
            if h:
                assert by_h.setdefault(h, o) == o, "a height class was split"
        if w >= 2:
            assert own[1] == own[3] and own[1] != own[2]  # the two 2^20 circuits together, the 2^19 one elsewhere
    assert msd.assign_owners(heights, 2) == msd.assign_owners(heights, 2)
