"""One rank of tests/test_gpu_constraints.py's row-sharded lookup cases: every case is a one-circuit system built from a graph
descriptor, proved by RowShardProver over gloo on cuda:0 and, on rank 0, by the single-GPU Prover. Launched with RANK /
WORLD_SIZE / MASTER_ADDR / MASTER_PORT in the environment.
argv: cases json ([{"graph": ..., "trace": [[...]...]}...]) out_prefix
Writes out_prefix.rank<r>.json: per case {"error": message or null, "proof": hex or null, "single": hex (rank 0 only)}."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import multi_stark_b200 as ms  # noqa: E402
from multi_stark_b200 import dist as msd  # noqa: E402


def main():
    cases = json.load(open(sys.argv[1]))
    out_prefix = sys.argv[2]
    rank = int(os.environ["RANK"])
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    ctx = ms.GpuContext(0)
    results = []
    for case in cases:
        g = case["graph"]
        g["nodes"] = [tuple(n) for n in g["nodes"]]
        g["lookups"] = [(m, list(a)) for m, a in g["lookups"]]
        system = ms.System.from_graphs([g], log_blowup=1, num_queries=8)
        trace = np.array(case["trace"], dtype=np.uint64)
        res = {"error": None, "proof": None}
        prover = msd.RowShardProver(ctx, system)
        try:
            res["proof"] = prover.prove([trace], None).hex()
        except Exception as e:  # the refusal under test: every rank reports it
            res["error"] = str(e)
        prover.close()
        dist.barrier()
        if rank == 0:
            single = ms.Prover(ctx, system)
            res["single"] = single.prove([trace], None).hex()
            single.close()
        system.close()
        results.append(res)
    with open("%s.rank%d.json" % (out_prefix, rank), "w") as f:
        json.dump(results, f)
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
