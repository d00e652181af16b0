"""One rank of a sharded proof (tests/test_gpu_dist_prove.py, tools/dist_prove.py). Launched with RANK / WORLD_SIZE /
MASTER_ADDR / MASTER_PORT in the environment. backend gloo: every rank uses cuda:0 (single-GPU box), device buffers are staged
through the host; backend nccl: rank r uses cuda:r and device buffers travel over NVLink.
argv: backend kind log_heights(comma separated; first = byte table is implicit) owners(comma separated or "auto") out_prefix [params json]
kind "commit:W" commits one 2^log_height x W matrix over the row shards instead of proving: the result files then hold roots."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import multi_stark_b200 as ms  # noqa: E402
from multi_stark_b200 import dist as msd  # noqa: E402


def main():
    backend, kind, lhs, owners, out_prefix = sys.argv[1:6]
    params = json.loads(sys.argv[6]) if len(sys.argv) > 6 else dict(log_blowup=1, num_queries=20)
    reps = int(os.environ.get("DIST_REPS", "1"))
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = rank if backend == "nccl" else 0
    torch.cuda.set_device(dev)
    if backend == "nccl":
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    else:
        dist.init_process_group("gloo")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = ms.GpuContext(dev, stream=stream.cuda_stream)
    if kind.startswith("commit:"):
        commit_rows(ctx, int(kind[7:]), int(lhs), params, out_prefix, rank)
        ctx.close()
        dist.destroy_process_group()
        return
    system = ms.System(kind, **params)
    log_heights = [int(x) for x in lhs.split(",")]
    if kind.startswith("multi:"):
        traces, claims = ms.multi_workload(log_heights)
    elif kind == "mixed":
        byte, add, claims = ms.u32_add_workload(1 << log_heights[0])
        traces = [ms.fib_trace(1 << log_heights[1]), byte, add]
    elif kind == "u32_add":
        byte, add, claims = ms.u32_add_workload(1 << log_heights[0])
        traces = [byte, add]
    elif kind.startswith("wide:") and owners == "rowshard" and os.environ.get("DIST_BLOCKS") == "1":
        # only the rows this rank reads are generated (a 256 x 2^22 trace is 8.6 GB per process otherwise)
        w, h = int(kind[5:]), 1 << log_heights[0]
        rows = h // world if (world > 1 and w >= world and h >= world * 64) else h
        traces, claims = [ms.wide_trace(rows, w, row0=rows * rank if rows != h else 0)], np.zeros((0, 1), dtype=np.uint64)
        block_heights = [h]
    elif kind.startswith("wide:"):
        traces, claims = [ms.wide_trace(1 << log_heights[0], int(kind[5:]))], np.zeros((0, 1), dtype=np.uint64)
    elif kind == "fib":
        traces, claims = [ms.fib_trace(1 << log_heights[0])], np.zeros((0, 1), dtype=np.uint64)
    else:
        raise SystemExit("unknown kind")
    traces = [ctx.pinned_copy(t) for t in traces]  # what a production caller hands over: page-locked host buffers
    claims = ctx.pinned_copy(claims) if len(claims) else claims
    heights = [t.shape[0] for t in traces]
    rowshard = owners == "rowshard"
    block_heights = locals().get("block_heights")
    if rowshard:  # every matrix split by rows over all ranks (host/rowshard_backend.hpp)
        owner = []
        prover = msd.RowShardProver(ctx, system)
    else:
        owner = msd.assign_owners(heights, world) if owners == "auto" else [int(x) for x in owners.split(",")]
        prover = msd.DistProver(ctx, system, owner)
    local = [t if owner[i] == rank else None for i, t in enumerate(traces)] if not rowshard else None
    times = []
    for _ in range(reps):
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if _ == reps - 1:
            prover.comm.seconds.clear()  # the collectives of the last proof only (the first ones carry NCCL's start-up)
        proof = prover.prove(traces, claims, heights=block_heights) if rowshard else prover.prove(local, heights, claims)
        times.append((time.perf_counter() - t0) * 1e3)
    with open("%s.rank%d.proof" % (out_prefix, rank), "wb") as f:
        f.write(proof)
    info = {"rank": rank, "owner": owner, "heights": heights, "ms": times, "stages": prover.last_stage_ms,
            "bytes_dev": prover.bytes_dev // reps, "bytes_host": prover.comm.bytes_host // reps, "launches": ctx.launches,
            "comm_ms_per_proof": {k: v * 1e3 for k, v in prover.comm.seconds.items()},
            "pre_commit": (prover.preprocessed_commit() or b"").hex()}
    if rank == 0 and os.environ.get("DIST_SINGLE", "1") == "1" and block_heights is None:
        # the same proof on one GPU through the ordinary prover
        single = ms.Prover(ctx, system)
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            want = single.prove(traces, claims)
            ts.append((time.perf_counter() - t0) * 1e3)
        info["single_ms"] = ts
        info["single_stages"] = single.last_stage_ms
        with open("%s.single.proof" % out_prefix, "wb") as f:
            f.write(want)
        single.close()
    with open("%s.rank%d.json" % (out_prefix, rank), "w") as f:
        json.dump(info, f)
    dist.barrier()
    prover.close()
    ctx.close()
    dist.destroy_process_group()


def commit_rows(ctx, width, log_rows, params, out_prefix, rank):
    """`Pcs::commit` of one matrix of any width by RowShardProver.commit, each rank handing over only the rows it reads; rank 0
    also commits the whole matrix on one GPU (GpuPcs) for reference."""
    h = 1 << log_rows
    whole = np.random.default_rng(h * width).integers(0, ms.P, size=(h, width), dtype=np.uint64)
    prover = msd.RowShardProver(ctx, ms.System("fib", **params))  # the commitment reads only the system's log_blowup
    row0, rows = prover.block_rows(h, width)
    root = prover.commit([whole[row0:row0 + rows]], [h], [width], host=True)
    with open("%s.rank%d.proof" % (out_prefix, rank), "wb") as f:
        f.write(root)
    with open("%s.rank%d.json" % (out_prefix, rank), "w") as f:
        json.dump({"rank": rank, "rows": rows, "bytes_dev": prover.bytes_dev, "launches": ctx.launches}, f)
    if rank == 0:
        want, pd = ms.GpuPcs(ctx, params["log_blowup"]).commit([whole])
        pd.free()
        with open("%s.single.proof" % out_prefix, "wb") as f:
            f.write(bytes(want))
    dist.barrier()
    prover.close()


if __name__ == "__main__":
    main()
