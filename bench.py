#!/usr/bin/env python
"""bench.py -- commitment hot path of multi-stark on B200 (see DESIGN.md "Measurement").

A step = one pass of the hot path over one batch of synthetic input: the two trace commitments of
BASELINE.json configs[1] (U32-add circuit with lookups at 2^20 rows + the 256-row byte table,
log_blowup 1): stage-1 `pcs.commit` (reference src/prover.rs:350) and stage-2 `pcs.commit`
(src/prover.rs:419) -- coset LDE of every matrix + BLAKE3 Merkle tree, roots read back.

  python bench.py [--gpus N] [--steps K] [--warmup W]       our CUDA path (one JSON line on rank 0)
  python bench.py --impl reference ...                      CPU restatement of the reference path
  python bench.py ... --dump-outputs DIR                    also write the last timed step's outputs (see dump_commit)

metric = LDE+Merkle Gelem/s (committed LDE elements sum(n*B*w) per second, whole job).
`value`: inputs resident in HBM.  `e2e`: through the host-pointer C-ABI call (`msgpu_commit`) with
pinned host buffers, H2D copies and the root D2H inside the timed region."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

P = 2**64 - 2**32 + 1


# ------------------------------------------------------------------------------------------------
# workload (reference benches/multi_stark.rs:171-217): U32Add trace rows = [x bytes, y bytes, z bytes,
# carry, 1] from two xorshift32 streams; byte table multiplicities. Stage-2 (lookup accumulator)
# columns are synthetic field elements of the stage-2 shape (26 / 2 base columns).
# ------------------------------------------------------------------------------------------------
def _xs_step(x):
    x ^= (x << 13) & 0xFFFFFFFF
    x ^= x >> 17
    x ^= (x << 5) & 0xFFFFFFFF
    return x


def xorshift_stream(seed, n, block=4096):
    """The xorshift32 stream of benches/multi_stark.rs:180-187. x_{i+1} = T x_i is linear over GF(2): the first `block` values
    are generated one by one, then whole blocks at once with T^block applied through four byte-indexed tables."""
    block = min(block, n)
    first = np.empty(block, dtype=np.uint32)
    x = seed
    for i in range(block):
        x = _xs_step(x)
        first[i] = x
    if block == n:
        return first

    def apply(M, v):
        r = 0
        for j in range(32):
            if (v >> j) & 1:
                r ^= M[j]
        return r
    base = [_xs_step(1 << j) for j in range(32)]  # columns of T
    R, e = None, block
    while e:
        if e & 1:
            R = base if R is None else [apply(base, c) for c in R]
        base = [apply(base, c) for c in base]
        e >>= 1
    tabs = []
    for k in range(4):
        t = np.zeros(256, dtype=np.uint32)
        for v in range(256):
            r = 0
            for bit in range(8):
                if (v >> bit) & 1:
                    r ^= R[8 * k + bit]
            t[v] = r
        tabs.append(t)
    out = np.empty(n, dtype=np.uint32)
    out[:block] = first
    cur, pos = first, block
    while pos < n:
        cur = tabs[0][cur & 0xFF] ^ tabs[1][(cur >> 8) & 0xFF] ^ tabs[2][(cur >> 16) & 0xFF] ^ tabs[3][cur >> 24]
        m = min(block, n - pos)
        out[pos:pos + m] = cur[:m]
        pos += m
    return out


def u32_add_traces(log_rows):
    """benches/multi_stark.rs:171-238 in numpy (no product library: the reference arm uses this too): the byte table's
    multiplicity trace (256 x 1), the U32-add trace (n x 14) and the claims [1, x, y, z] (n x 4)."""
    n = 1 << log_rows
    x = xorshift_stream(0xDEADBEEF, n)
    y = xorshift_stream(0xCAFEBABE, n)
    zsum = x.astype(np.uint64) + y.astype(np.uint64)
    z = (zsum & 0xFFFFFFFF).astype(np.uint32)
    main = np.empty((n, 14), dtype=np.uint64)
    for k, v in enumerate((x, y, z)):
        for b in range(4):
            main[:, 4 * k + b] = (v >> (8 * b)) & 0xFF
    main[:, 12] = zsum >> 32
    main[:, 13] = 1
    mult = np.bincount(main[:, :12].astype(np.int64).reshape(-1), minlength=256).astype(np.uint64)
    claims = np.empty((n, 4), dtype=np.uint64)
    claims[:, 0] = 1
    claims[:, 1], claims[:, 2], claims[:, 3] = x, y, z
    return mult.reshape(256, 1), main, claims


def u32_add_workload(log_rows, seed=0):
    """The two commit calls of prove(): stage 1 (byte table multiplicities, U32-add trace) then stage 2 (synthetic field
    elements of the stage-2 shapes: 2 / 26 base columns), matrices in circuit order."""
    n = 1 << log_rows
    byte_main, main, _ = u32_add_traces(log_rows)
    rng = np.random.default_rng(seed + 1)
    s2_main = rng.integers(0, P, size=(n, 26), dtype=np.uint64)
    s2_byte = rng.integers(0, P, size=(256, 2), dtype=np.uint64)
    return [[byte_main, main], [s2_byte, s2_main]]


def committed_elements(stages, log_blowup):
    return sum(m.shape[0] * m.shape[1] for st in stages for m in st) << log_blowup


def lde_bytes(stages, log_blowup):
    """SURVEY 8(d): LDE of n x w moves 8*n*w*(1+B) compulsory bytes."""
    return sum(8 * m.shape[0] * m.shape[1] * (1 + (1 << log_blowup)) for st in stages for m in st)


def merkle_bytes(stages, log_blowup):
    """SURVEY 8(d): 8*nB*W + 32*nB (leaves) + 96*(nB - 1) (nodes) per tree."""
    tot = 0
    for st in stages:
        nb = max(m.shape[0] for m in st) << log_blowup
        tot += sum(8 * (m.shape[0] << log_blowup) * m.shape[1] + 32 * (m.shape[0] << log_blowup) for m in st)
        tot += 96 * (nb - 1)
    return tot


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path hands its caller, so that two builds can be compared output for output. Every value
# is an exact integer stored as float64: a byte as it is, a 64-bit field element as [low 32 bits, high 32 bits].
# ------------------------------------------------------------------------------------------------
DUMP_ROWS = 4096  # rows kept of each tall LDE matrix: 43 columns x 4096 rows x 16 bytes = 2.8 MB in all


def u64_halves(a):
    a = np.asarray(a, dtype=np.uint64)
    return np.stack([a & np.uint64(0xFFFFFFFF), a >> np.uint64(32)], axis=-1).astype(np.float64)


def dump_commit(out_dir, pds):
    """The ProverData of one step's commitments (stage s = 1, 2): stage{s}_root, the 32 root bytes, and for every committed
    matrix i (LDE rows in bit-reversed order, as ProverData holds them) stage{s}_lde{i}, the rows listed in stage{s}_lde{i}_rows:
    all rows of a matrix of at most DUMP_ROWS rows, else DUMP_ROWS rows drawn with the fixed seed (s, i)."""
    os.makedirs(out_dir, exist_ok=True)
    for s, pd in enumerate(pds, 1):
        np.save(os.path.join(out_dir, "stage%d_root.npy" % s), np.asarray(pd.root, dtype=np.float64))
        for i in range(pd.num_matrices):
            lde = pd.read_rows(i)
            rows = np.arange(len(lde)) if len(lde) <= DUMP_ROWS else np.sort(
                np.random.default_rng([s, i]).choice(len(lde), DUMP_ROWS, replace=False))
            np.save(os.path.join(out_dir, "stage%d_lde%d.npy" % (s, i)), u64_halves(lde[rows]))
            np.save(os.path.join(out_dir, "stage%d_lde%d_rows.npy" % (s, i)), rows.astype(np.float64))


def dump_proof(out_dir, name, proof):
    """Proof::to_bytes of a prove() leg's last timed call, one float64 per byte."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), np.frombuffer(proof, dtype=np.uint8).astype(np.float64))


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clocks / throttle reasons DURING the timed region, read through NVML inside this process (nvidia_ml_py).
    The recipe's `nvidia-smi -lms 100` subprocess stalls this library's host-side driver calls (stream-ordered alloc/free,
    root read-back) by several ms per step (tools/diag_step.py: 4.7 ms/step alone, 10-25 ms/step with nvidia-smi polling,
    4.7 ms/step with NVML polling), so the same counters are polled with NVML from a thread at 20 Hz instead."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, device):
        self.device = device
        self.sm, self.mask, self.stop_flag, self.thread, self.max_mhz = [], 0, False, None, None

    @property
    def lines(self):  # number of samples so far
        return self.sm

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # torch's device index follows CUDA_VISIBLE_DEVICES; NVML enumerates physical devices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.device
            if vis:
                try:
                    idx = int(vis.split(",")[self.device])
                except (ValueError, IndexError):
                    idx = self.device
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                pass
            time.sleep(0.05)

    def stop(self):
        if not self.thread:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.thread.join(timeout=2)
        reasons = sorted(nm for nm, bit in self.REASONS if self.mask & bit)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "samples": len(self.sm), "reasons": reasons, "source": "NVML (in-process, 20 Hz)"}


def step_counters():
    """ncu counters of one bench step (tools/one_step.py + tools/ncu_inst_counts.py): data-independent instruction counts
    and DRAM traffic per stage, committed under profiles/."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "step_counters_*.json")))
    if not files:
        return None, None
    try:
        with open(files[-1]) as f:
            return json.load(f), os.path.basename(files[-1])
    except Exception:
        return None, None


def ncu_pipe_busy():
    """Per-kernel ALU / FMA-heavy pipe busy percentages from the committed `ncu --set full` capture of the same kernels
    (tools/ncu_pipe_busy.py): static annotation of the bench line, labelled with its source file."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "pipe_busy_*.json")))
    if not files:
        return None
    try:
        with open(files[-1]) as f:
            d = json.load(f)
        return {"file": os.path.basename(files[-1]), "what": d.get("what"),
                "kernels": {k: v for k, v in d.get("kernels", {}).items() if not k.startswith("k_fill")}}
    except Exception:
        return None


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
def load_oracle():
    """CPU restatement of the reference path (oracle/): ONLY for the cpu_baseline / --impl reference legs. Uses every host
    core whatever OMP_NUM_THREADS says (torchrun exports OMP_NUM_THREADS=1 to its workers)."""
    from tests import _oracle
    L = _oracle.lib()
    L.orc_set_num_threads(os.cpu_count() or 1)
    return _oracle, L


def cpu_commit_time(stages, log_blowup, reps=1):
    orc, L = load_oracle()
    # warm the twiddle caches on a tiny instance of the same shapes
    for st in stages:
        _, h = orc.pcs_commit(L, [m[:min(len(m), 64)] for m in st], log_blowup)
        L.orc_mmcs_free(h)
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        for st in stages:
            _, h = orc.pcs_commit(L, st, log_blowup)
            L.orc_mmcs_free(h)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best, int(L.orc_num_threads())


def sample_stages(stages, log_sample):
    """Bounded sample of the workload for the CPU legs: the first 2^log_sample rows of the tall matrices."""
    n = 1 << log_sample
    return [[m if m.shape[0] <= n else m[:n] for m in st] for st in stages]


CPU_NOTE = ("oracle/: C++/OpenMP restatement of the reference path with AVX-512/AVX2 Goldilocks row kernels, 16-lane BLAKE3 and a "
            "cache-blocked two-pass DFT; NOT the Rust reference binary (no cargo here, Plonky3 un-vendored); the stage-2, quotient "
            "and opening stages of its prove() are scalar + OpenMP")


def prove_params(args):
    """BASELINE configs[0]/[1]: log_blowup as given, 100 queries, final poly len 1, binary folding, PoW 0/0 (deterministic)."""
    return dict(log_blowup=args.log_blowup, log_final_poly_len=0, max_log_arity=1, num_queries=100, commit_pow_bits=0,
                query_pow_bits=0)


def cpu_prove_time(args, log_rows, reps=1):
    """The oracle's CPU prover (restatement of src/prover.rs:289-603 over restated Plonky3 semantics) on all host cores, on the
    numpy-generated workload (no product library involved)."""
    orc, L = load_oracle()
    S = orc.OracleSystem(L, "u32_add", **prove_params(args))
    byte, add, claims = u32_add_traces(log_rows)
    claims_list = list(claims)
    best, stages = None, None
    for _ in range(reps):
        t0 = time.perf_counter()
        proof, ms_stages = S.prove([byte, add], claims_list)
        dt = (time.perf_counter() - t0) * 1e3
        if best is None or dt < best:
            best, stages = dt, ms_stages
    ok = S.verify(claims_list, proof)
    S.close()
    names = ["stark/stage1_commit", "stark/claims", "stark/stage2_commit", "stark/quotient", "stark/fri_open", "stark/prove"]
    # `ms` = the prover's own clock (sum of its stages), like the GPU leg's stages; `wall_ms` adds the ctypes marshalling
    return {"rows": 1 << log_rows, "ms": float(stages[5]), "wall_ms": best, "stages_ms": dict(zip(names, stages)),
            "cores": int(L.orc_num_threads()), "simd_level": int(L.orc_simd_level()), "kind": "port", "verified": ok == "Ok",
            "proof_bytes": len(proof), "digest": __import__("hashlib").sha256(proof).hexdigest()}


def prove_stage_bytes(log_rows, log_blowup):
    """SURVEY 8(d) algorithmic bytes of the prove() stages after the trace commitments, for the U32-add system (byte table:
    n = 256, widths pre 1 / main 1 / stage-2 2, q = 1; U32-add: n = 2^log_rows, widths 14 / 26, q = 1; D = 2)."""
    B = 1 << log_blowup
    out = {"quotient": 0, "open": 0, "fri": 0}
    heights = set()
    for n, wp, w1, w2, q in ((256, 1, 1, 2, 1), (1 << log_rows, 0, 14, 26, 1)):
        nq, W = n * q, wp + w1 + w2 + 2 * q
        out["quotient"] += 8 * nq * (wp + w1 + w2) + 16 * nq          # quotient evaluation
        out["quotient"] += 16 * nq + 8 * n * 2 * q * (1 + B)           # quotient DFT / slices + LDE
        out["open"] += 8 * n * W                                       # barycentric sums over the first n rows
        out["open"] += 8 * n * B * W                                   # reduced openings: every LDE read once
        heights.add(n * B)
    out["open"] += 16 * sum(heights)
    out["fri"] = 96 * max(heights)                                     # sum_k 48 * nB / 2^k
    return out


def gpu_prove_leg(args, ms, ctx, log_rows, steps, warmup, verify, peak=None):
    """prove() end to end through the public API: HOST (pinned) traces and claims in, Proof::to_bytes out.
    Returns (results, the proof of the last timed call)."""
    system = ms.System("u32_add", **prove_params(args))
    prover = ms.Prover(ctx, system)  # System::new: programs + preprocessed commitment (setup, untimed like Criterion's setup)
    byte, add, claims = u32_add_traces(log_rows)
    rk = int(os.environ.get("RANK", "0"))
    if rk:  # every rank proves its own instance: the same additions in a rotated row order
        add, claims = np.roll(add, rk, axis=0), np.roll(claims, rk, axis=0)
    byte, add, claims = ctx.pinned_copy(byte), ctx.pinned_copy(add), ctx.pinned_copy(claims)
    for _ in range(warmup):
        proof = prover.prove([byte, add], claims)
    times, stage_acc = [], {}
    l0 = ctx.launches
    for _ in range(steps):
        t0 = time.perf_counter()
        proof = prover.prove([byte, add], claims)
        times.append((time.perf_counter() - t0) * 1e3)
        for k, v in prover.last_stage_ms.items():
            stage_acc.setdefault(k, []).append(v)
    launches = (ctx.launches - l0) // max(steps, 1)
    out = {"rows": 1 << log_rows, "ms": float(np.median(times)), "ms_min": float(np.min(times)), "steps": steps,
           "stages_ms": {k: float(np.median(v)) for k, v in stage_acc.items()}, "proof_bytes": len(proof),
           "digest": __import__("hashlib").sha256(proof).hexdigest(),
           "h2d_bytes": int(byte.nbytes + add.nbytes + claims.nbytes), "gpu_launches": int(launches),
           "timing": "host wall clock around the call (host buffers in, proof bytes out)"}
    # per-launch CUDA events of one more proof: device time per stage, and the HBM roofline of the stages SURVEY 8(d) gives
    # algorithmic bytes for (quotient, opening = barycentric + reduced openings, FRI folds)
    ctx.profile_begin()
    prover.prove([byte, add], claims)
    dev = {}
    for rec in ctx.profile_end():
        dev[rec["stage"] or "other"] = dev.get(rec["stage"] or "other", 0.0) + rec["ms"]
    out["device_ms_by_stage"] = {k: round(v, 4) for k, v in sorted(dev.items())}
    out["device_ms"] = float(sum(dev.values()))
    if peak:
        alg = prove_stage_bytes(log_rows, args.log_blowup)
        out["stage_roofline"] = [{"stage": st, "ms": dev[st], "algorithmic_bytes": alg[st],
                                  "achieved_gbs": alg[st] / (dev[st] / 1e3) / 1e9, "frac": alg[st] / (dev[st] / 1e3) / 1e9 / peak,
                                  "note": "fri = folds + layer commitments (BLAKE3): integer-bound, bytes are the folds' only"
                                  if st == "fri" else "HBM fraction of measured copy bandwidth"}
                                 for st in ("quotient", "open", "fri") if dev.get(st)]
    if verify:
        orc, L = load_oracle()
        S = orc.OracleSystem(L, "u32_add", **prove_params(args))
        out["verified"] = S.verify(list(claims), proof) == "Ok"
        S.close()
    prover.close()
    return out, proof


def sharded_prove_leg(args, ms, msd, ctx, rank, world, steps):
    """ONE proof over all ranks (BASELINE configs[3] shape, SURVEY 8e partitioning A): byte table + 7 U32-add circuits of
    2^18..2^22 rows, circuits -> ranks by height class; compared with the same proof on one GPU (rank 0)."""
    import hashlib
    import torch
    log_heights = [min(h, args.log_rows + 2) for h in (22, 21, 21, 20, 20, 19, 18)]
    system = ms.System("multi:%d" % len(log_heights), **prove_params(args))
    traces, claims = ms.multi_workload(log_heights)
    heights = [t.shape[0] for t in traces]
    owner = msd.assign_owners(heights, world)
    prover = msd.DistProver(ctx, system, owner)
    local = [ctx.pinned_copy(t) if owner[i] == rank else None for i, t in enumerate(traces)]
    claims_p = ctx.pinned_copy(claims)
    times = []
    for it in range(steps + 1):
        msd.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        proof = prover.prove(local, heights, claims_p)
        if it:
            times.append((time.perf_counter() - t0) * 1e3)
    out = {"log_heights": log_heights, "owner": owner, "ms": msd.max_over_ranks(float(np.median(times))),
           "stages_ms_rank0": prover.last_stage_ms, "proof_bytes": len(proof), "digest": hashlib.sha256(proof).hexdigest(),
           "device_bytes_exchanged_this_rank": prover.comm.bytes_dev // (steps + 1),
           "timing": "host wall clock around the call on every rank, median, max over ranks"}
    digests = msd.gather_digests([bytes.fromhex(out["digest"])])
    out["all_ranks_same_proof"] = len(set(digests)) == 1
    prover.close()
    if rank == 0:
        single = ms.Prover(ctx, system)
        pinned = [ctx.pinned_copy(t) for t in traces]
        ts = []
        for it in range(3):
            t0 = time.perf_counter()
            want = single.prove(pinned, claims_p)
            ts.append((time.perf_counter() - t0) * 1e3)
        out["single_gpu_ms"] = float(np.min(ts[1:]))
        out["identical_to_single_gpu_proof"] = want == proof
        single.close()
    msd.barrier()
    return out


def rowshard_commit_leg(args, ms, msd, ctx, rs, rank, world, steps, warmup):
    """The bench step -- both trace commitments of configs[1] -- as ONE job over all ranks: every matrix split by rows
    (host/rowshard_backend.hpp): column-sharded NTT between two all-to-alls, leaf hashing and subtrees per rank, 32-byte subtree
    roots all-gathered. Same work for every N (strong scaling). Returns (ms/step resident, ms/step from host, roots)."""
    import torch
    stages = u32_add_workload(args.log_rows, seed=0)  # the SAME matrices on every rank
    hs = [[m.shape[0] for m in st] for st in stages]
    ws = [[m.shape[1] for m in st] for st in stages]
    def my_rows(m):
        r0, n = rs.block_rows(m.shape[0], m.shape[1])
        return np.ascontiguousarray(m[r0:r0 + n])
    blocks = [[my_rows(m) for m in st] for st in stages]
    pinned = [[ctx.pinned_copy(b) for b in st] for st in blocks]
    dev = [[ctx.upload(b) for b in st] for st in blocks]

    def step(host):
        return [rs.commit(pinned[i] if host else dev[i], hs[i], ws[i], host) for i in range(len(stages))]

    out = {}
    for host in (False, True):
        for _ in range(warmup):
            roots = step(host)
        msd.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            roots = step(host)
        e1.record()
        torch.cuda.synchronize()
        out["host" if host else "resident"] = msd.max_over_ranks(e0.elapsed_time(e1)) / steps
        msd.barrier()
    for st in dev:
        for p in st:
            ctx.free(p)
    return out["resident"], out["host"], roots, sum(b.nbytes for st in blocks for b in st)


def rowshard_prove_leg(args, ms, msd, ctx, rank, world, kind, log_heights, steps):
    """ONE proof over the row shards of every matrix, all ranks (kind "u32_add": one circuit of 2^log_heights[0] rows; "multi:K":
    BASELINE configs[3] shape). Compared with the same proof on one GPU (rank 0): the bytes must be identical."""
    import hashlib
    import torch
    system = ms.System(kind, **prove_params(args))
    if kind == "u32_add":
        byte, add, claims = u32_add_traces(log_heights[0])
        traces = [byte, add]
    else:
        traces, claims = ms.multi_workload(log_heights)
    rs = msd.RowShardProver(ctx, system)
    heights = [t.shape[0] for t in traces]
    mine = []
    for t in traces:  # every rank pins only the rows it reads
        r0, n = rs.block_rows(t.shape[0], t.shape[1])
        mine.append(ctx.pinned_copy(t[r0:r0 + n]))
    claims_p = ctx.pinned_copy(np.ascontiguousarray(claims))
    times = []
    for it in range(steps + 1):
        msd.barrier()
        torch.cuda.synchronize()
        if it == steps:
            rs.comm.seconds.clear()
            bytes0 = rs.bytes_dev
        t0 = time.perf_counter()
        proof = rs.prove(mine, claims_p, heights=heights)
        if it:
            times.append((time.perf_counter() - t0) * 1e3)
    out = {"kind": kind, "log_heights": log_heights, "ms": msd.max_over_ranks(float(np.median(times))), "stages_ms_rank0": rs.last_stage_ms,
           "proof_bytes": len(proof), "digest": hashlib.sha256(proof).hexdigest(),
           "device_bytes_exchanged_this_rank": int(rs.bytes_dev - bytes0), "peer_memory": rs.peer_memory,
           "comm_ms_this_rank": {k: round(v * 1e3, 3) for k, v in rs.comm.seconds.items()},
           "timing": "host wall clock around the call on every rank (row blocks of pinned host traces in, proof bytes out), median, max over ranks"}
    out["all_ranks_same_proof"] = len(set(msd.gather_digests([bytes.fromhex(out["digest"])]))) == 1
    rs.close()
    if rank == 0:
        single = ms.Prover(ctx, system)
        pinned = [ctx.pinned_copy(t) for t in traces]
        ts = []
        for it in range(3):
            t0 = time.perf_counter()
            want = single.prove(pinned, claims_p)
            ts.append((time.perf_counter() - t0) * 1e3)
        out["single_gpu_ms"] = float(np.min(ts[1:]))
        out["identical_to_single_gpu_proof"] = want == proof
        out["speedup_vs_one_gpu"] = out["single_gpu_ms"] / out["ms"]
        single.close()
    msd.barrier()
    return out


def run_reference(args):
    """The reference arm: the CPU restatement of the SAME step (both trace commitments of configs[1] at the full 2^log_rows
    rows) on every host core, plus its prove() at the same rows and at 2^big rows. Imports nothing of the product."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    stages = u32_add_workload(args.log_rows)
    log_sample = min(args.log_rows, args.cpu_log_rows)
    sample = sample_stages(stages, log_sample)
    for _ in range(min(args.warmup, 1)):
        cpu_commit_time(sample, args.log_blowup)
    times = []
    threads = 1
    for _ in range(args.steps):
        dt, threads = cpu_commit_time(sample, args.log_blowup)
        times.append(dt)
    elems = committed_elements(sample, args.log_blowup)
    ms = 1e3 * float(np.mean(times))
    value = elems / (ms / 1e3) / 1e9
    desc = ("the full step: both trace commitments at 2^%d rows, %d steps" % (args.log_rows, args.steps) if log_sample == args.log_rows
            else "first 2^%d of 2^%d rows of each trace matrix, %d steps" % (log_sample, args.log_rows, args.steps))
    prove = prove_big = None
    if not args.no_prove:
        prove = cpu_prove_time(args, min(args.log_rows, args.cpu_prove_log_rows))
        if args.big_log_rows > args.log_rows:
            prove_big = cpu_prove_time(args, args.big_log_rows)
    orc, L = load_oracle()
    print(json.dumps({
        "impl": "reference", "metric": "lde_merkle_gelem_per_s", "value": value, "unit": "Gelem/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": "Gelem/s", "cores": threads, "kind": "port", "sample": desc,
                         "simd_level": int(L.orc_simd_level()), "baseline_is_reference_binary": False, "note": CPU_NOTE},
        "e2e": {"value": value, "unit": "Gelem/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "prove": prove, "prove_big": prove_big,
    }))


def workload_config(args):
    return {"workload": "BASELINE configs[1]: U32-add circuit with lookups at 2^%d rows + 256-row byte table, "
                        "stage-1 (w=1,14) and stage-2 (w=2,26) pcs.commit, log_blowup=%d" % (args.log_rows, args.log_blowup),
            "log_rows": args.log_rows, "log_blowup": args.log_blowup,
            "cache": "inputs (%d MB/step) and LDE outputs exceed the 126 MB L2; no explicit flush" %
                     ((40 << args.log_rows) * 8 >> 20)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-rows", type=int, default=20)
    ap.add_argument("--log-blowup", type=int, default=1)
    ap.add_argument("--cpu-log-rows", type=int, default=20, help="rows of the CPU-baseline commit (default: the full 2^20)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-prove-log-rows", type=int, default=20, help="rows of the CPU prove() baseline (default: the GPU leg's)")
    ap.add_argument("--big-log-rows", type=int, default=22, help="second prove() leg, GPU and CPU (north_star: 2^22 rows); 0 = off")
    ap.add_argument("--no-prove", action="store_true", help="skip the prove() leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy "
                    "(commitment roots, a seeded sample of the LDE rows, proof bytes)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path; it has no meaning with --impl reference")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    import multi_stark_b200 as ms
    from multi_stark_b200 import dist as msd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libmsgpu has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("TORCH_NCCL_SHOW_EAGER_INIT_P2P_SERIALIZATION_WARNING", "false")
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner out of stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    stages = u32_add_workload(args.log_rows, seed=rank)
    B = args.log_blowup
    stream = torch.cuda.Stream()  # a real (non-default) stream shared by torch's events and libmsgpu's launches
    torch.cuda.set_stream(stream)
    ctx = ms.GpuContext(local_rank, stream=stream.cuda_stream)
    pcs = ms.GpuPcs(ctx, B)

    # host side: pinned buffers (what a Rust caller would hand to msgpu_commit); device side: resident copies
    pinned = [[torch.from_numpy(m.view(np.int64)).pin_memory() for m in st] for st in stages]
    pinned_np = [[t.numpy().view(np.uint64) for t in st] for st in pinned]
    resident = [[t.cuda(non_blocking=True) for t in st] for st in pinned]
    resident_args = [[(t.data_ptr(), t.shape[0], t.shape[1]) for t in st] for st in resident]
    torch.cuda.synchronize()

    def step_resident(keep=None):
        roots = []
        for st in resident_args:
            root, pd = pcs.commit_dev(st)
            roots.append(bytes(root))
            if keep is None:
                pd.free()
            else:
                keep.append(pd)
        return roots

    def step_e2e_serial():
        roots = []
        for st in pinned_np:
            root, pd = pcs.commit(st)
            roots.append(bytes(root))
            pd.free()
        return roots

    # The same commitments through the two-step host-pointer ABI (msgpu_upload_begin / msgpu_commit_upload): the upload of
    # commitment k + 1 is enqueued on the copy stream BEFORE the kernels of commitment k, so in steady state PCIe and the SMs
    # work at the same time (a prover streams its next trace in while the current one is extended).
    pend = {"up": None}

    def step_e2e():
        roots = []
        for i, st in enumerate(pinned_np):
            up = pend["up"] if pend["up"] is not None else pcs.upload_begin(st)
            pend["up"] = pcs.upload_begin(pinned_np[(i + 1) % len(pinned_np)])
            root, pd = pcs.commit_upload(up)
            roots.append(bytes(root))
            pd.free()
        return roots

    def e2e_drain():
        if pend["up"] is not None:
            pcs.upload_free(pend["up"])
            pend["up"] = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, profile=False, last=None):
        """`last`, if given, runs in place of `fn` as the final timed step."""
        barrier()
        if profile:
            ctx.profile_begin()
        l0 = ctx.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            out = last() if last is not None and i == steps - 1 else fn()
        e1.record()
        torch.cuda.synchronize()
        ms_total = e0.elapsed_time(e1)
        prof = ctx.profile_end() if profile else None
        launches = ctx.launches - l0
        ms_total = msd.max_over_ranks(ms_total)  # the job takes as long as its slowest rank
        barrier()
        return ms_total, launches, prof, out

    for _ in range(max(args.warmup, 3)):
        r_res = step_resident()
    for _ in range(2):
        r_e2e = step_e2e()
    e2e_drain()
    assert r_res == r_e2e == step_e2e_serial(), "resident and host-pointer paths disagree"

    sampler = ClockSampler(local_rank)
    sampler.start()
    t_s = time.perf_counter()
    while len(sampler.lines) < 1 and time.perf_counter() - t_s < 3.0:  # nvidia-smi needs ~0.5 s to print its first sample
        step_resident()
    kept = []  # ProverData of the last timed step, kept for --dump-outputs
    ms_res, launches, prof, _ = timed(step_resident, args.steps, profile=True,
                                      last=(lambda: step_resident(keep=kept)) if args.dump_outputs else None)
    if kept:
        if rank == 0:
            dump_commit(args.dump_outputs, kept)
        for pd in kept:
            pd.free()
    ms_e2e, _, _, _ = timed(step_e2e, args.steps)
    e2e_drain()
    ms_e2e_serial, _, _, _ = timed(step_e2e_serial, args.steps)
    t_s = time.perf_counter()
    while len(sampler.lines) < 8 and time.perf_counter() - t_s < 2.0:  # same kernels, untimed: enough samples under load
        step_resident()
    clocks = sampler.stop()

    elems = committed_elements(stages, B)
    ms_step = ms_res / args.steps
    value = world * elems / (ms_step / 1e3) / 1e9
    e2e_value = world * elems / (ms_e2e / args.steps / 1e3) / 1e9
    h2d = sum(m.nbytes for st in stages for m in st)
    replicas = None
    if world > 1:
        # N > 1: the headline is ONE job over all ranks (the same two commitments, every matrix split by rows: strong scaling);
        # the independent replicas measured above (no data-path collective) are kept as an extra key
        replicas = {"value": value, "unit": "Gelem/s", "ms_per_step": ms_step, "e2e_value": e2e_value, "scaling": "weak",
                    "note": "every rank commits its own instance of the step: independent units, no data-path collective"}
        rs_system = ms.System("u32_add", **prove_params(args))
        rs = msd.RowShardProver(ctx, rs_system)
        ms_step, ms_host, rs_roots, h2d = rowshard_commit_leg(args, ms, msd, ctx, rs, rank, world, args.steps, max(args.warmup, 3))
        n_commits = 2 * (args.steps + max(args.warmup, 3)) * len(stages)
        rs_bytes_per_step = rs.bytes_dev // max(n_commits // len(stages), 1)
        rs_peer = rs.peer_memory
        rs.close()
        value = elems / (ms_step / 1e3) / 1e9
        e2e_value = elems / (ms_host / 1e3) / 1e9
        ms_e2e = ms_host * args.steps
        # rank 0's replica commits the same matrices (seed 0): the sharded roots must be the single-GPU roots
        rs_roots_ok = (rs_roots == step_resident()) if rank == 0 else None

    # roofline of the dominant stage: algorithmic bytes (SURVEY 8d) / CUDA-event time of its launches
    peak, peak_src = measured_peaks()
    stage_ms, stage_launch, kernels = {}, {}, []
    for rec in prof:
        stage_ms[rec["stage"]] = stage_ms.get(rec["stage"], 0.0) + rec["ms"] / args.steps
        stage_launch[rec["stage"]] = stage_launch.get(rec["stage"], 0) + rec["launches"] // args.steps
        kernels.append({"stage": rec["stage"], "kernel": rec["kernel"], "launches_per_step": rec["launches"] // args.steps,
                        "ms_per_step": rec["ms"] / args.steps})
    alg = {"lde": lde_bytes(stages, B), "merkle": merkle_bytes(stages, B)}
    stages_out = []
    for st, msv in stage_ms.items():
        if st in alg and msv > 0:
            gbs = alg[st] / (msv / 1e3) / 1e9
            stages_out.append({"stage": st, "ms_per_step": msv, "launches_per_step": stage_launch[st],
                               "algorithmic_bytes": alg[st], "achieved_gbs": gbs, "frac": gbs / peak})
    dom = max(stages_out, key=lambda s: s["ms_per_step"]) if stages_out else None
    roofline = None
    if dom:
        # integer roofline: both stages are bound by the INT32 pipes, not by HBM. Peak = live microbenchmark
        # (msgpu_measure_int_peak); instructions per step = ncu counters of the same step (data independent).
        ipk = ctx.measure_int_peak()
        counters, counters_file = step_counters()
        default_shape = args.log_rows == 20 and args.log_blowup == 1
        for st in stages_out:
            c = counters["stages"].get(st["stage"]) if counters and default_shape else None
            if c:
                rate = c["thread_inst_per_step"] / (st["ms_per_step"] / 1e3) / 1e9
                st["int_pipe"] = {"thread_inst_per_step": c["thread_inst_per_step"], "achieved_ginst_s": rate,
                                  "frac_of_mixed_peak": rate / ipk["mixed"]}
                st["dram_traffic_bytes_per_step"] = c["dram_bytes_per_step"]
        traffic = dom.get("dram_traffic_bytes_per_step")
        top = max((k for k in kernels if k["stage"] == dom["stage"]), key=lambda k: k["ms_per_step"])
        # the dominant kernel on its own: k_lde_mid reads every evaluation once and writes every LDE element once, i.e. it
        # moves the whole stage's algorithmic bytes by itself (the strided passes around it are in-place re-reads)
        dom_kernel = {"name": top["kernel"], "launches_per_step": top["launches_per_step"], "ms_per_step": top["ms_per_step"]}
        if top["kernel"] in ("k_lde_mid", "k_hash_rows_staged", "k_hash_rows_stream"):
            kb = dom["algorithmic_bytes"] if top["kernel"] == "k_lde_mid" else sum(
                8 * (m.shape[0] << B) * m.shape[1] + 32 * (m.shape[0] << B) for st in stages for m in st)
            dom_kernel.update({"algorithmic_bytes_per_launch": kb / top["launches_per_step"],
                               "achieved_gbs": kb / (top["ms_per_step"] / 1e3) / 1e9,
                               "frac": kb / (top["ms_per_step"] / 1e3) / 1e9 / peak})
            kc = (counters or {}).get("kernels", {}).get(top["kernel"]) if default_shape else None
            if kc:
                dom_kernel["dram_traffic_bytes_per_launch"] = kc["dram_bytes_per_step"] / kc["launches_per_step"]
                dom_kernel["int_pipe_frac_of_mixed_peak"] = kc["thread_inst_per_step"] / (top["ms_per_step"] / 1e3) / 1e9 / ipk["mixed"]
        roofline = {"bound": "hbm", "stage": "%s (%d launches/step)" % (dom["stage"], dom["launches_per_step"]),
                    "kernel": "%s (%d launches/step, %.3f ms/step)" % (top["kernel"], top["launches_per_step"], top["ms_per_step"]),
                    "achieved": dom["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": dom["frac"],
                    "traffic": traffic / dom["launches_per_step"] if traffic else None,
                    "traffic_note": "dram read+write bytes per launch (ncu, %s); achieved/frac use ALGORITHMIC bytes per launch" % counters_file,
                    "peak_source": peak_src, "algorithmic_bytes_per_step": dom["algorithmic_bytes"],
                    "algorithmic_bytes_per_launch": dom["algorithmic_bytes"] / dom["launches_per_step"],
                    "share_of_step": dom["ms_per_step"] / ms_step, "dominant_kernel": dom_kernel,
                    "binding_resource": "INT32 pipes (ALU + FMA-heavy): see int_pipe; HBM is not the bound for this stage",
                    "int_pipe": {"unit": "G thread-inst/s", "peak_alu_only": ipk["alu"], "peak_imad_only": ipk["imad"],
                                 "peak_mixed": ipk["mixed"], "peak_source": "msgpu_measure_int_peak, live, CUDA events",
                                 "achieved": dom.get("int_pipe", {}).get("achieved_ginst_s"),
                                 "frac": dom.get("int_pipe", {}).get("frac_of_mixed_peak")},
                    "stages": stages_out, "kernels": kernels, "ncu_pipe_busy": ncu_pipe_busy()}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        log_sample = min(args.log_rows, args.cpu_log_rows)
        sample = sample_stages(stages, log_sample)
        dt, threads = cpu_commit_time(sample, B, reps=2)
        orc, L = load_oracle()
        cpu = {"value": committed_elements(sample, B) / dt / 1e9, "unit": "Gelem/s", "cores": threads, "kind": "port",
               "simd_level": int(L.orc_simd_level()), "baseline_is_reference_binary": False, "note": CPU_NOTE,
               "sample": ("the full step (both trace commitments at 2^%d rows), best of 2" % args.log_rows) if log_sample == args.log_rows
               else "first 2^%d of 2^%d rows of each trace matrix, best of 2" % (log_sample, args.log_rows)}
        # parity spot check of the timed path against the oracle on the same matrices
        for st in sample:
            want, h = orc.pcs_commit(L, st, B)
            L.orc_mmcs_free(h)
            got, pd = pcs.commit(st)
            pd.free()
            assert bytes(got) == want, "GPU root differs from the oracle"

    prove = prove_big = None
    if not args.no_prove:
        barrier()
        prove, proof = gpu_prove_leg(args, ms, ctx, args.log_rows, steps=args.steps, warmup=2, verify=(rank == 0), peak=peak)
        if args.dump_outputs and rank == 0:
            dump_proof(args.dump_outputs, "prove_proof", proof)
        if world > 1:
            prove["ms_max_over_ranks"] = msd.max_over_ranks(prove["ms"])
            prove["proofs_per_s_all_ranks"] = world * 1e3 / prove["ms_max_over_ranks"]
            prove["proof_digests"] = [d.hex()[:16] for d in msd.gather_digests([bytes.fromhex(prove["digest"])])]
        if cpu is not None:
            prove["cpu"] = cpu_prove_time(args, min(args.log_rows, args.cpu_prove_log_rows))
            if prove["cpu"]["rows"] == prove["rows"]:
                prove["identical_to_cpu_proof"] = prove["cpu"]["digest"] == prove["digest"]
                prove["speedup_vs_cpu_port"] = prove["cpu"]["ms"] / prove["ms"]
        barrier()
        # north_star: prove() at 2^22 rows against the host-core parallel CPU prover, both measured here
        if world == 1 and args.big_log_rows > args.log_rows:
            prove_big, proof = gpu_prove_leg(args, ms, ctx, args.big_log_rows, steps=args.steps, warmup=1, verify=(rank == 0), peak=peak)
            if args.dump_outputs:
                dump_proof(args.dump_outputs, "prove_big_proof", proof)
            if cpu is not None:
                prove_big["cpu"] = cpu_prove_time(args, args.big_log_rows)
                prove_big["identical_to_cpu_proof"] = prove_big["cpu"]["digest"] == prove_big["digest"]
                prove_big["speedup_vs_cpu_port"] = prove_big["cpu"]["ms"] / prove_big["ms"]
        if world > 1:
            prove["sharded"] = sharded_prove_leg(args, ms, msd, ctx, rank, world, args.steps)
            # every matrix split by rows over all ranks: one tall circuit (2^log_rows and 2^big rows) and the 7-circuit system
            prove["rowshard"] = rowshard_prove_leg(args, ms, msd, ctx, rank, world, "u32_add", [args.log_rows], args.steps)
            if args.big_log_rows > args.log_rows:
                prove_big = rowshard_prove_leg(args, ms, msd, ctx, rank, world, "u32_add", [args.big_log_rows], args.steps)
            lhs = [min(h, args.log_rows + 2) for h in (22, 21, 21, 20, 20, 19, 18)]
            prove["rowshard_multi7"] = rowshard_prove_leg(args, ms, msd, ctx, rank, world, "multi:7", lhs, args.steps)

    if rank == 0:
        if roofline is not None and prove is not None and prove.get("stage_roofline"):
            roofline["prove_stages"] = prove["stage_roofline"]
        print(json.dumps({
            "metric": "lde_merkle_gelem_per_s", "value": value, "unit": "Gelem/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak" if world == 1 else "strong",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": workload_config(args),
            "e2e": {"value": e2e_value, "unit": "Gelem/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 64,
                    "ms_per_step": ms_e2e / args.steps,
                    "call": ("msgpu_upload_begin + msgpu_commit_upload on pinned host matrices, the next commitment's upload enqueued "
                             "before this one's kernels") if world == 1 else
                            "msh_rowshard_commit on pinned host row blocks (each rank uploads 1 / N of every tall matrix)",
                    "serial": {"value": world * elems / (ms_e2e_serial / args.steps / 1e3) / 1e9, "ms_per_step": ms_e2e_serial / args.steps,
                               "call": "msgpu_commit (upload, then kernels, then root; no overlap between calls)"}},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "prove": prove,
            "prove_big": prove_big, "replicas": replicas,
            "sharding": None if world == 1 else {
                "mode": "every committed matrix split by rows over the ranks (host/rowshard_backend.hpp): ONE job, the same work at every N",
                "exchange": ("peer memory: NVLink stores / loads issued by this library's kernels into CUDA-IPC windows (csrc/peer.cu), "
                             "flag barriers in peer memory; no NCCL call on the data path") if rs_peer else "NCCL all-to-all / all-gather",
                "device_bytes_exchanged_this_rank_per_step": int(rs_bytes_per_step), "roots_equal_single_gpu_commit": rs_roots_ok},
        }))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
