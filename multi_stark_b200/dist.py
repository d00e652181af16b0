"""Multi-GPU plumbing: one process per GPU, `torch.distributed` (NCCL on the GPU box, gloo in the CPU tests).

The commitment path shards by independent units -- whole proofs, or the circuit groups of SURVEY section 8(e) partitioning A --
so there is NO data-path collective: every rank runs the full single-GPU pipeline on its own units. Ranks exchange only
what the protocol makes public anyway (32-byte commitments / proof digests) and the timing needed for an honest aggregate
(max over ranks). The reference has no multi-process story at all (SURVEY section 2: rayon inside one process)."""
import contextlib
import ctypes as _C
import hashlib
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

from ._ffi import check, host_error, host_lib
from .pcs import ProverData
from .system import ProverBase


def world():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def rank():
    return dist.get_rank() if dist.is_available() and dist.is_initialized() else 0


def _device():
    """tensors for collectives live where the backend wants them"""
    if dist.is_initialized() and dist.get_backend() == "nccl":
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


def shard_units(n_units, world_size=None, r=None):
    """Contiguous balanced partition of unit ids [0, n_units): the first n_units % world ranks get one more."""
    w = world() if world_size is None else world_size
    r = rank() if r is None else r
    if w <= 0 or not 0 <= r < w:
        raise ValueError("bad rank / world size")
    base, rem = divmod(n_units, w)
    lo = r * base + min(r, rem)
    return range(lo, lo + base + (1 if r < rem else 0))


def barrier():
    if world() > 1:
        dist.barrier()


def max_over_ranks(value):
    """Device-side max of a per-rank scalar (elapsed ms): the job takes as long as its slowest rank."""
    if world() == 1:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=_device())
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(value):
    if world() == 1:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=_device())
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def gather_digests(digests):
    """All-gather of this rank's 32-byte digests (commitments or SHA-256 of proof bytes), one per local unit.
    Returns the list over all ranks in unit order. Every rank must contribute the same count per unit shard rule."""
    w = world()
    if w == 1:
        return list(digests)
    counts = torch.tensor([len(digests)], dtype=torch.int64, device=_device())
    all_counts = [torch.zeros_like(counts) for _ in range(w)]
    dist.all_gather(all_counts, counts)
    cap = max(int(c.item()) for c in all_counts)
    buf = torch.zeros((max(cap, 1), 32), dtype=torch.uint8)
    for i, d in enumerate(digests):
        if len(d) != 32:
            raise ValueError("digests must be 32 bytes")
        buf[i] = torch.frombuffer(bytearray(d), dtype=torch.uint8)
    buf = buf.to(_device())
    out = [torch.zeros_like(buf) for _ in range(w)]
    dist.all_gather(out, buf)
    res = []
    for r_, c in enumerate(all_counts):
        rows = out[r_].cpu()
        for i in range(int(c.item())):
            res.append(bytes(rows[i].tolist()))
    return res


def proof_digest(proof_bytes):
    return hashlib.sha256(proof_bytes).digest()


def prove_sharded(units, prove_fn):
    """Runs prove_fn(unit) for the units of this rank's shard; returns (local {unit_id: proof}, digests of ALL units in
    unit order, gathered over the ranks). `units` is the same list on every rank."""
    mine = shard_units(len(units))
    proofs = {u: prove_fn(units[u]) for u in mine}
    digests = gather_digests([proof_digest(proofs[u]) for u in mine])
    return proofs, digests


# ------------------------------------------------------------------------------------------------------------------
# One proof over several GPUs: the collectives the sharded prover (host/dist_backend.hpp) calls back into.
# ------------------------------------------------------------------------------------------------------------------
_ALLGATHER = _C.CFUNCTYPE(_C.c_int, _C.c_void_p, _C.c_void_p, _C.c_void_p, _C.c_uint64)
_BCAST = _C.CFUNCTYPE(_C.c_int, _C.c_void_p, _C.c_void_p, _C.c_uint64, _C.c_int32)
_SENDRECV = _C.CFUNCTYPE(_C.c_int, _C.c_void_p, _C.c_void_p, _C.c_uint64, _C.c_int32, _C.c_int32)
_ALLTOALL = _C.CFUNCTYPE(_C.c_int, _C.c_void_p, _C.c_void_p, _C.POINTER(_C.c_uint64), _C.c_void_p, _C.POINTER(_C.c_uint64))
_ALLGATHER_DEV = _C.CFUNCTYPE(_C.c_int, _C.c_void_p, _C.c_void_p, _C.c_void_p, _C.c_uint64)


class MshComm(_C.Structure):
    """`msh_comm` of host/dist_backend.hpp"""
    _fields_ = [("user", _C.c_void_p), ("rank", _C.c_int32), ("world", _C.c_int32), ("allgather_host", _ALLGATHER),
                ("bcast_host", _BCAST), ("sendrecv_dev", _SENDRECV), ("alltoall_dev", _ALLTOALL), ("allgather_dev", _ALLGATHER_DEV), ("peer_memory", _C.c_int32)]


class _DevView:
    """A raw device range as something torch.as_tensor understands (zero copy)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2,
                                         "strides": None}


class TorchComm:
    """Collectives over the default torch.distributed group. Host buffers travel as CPU tensors over gloo, or staged through
    the device over NCCL; device buffers travel device-to-device over NCCL (NVLink), or staged through pinned host memory
    over gloo (the single-GPU tests run two ranks on one device that way). Each collective raises on failure; `struct` holds
    them as the C callbacks of `msh_comm`, which report a failure as 1 and its exception in `errors`."""

    def __init__(self, ctx, group=None):
        self.ctx = ctx
        self.group = group
        self.nccl = dist.get_backend(group) == "nccl"
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.bytes_dev = 0   # device bytes sent or received by this rank (reported by bench / tools)
        self.bytes_host = 0
        self.errors = []
        self.seconds = {}    # wall time spent inside the collectives, by kind
        self._stage = None
        self._seq = 0
        self.trace = bool(os.environ.get("MSH_TRACE"))
        self.trace2 = int(os.environ.get("MSH_TRACE") or 0) >= 2
        if self.nccl:
            # NCCL calls are ordered against torch's CURRENT stream, the library's kernels against the context's: they must be
            # the same stream, or a send could leave before the kernel that fills the buffer has run (ADVICE r1)
            cur = torch.cuda.current_stream().cuda_stream
            if int(ctx.stream or 0) != int(cur):
                raise ValueError("TorchComm: create the GpuContext on torch's current stream (GpuContext(dev, stream=torch.cuda.current_stream().cuda_stream))")
        self._cb = (self._callback(_ALLGATHER, self.allgather_host), self._callback(_BCAST, self.bcast_host),
                    self._callback(_SENDRECV, self.sendrecv_dev), self._callback(_ALLTOALL, self.all_to_all_dev),
                    self._callback(_ALLGATHER_DEV, self.allgather_dev))  # keep the thunks alive
        # peer memory (csrc/peer.cu): NCCL ranks of one node, one GPU each; MSGPU_P2P=0 keeps every exchange on the collectives
        self.peer_memory = int(self.nccl and self.world > 1 and os.environ.get("MSGPU_P2P", "1") != "0"
                               and torch.cuda.device_count() >= self.world)
        self.struct = MshComm(None, self.rank, self.world, *self._cb, self.peer_memory)

    def _callback(self, cfunctype, collective):
        """`collective` as an msh_comm callback (its first argument, `user`, is unused)"""
        def cb(user, *args):
            if self.trace2:
                print("[comm %d] %s%r" % (self.rank, collective.__name__, args), file=sys.stderr, flush=True)
            try:
                collective(*args)
                return 0
            except Exception as e:  # never unwind into C++
                self.errors.append(repr(e))
                return 1
        return cfunctype(cb)

    @contextlib.contextmanager
    def _timed(self, kind):
        t0 = time.perf_counter()
        try:
            yield
        finally:
            self.seconds[kind] = self.seconds.get(kind, 0.0) + time.perf_counter() - t0

    def _global(self, r):
        return dist.get_global_rank(self.group, r) if self.group is not None else r

    def _same_call(self, kind):
        """gloo only: the staged device exchanges below move data pairwise, so a rank that SKIPPED one (a rank-dependent branch
        around a collective -- a hang under NCCL) would go unnoticed by the single-GPU tests. Every rank announces (sequence
        number, kind) first; a mismatch fails the call on every rank."""
        if self.nccl:
            return
        self._seq += 1
        mine = torch.tensor([self._seq, kind], dtype=torch.int64)
        allv = torch.empty(2 * self.world, dtype=torch.int64)
        dist.all_gather_into_tensor(allv, mine, group=self.group)
        if any(allv[2 * r] != self._seq or allv[2 * r + 1] != kind for r in range(self.world)):
            raise RuntimeError("ranks disagree on the sequence of device collectives: %s" % allv.tolist())

    # ---- host buffers
    def _host_tensor(self, ptr, nbytes):
        return torch.frombuffer((_C.c_uint8 * nbytes).from_address(ptr), dtype=torch.uint8)

    def _staging(self, nbytes):
        """persistent pinned-host and device staging buffers (grow-only): a fresh pageable tensor per call costs ms"""
        if self._stage is None or self._stage[0].numel() < nbytes:
            cap = 1 << max(16, int(nbytes - 1).bit_length())
            dev = torch.device("cuda", torch.cuda.current_device())
            self._stage = (torch.empty(cap, dtype=torch.uint8).pin_memory(), torch.empty(cap, dtype=torch.uint8, device=dev))
        return self._stage

    def allgather_host(self, send, recv, nbytes):
        """Host all-gather of equal chunks: recv = world chunks of nbytes in rank order."""
        with self._timed("allgather"):
            nbytes = int(nbytes)
            s = self._host_tensor(send, nbytes)
            r = self._host_tensor(recv, nbytes * self.world)
            if self.nccl:
                tr = [time.perf_counter()]
                pin, dev = self._staging(nbytes * (self.world + 1))
                tr.append(time.perf_counter())
                total = nbytes * self.world
                _C.memmove(pin.data_ptr(), send, nbytes)  # (torch's CPU copy_ spins up its thread pool: ms for 1 MB)
                dev[total:total + nbytes].copy_(pin[:nbytes], non_blocking=True)
                tr.append(time.perf_counter())
                dist.all_gather_into_tensor(dev[:total], dev[total:total + nbytes], group=self.group)
                tr.append(time.perf_counter())
                pin[:total].copy_(dev[:total], non_blocking=True)
                torch.cuda.current_stream().synchronize()
                tr.append(time.perf_counter())
                _C.memmove(recv, pin.data_ptr(), total)
                tr.append(time.perf_counter())
                if self.trace:
                    print("[comm] rank %d allgather %d B: staging %.3f, h2d %.3f, nccl call %.3f, d2h+sync %.3f, copy out %.3f ms" % (
                        (self.rank, nbytes) + tuple((b - a) * 1e3 for a, b in zip(tr, tr[1:]))), file=sys.stderr, flush=True)
            else:
                dist.all_gather_into_tensor(r, s.clone(), group=self.group)
            self.bytes_host += nbytes * self.world

    def bcast_host(self, buf, nbytes, root):
        """Host broadcast of nbytes from rank `root`."""
        with self._timed("bcast"):
            nbytes = int(nbytes)
            t = self._host_tensor(buf, nbytes)
            if self.nccl:
                pin, dev = self._staging(nbytes)
                if self.rank == root:
                    _C.memmove(pin.data_ptr(), buf, nbytes)
                    dev[:nbytes].copy_(pin[:nbytes], non_blocking=True)
                dist.broadcast(dev[:nbytes], src=self._global(root), group=self.group)
                if self.rank != root:
                    pin[:nbytes].copy_(dev[:nbytes], non_blocking=True)
                    torch.cuda.current_stream().synchronize()
                    _C.memmove(buf, pin.data_ptr(), nbytes)
            else:
                dist.broadcast(t, src=self._global(root), group=self.group)
            self.bytes_host += nbytes

    # ---- device buffers
    def _d2h(self, dev, nbytes):
        """gloo staging: nbytes of device memory in a new host tensor"""
        host = torch.empty(nbytes, dtype=torch.uint8)
        if nbytes:
            check(self.ctx.L.msgpu_memcpy_d2h(self.ctx.h, _C.c_void_p(host.data_ptr()), _C.c_void_p(dev), nbytes))
        return host

    def _h2d(self, dev, host):
        """gloo staging: a host tensor back to device memory"""
        if host.numel():
            check(self.ctx.L.msgpu_memcpy_h2d(self.ctx.h, _C.c_void_p(dev), _C.c_void_p(host.data_ptr()), host.numel()))

    def sendrecv_dev(self, dev, nbytes, src, dst):
        """Device point-to-point: rank `src` sends nbytes at `dev`, rank `dst` receives them at its `dev`."""
        with self._timed("sendrecv"):
            nbytes = int(nbytes)
            self.bytes_dev += nbytes
            if self.nccl:
                t = torch.as_tensor(_DevView(dev, nbytes), device=torch.device("cuda", torch.cuda.current_device()))
                if self.rank == src:
                    dist.send(t, dst=self._global(dst), group=self.group)
                else:
                    dist.recv(t, src=self._global(src), group=self.group)
                torch.cuda.current_stream().synchronize()
            elif self.rank == src:
                dist.send(self._d2h(dev, nbytes), dst=self._global(dst), group=self.group)
            else:
                host = torch.empty(nbytes, dtype=torch.uint8)
                dist.recv(host, src=self._global(src), group=self.group)
                self._h2d(dev, host)

    def all_to_all_dev(self, send_ptr, send_counts, recv_ptr, recv_counts):
        """Device all-to-all with per-peer byte counts (chunks in rank order in both buffers)."""
        with self._timed("all_to_all"):
            self._same_call(1)
            send_counts = [int(send_counts[k]) for k in range(self.world)]
            recv_counts = [int(recv_counts[k]) for k in range(self.world)]
            self.bytes_dev += sum(send_counts) - send_counts[self.rank] + sum(recv_counts) - recv_counts[self.rank]
            if self.nccl:
                dev = torch.device("cuda", torch.cuda.current_device())
                empty = torch.empty(0, dtype=torch.uint8, device=dev)
                s = torch.as_tensor(_DevView(send_ptr, sum(send_counts)), device=dev) if sum(send_counts) else empty
                r = torch.as_tensor(_DevView(recv_ptr, sum(recv_counts)), device=dev) if sum(recv_counts) else empty
                # stream-ordered on the context's stream (checked in __init__): later kernels see the data, no host wait needed
                dist.all_to_all_single(r, s, output_split_sizes=recv_counts, input_split_sizes=send_counts, group=self.group)
                return
            # gloo: staged through the host, pairwise
            so = [sum(send_counts[:k]) for k in range(self.world)]
            ro = [sum(recv_counts[:k]) for k in range(self.world)]
            host_s = self._d2h(send_ptr, sum(send_counts))
            host_r = torch.empty(sum(recv_counts), dtype=torch.uint8)
            reqs = []
            for k in range(self.world):
                if k == self.rank:
                    host_r[ro[k]:ro[k] + recv_counts[k]] = host_s[so[k]:so[k] + send_counts[k]]
                    continue
                if send_counts[k]:
                    reqs.append(dist.isend(host_s[so[k]:so[k] + send_counts[k]], dst=self._global(k), group=self.group))
                if recv_counts[k]:
                    reqs.append(dist.irecv(host_r[ro[k]:ro[k] + recv_counts[k]], src=self._global(k), group=self.group))
            for q in reqs:
                q.wait()
            self._h2d(recv_ptr, host_r)

    def allgather_dev(self, send, recv, nbytes):
        """Device all-gather of equal chunks: recv = world chunks of nbytes in rank order."""
        with self._timed("allgather_dev"):
            self._same_call(2)
            nbytes = int(nbytes)
            self.bytes_dev += nbytes * (self.world - 1) * 2
            if self.nccl:
                dev = torch.device("cuda", torch.cuda.current_device())
                s = torch.as_tensor(_DevView(send, nbytes), device=dev)
                r = torch.as_tensor(_DevView(recv, nbytes * self.world), device=dev)
                dist.all_gather_into_tensor(r, s, group=self.group)  # stream-ordered, as the all-to-all
            else:  # gloo: staged through the host
                host = torch.empty(nbytes * self.world, dtype=torch.uint8)
                dist.all_gather_into_tensor(host, self._d2h(send, nbytes), group=self.group)
                self._h2d(recv, host)


def assign_owners(heights, world_size):
    """Circuit -> rank for one sharded proof. Circuits of one trace height must share a rank (their rows share leaf digests
    and reduced openings); height classes are placed greedily, heaviest first, on the least loaded rank. `heights[i]` = trace
    rows of circuit i (0 = inactive; such circuits go to rank 0), weights = rows (a proxy for the LDE + Merkle work).
    Deterministic, so every rank computes the same assignment."""
    classes = {}
    for i, h in enumerate(heights):
        classes.setdefault(int(h), []).append(i)
    load = [0] * world_size
    owner = [0] * len(heights)
    for h in sorted(classes, reverse=True):
        if h == 0:
            continue
        r = min(range(world_size), key=lambda k: (load[k], k))
        load[r] += h * len(classes[h])
        for i in classes[h]:
            owner[i] = r
    return owner


class _ShardedProver(ProverBase):
    """A prover whose backend calls back into a TorchComm; its errors carry the communicator's. No __del__: the teardown
    unmaps peer memory, so these provers are freed by an explicit close()."""

    def __init__(self, ctx, system, group, create, *args):
        self.comm = TorchComm(ctx, group)
        super().__init__(ctx, system, create, _C.byref(self.comm.struct), *args)

    def _error(self, code):
        return host_error(code, "; ".join(self.comm.errors))

    @property
    def bytes_dev(self):
        """device bytes this rank exchanged so far"""
        return self.comm.bytes_dev


class DistProver(_ShardedProver):
    """`System::prove_multiple_claims` (src/prover.rs:289-603) as ONE proof over the ranks of a torch.distributed group: each
    rank owns whole circuits (`owner[i]`), builds and commits their traces and answers their openings; the proof bytes are
    identical on every rank and identical to the single-GPU proof."""

    def __init__(self, ctx, system, owner, group=None):
        self.owner = [int(o) for o in owner]
        if len(self.owner) != system.num_circuits:
            raise ValueError("one owner per circuit expected")
        super().__init__(ctx, system, group, host_lib().msh_dist_prover_create, (_C.c_int32 * len(self.owner))(*self.owner))

    def prove(self, traces, heights, claims):
        """traces[i]: (h x main_width) uint64 array for the circuits this rank owns, None otherwise; heights[i]: trace rows of
        EVERY circuit (0 = inactive); claims: as Prover.prove takes them, the same on every rank. Returns `Proof::to_bytes`."""
        mats = [None if t is None else np.ascontiguousarray(t, dtype=np.uint64) for t in traces]
        for i in range(self.system.num_circuits):
            if self.owner[i] == self.comm.rank and heights[i] and (mats[i] is None or mats[i].shape[0] != heights[i]):
                raise ValueError("the trace of circuit %d (owned by this rank) is missing or has the wrong height" % i)
        return self._prove([m.ctypes.data if (m is not None and m.size and self.owner[i] == self.comm.rank) else None
                            for i, m in enumerate(mats)], heights, claims)


class RowShardProver(_ShardedProver):
    """`System::prove_multiple_claims` as ONE proof over the ROW SHARDS of every committed matrix (host/rowshard_backend.hpp):
    rank d of N holds rows [d H / N, (d + 1) H / N) of every LDE, so a single tall circuit is proved by all GPUs. Every rank
    passes ALL traces (it reads only its row block of the tall ones); the proof bytes are identical on every rank and identical
    to the single-GPU proof."""

    def __init__(self, ctx, system, group=None):
        super().__init__(ctx, system, group, host_lib().msh_rowshard_prover_create)

    def shardable(self, height, width):
        """the backend's rule (RowShardBackend::shardable): such a trace is read as natural-order row blocks"""
        return self.H.msh_rowshard_shardable(self.h, int(height), int(width)) == 1

    @property
    def bytes_dev(self):
        """device bytes this rank exchanged so far: NCCL collectives + NVLink loads / stores of the peer-memory kernels"""
        return int(self.comm.bytes_dev) + int(self.H.msh_rowshard_peer_bytes(self.h))

    @property
    def peer_memory(self):
        """True when the ranks exchange matrices through each other's device memory (csrc/peer.cu) rather than NCCL"""
        return self.H.msh_rowshard_peer_memory(self.h) == 1

    def block_rows(self, height, width):
        """(row0, rows) of the part of a height x width trace this rank reads"""
        if not self.shardable(height, width):
            return 0, height
        rows = height // self.comm.world
        return rows * self.comm.rank, rows

    def commit(self, mats, heights, widths, host):
        """`Pcs::commit` over the row shards alone. host=False: mats[i] = DEVICE pointer of this rank's natural-order row block
        (block_rows(heights[i], widths[i])); host=True: mats[i] = numpy array holding the rows this rank reads. Returns the root."""
        n = len(mats)
        if host:
            keep = [np.ascontiguousarray(m, dtype=np.uint64) for m in mats]
            plist = [m.ctypes.data - self.block_rows(int(h), int(w))[0] * int(w) * 8 for m, h, w in zip(keep, heights, widths)]
        else:
            plist = [int(m) for m in mats]
        ptrs = (_C.c_void_p * n)(*plist)
        hs = (_C.c_uint64 * n)(*[int(h) for h in heights])
        ws = (_C.c_uint64 * n)(*[int(w) for w in widths])
        root = np.zeros(32, dtype=np.uint8)
        if self.H.msh_rowshard_commit(self.h, ptrs, hs, ws, n, 1 if host else 0, root.ctypes.data_as(_C.c_void_p)) != 0:
            raise self._error(-1)
        return bytes(root)

    def prove(self, traces, claims, heights=None):
        """traces[i]: (h x main_width) uint64 array of circuit i on EVERY rank (h = 0: inactive); claims: as Prover.prove takes
        them, the same on every rank. With `heights` (trace rows of every circuit) traces[i] may instead hold only the rows this
        rank reads -- block_rows(heights[i], width) -- so that no rank needs the whole of a tall trace in host memory.
        Returns `Proof::to_bytes`."""
        mats = [np.ascontiguousarray(t, dtype=np.uint64) for t in traces]
        if heights is None:
            return self._prove([m.ctypes.data if m.size else None for m in mats], [m.shape[0] for m in mats], claims)
        ptrs = []
        for m, h in zip(mats, heights):
            row0, rows = self.block_rows(int(h), m.shape[1])
            if m.shape[0] != rows:
                raise ValueError("a trace given as a row block must hold exactly the rows this rank reads")
            ptrs.append(m.ctypes.data - row0 * m.shape[1] * 8 if m.size else None)  # the library touches [row0, row0 + rows) only
        return self._prove(ptrs, heights, claims)


# ------------------------------------------------------------------------------------------------------------------
# Pcs::commit of ONE wide matrix over the ranks (SURVEY 8e partitioning B, BASELINE configs[2]): column blocks.
# ------------------------------------------------------------------------------------------------------------------
def column_blocks(width, world_size):
    """Contiguous balanced column blocks [c0, c1) per rank (the first width % world ranks get one more column)."""
    base, rem = divmod(width, world_size)
    out, c = [], 0
    for r in range(world_size):
        n = base + (1 if r < rem else 0)
        out.append((c, c + n))
        c += n
    return out


class WideCommit:
    """Prover data of a column-block sharded commitment: this rank's ROW shard of the LDE (every column, rows
    [rank * H / N, (rank + 1) * H / N) of the bit-reversed storage) with its Merkle subtree, and the top of the tree."""

    def __init__(self, ctx, comm, local, top, root, lde_height, widths, recv_buf):
        self.ctx, self.comm, self.local, self.top, self.root = ctx, comm, local, top, root
        self.lde_height, self.widths, self._recv = lde_height, widths, recv_buf

    def open_batch(self, indices):
        """Mmcs::open_batch: (rows [n, width], sibling paths [n, log2(H), 32]) -- the same on every rank. The row and the
        lower log2(H / N) siblings come from the rank that holds the row, the top log2(N) siblings from the top tree
        (which every rank holds)."""
        n, world = len(indices), self.comm.world
        shard = self.lde_height // world
        lo_depth, top_depth, width = shard.bit_length() - 1, world.bit_length() - 1, sum(self.widths)
        owner = [int(i) // shard for i in indices]
        rows = np.zeros((n, width), dtype=np.uint64)
        low = np.zeros((n, lo_depth, 32), dtype=np.uint8)
        mine = [k for k in range(n) if owner[k] == self.comm.rank]
        if mine:
            o, p = self.local.open_batch([int(indices[k]) % shard for k in mine])
            rows[mine] = o
            low[mine] = p
        if world == 1:
            return rows, low
        # every rank contributes the openings of the rows it holds (zeros elsewhere); pick each index from its owner
        blob = np.concatenate([rows.view(np.uint8).ravel(), low.ravel()])
        gathered = np.zeros(blob.size * world, dtype=np.uint8)
        self.comm.allgather_host(blob.ctypes.data, gathered.ctypes.data, blob.size)
        gathered = gathered.reshape(world, -1)
        all_rows = gathered[:, :rows.nbytes].copy().view(np.uint64).reshape(world, n, width)
        all_low = gathered[:, rows.nbytes:].reshape(world, n, lo_depth, 32)
        paths = np.zeros((n, lo_depth + top_depth, 32), dtype=np.uint8)
        for k in range(n):
            rows[k] = all_rows[owner[k], k]
            paths[k, :lo_depth] = all_low[owner[k], k]
        # the top tree has no matrices: sibling paths only
        tidx = np.array(owner, dtype=np.uint64)
        tp = np.zeros((n, top_depth, 32), dtype=np.uint8)
        dummy = np.zeros(1, dtype=np.uint64)
        check(self.ctx.L.msgpu_open_batch(self.ctx.h, self.top.h, tidx.ctypes.data_as(_C.c_void_p), n,
                                          dummy.ctypes.data_as(_C.c_void_p), tp.ctypes.data_as(_C.c_void_p)))
        paths[:, lo_depth:] = tp
        return rows, paths

    def free(self):
        for h in (self.local, self.top):
            if h is not None:
                h.free()
        if self._recv:
            self.ctx.free(self._recv)
            self._recv = None


def commit_wide_sharded(ctx, comm, block, width, log_blowup, timings=None, keep_block=False):
    """`Pcs::commit` (src/prover.rs:350) of one n x `width` matrix whose COLUMN block `column_blocks(width, N)[rank]` is
    `block` (host array n x w_r, canonical values) on this rank. Per rank: upload + coset LDE of the block (the NTT is
    column-local), ONE all-to-all that turns column blocks into row shards (the block's rows [d * H / N, (d+1) * H / N) are
    contiguous and go to rank d), leaf hashing of the shard's full rows + its Merkle subtree, then the N subtree roots are
    all-gathered and the top log2(N) levels built on every rank. Root and openings are bit-identical to a single-GPU commit."""
    L = ctx.L
    world, rank = comm.world, comm.rank
    if world & (world - 1):
        raise ValueError("column-block sharding needs a power-of-two number of ranks")
    blocks = column_blocks(width, world)
    widths = [c1 - c0 for c0, c1 in blocks]
    a = np.ascontiguousarray(block, dtype=np.uint64)
    n, w = a.shape
    if w != widths[rank] or min(widths) == 0:
        raise ValueError("this rank's block must have %d columns (and every rank at least one)" % widths[rank])
    H = n << log_blowup
    if H % world or H // world < 1:
        raise ValueError("LDE height must be a multiple of the number of ranks")
    shard = H // world
    t = [time.perf_counter()]
    d_in = ctx.upload_canonical(a)
    t.append(time.perf_counter())
    d_lde = ctx.malloc(H * w * 8)
    check(L.msgpu_coset_lde_batch_bitrev_dev(ctx.h, _C.c_void_p(d_in), n, w, log_blowup, 7, _C.c_void_p(d_lde)))
    ctx.free(d_in)
    ctx.sync()
    t.append(time.perf_counter())
    # all-to-all: chunk d of my LDE (rows of shard d, my columns) -> rank d; I receive shard `rank` of every block
    recv = ctx.malloc(shard * width * 8)
    send_counts = [shard * w * 8] * world
    recv_counts = [shard * ws * 8 for ws in widths]
    comm.all_to_all_dev(d_lde, send_counts, recv, recv_counts)
    if not keep_block:
        ctx.free(d_lde)
        d_lde = None
    ctx.sync()
    t.append(time.perf_counter())
    # the shard as N matrices of one height: their rows concatenate in column order inside the leaf hash
    ptrs, off = [], 0
    for ws in widths:
        ptrs.append(recv + off)
        off += shard * ws * 8
    pa = (_C.c_void_p * world)(*ptrs)
    hs = (_C.c_uint64 * world)(*([shard] * world))
    wa = (_C.c_uint64 * world)(*widths)
    h = _C.c_void_p()
    sub_root = np.zeros(32, dtype=np.uint8)
    check(L.msgpu_commit_ldes_dev(ctx.h, pa, hs, wa, world, 0, _C.byref(h), sub_root.ctypes.data_as(_C.c_void_p)))
    local = ProverData(ctx, h, bytes(sub_root))
    t.append(time.perf_counter())
    top, root = None, bytes(sub_root)
    if world > 1:
        roots = np.zeros(32 * world, dtype=np.uint8)
        comm.allgather_host(sub_root.ctypes.data, roots.ctypes.data, 32)
        d_roots = ctx.upload(roots)
        th = _C.c_void_p()
        r32 = np.zeros(32, dtype=np.uint8)
        hh = (_C.c_uint64 * 1)(world)
        pp = (_C.c_void_p * 1)(d_roots)
        check(L.msgpu_tree_from_digests(ctx.h, 1, hh, pp, _C.byref(th), r32.ctypes.data_as(_C.c_void_p)))
        ctx.free(d_roots)
        top, root = ProverData(ctx, th, bytes(r32)), bytes(r32)
    t.append(time.perf_counter())
    if timings is not None:
        for k, name in enumerate(["upload", "lde", "all_to_all", "leaf_hash_subtree", "top"]):
            timings[name] = timings.get(name, 0.0) + (t[k + 1] - t[k]) * 1e3
    wc = WideCommit(ctx, comm, local, top, root, H, widths, recv)
    wc.lde_block = d_lde  # this rank's column block of the LDE (H x w), kept for prove_wide_sharded
    return root, wc


def prove_wide_sharded(ctx, comm, prover, block, width, log_blowup, claims=None, timings=None):
    """`prove()` of a system with ONE wide, lookup-free circuit (BASELINE configs[2]) whose trace arrives as column blocks, one
    per rank. The stage-1 commitment -- upload, LDE and leaf hashing of 256 columns, 83 % of the single-GPU proof -- is made
    by all ranks (commit_wide_sharded); rank 0 then gathers the LDE blocks and the shards' digest layers over NVLink,
    assembles ordinary prover data (msgpu_pdata_from_parts) and runs the remaining stages alone. Returns the proof bytes on
    rank 0 (None elsewhere); they equal the single-GPU proof byte for byte. `prover` is a `Prover` on rank 0, None elsewhere."""
    L = ctx.L
    t = [time.perf_counter()]
    root, wc = commit_wide_sharded(ctx, comm, block, width, log_blowup, timings=timings, keep_block=True)
    t.append(time.perf_counter())
    world, rank = comm.world, comm.rank
    H, widths = wc.lde_height, wc.widths
    dg, nd = _C.c_void_p(), _C.c_uint64()
    check(L.msgpu_pdata_digests(wc.local.h, _C.byref(dg), _C.byref(nd)))
    nd = int(nd.value)
    if rank == 0:
        blocks = [wc.lde_block] + [ctx.malloc(H * widths[r] * 8) for r in range(1, world)]
        parts = [dg.value] + [ctx.malloc(nd * 32) for r in range(1, world)]
        gathers = [(r, blocks[r], parts[r]) for r in range(1, world)]
    else:
        gathers = [(rank, wc.lde_block, dg.value)]
    for r, block_ptr, part_ptr in gathers:  # rank r's LDE block and digest layer -> rank 0
        comm.sendrecv_dev(block_ptr, H * widths[r] * 8, r, 0)
        comm.sendrecv_dev(part_ptr, nd * 32, r, 0)
    t.append(time.perf_counter())
    if rank == 0:
        pd, r32 = _C.c_void_p(), np.zeros(32, dtype=np.uint8)
        ba = (_C.c_void_p * world)(*blocks)
        wa = (_C.c_uint64 * world)(*widths)
        pa = (_C.c_void_p * world)(*parts)
        check(L.msgpu_pdata_from_parts(ctx.h, world, ba, wa, H, world, pa, _C.byref(pd), r32.ctypes.data_as(_C.c_void_p)))
        for r in range(1, world):
            ctx.free(blocks[r])
            ctx.free(parts[r])
        if bytes(r32) != root:
            L.msgpu_pdata_free(pd)
            raise RuntimeError("assembled commitment differs from the sharded one")
    ctx.free(wc.lde_block)
    wc.lde_block = None
    wc.free()  # the row shard and its subtree are not needed any more: on rank 0 the assembled prover data serves the openings
    t.append(time.perf_counter())
    proof = prover.prove_precommitted(pd, [H >> log_blowup], claims) if rank == 0 else None
    t.append(time.perf_counter())
    if timings is not None:
        names = ["commit_sharded", "gather"] + (["assemble", "prove_rest"] if rank == 0 else [])
        for k, name in enumerate(names):
            timings[name] = (t[k + 1] - t[k]) * 1e3
    return proof
