"""The row-sharded prover over PEER MEMORY (multi_stark_b200/csrc/peer.cu): one rank per GPU over NCCL, matrices exchanged by
this library's kernels through CUDA-IPC windows (row blocks pushed into the owners' column blocks, row shards assembled from the
peers' LDE column blocks by the leaf-hash pass, subtree roots stored into every peer, flag barriers in peer memory). Needs at
least two GPUs: skipped on a single-GPU box, where tests/test_gpu_rowshard.py covers the same protocol over gloo and
tests/test_gpu_merkle.py::test_commit_from_column_blocks the assembling leaf kernels. The proof must be byte-identical to the
single-GPU proof, with peer memory and (MSGPU_P2P=0) with the NCCL exchange."""
import pytest

from tests.test_gpu_dist_prove import run_world

pytestmark = pytest.mark.gpu


def _gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


CASES = [
    # world, kind, log_heights, params, extra environment
    (2, "u32_add", [12], dict(log_blowup=1, num_queries=20), {}),
    (2, "u32_add", [12], dict(log_blowup=1, num_queries=20), {"MSGPU_P2P": "0"}),             # the same over NCCL collectives
    (2, "multi:5", [13, 13, 13, 12, 11], dict(log_blowup=1, num_queries=10), {}),               # several assembled matrices per height
    (2, "multi:3", [14, 12, 13], dict(log_blowup=1, num_queries=10), {"MSGPU_PEER_WINDOW_MB": "1"}),  # the heap grows mid-proof
    (2, "wide:16", [12], dict(log_blowup=2, num_queries=10), {}),                               # narrow stage-2 trace split too
    (4, "u32_add", [13], dict(log_blowup=1, num_queries=15), {}),                               # next rows fetched from another shard
    (4, "multi:3", [14, 12, 13], dict(log_blowup=1, num_queries=10), {}),
    (8, "multi:3", [15, 13, 14], dict(log_blowup=1, num_queries=10), {}),
]


@pytest.mark.parametrize("world,kind,log_heights,params,env", CASES)
def test_peer_memory_proof_is_byte_identical(tmp_path, world, kind, log_heights, params, env):
    if _gpus() < world:
        pytest.skip("needs %d GPUs" % world)
    proofs, single, infos = run_world(tmp_path, world, kind, log_heights, "rowshard", params, backend="nccl", extra_env=env)
    for r in range(world):
        assert proofs[r] == single, "rank %d's proof differs from the single-GPU proof" % r
    assert all(i["bytes_dev"] > 0 for i in infos)


# ---- the peer-memory ABI on ONE GPU: N ranks inside this process ---------------------------------------------------------------
# Every "rank" is its own context (own stream) with its own window on device 0; the windows are opened with
# msgpu_peers_segment_open_local instead of CUDA IPC. The test drives the protocol of RowShardBackend::commit_blocks through the C
# ABI -- push row blocks into the owners' column blocks, flag barrier, column-local LDE, barrier, leaf pass that assembles the row
# shard from every rank's LDE column block, subtree roots into the ring, barrier, top tree -- phase by phase over all ranks
# (a barrier only completes once every rank has enqueued it), and checks root and shards against the single-GPU commit.
import ctypes as C  # noqa: E402

import numpy as np  # noqa: E402


def _col_split(w, n):
    base, rem = divmod(w, n)
    out, c = [], 0
    for e in range(n):
        wd = base + (1 if e < rem else 0)
        out.append((c, wd))
        c += wd
    return out


@pytest.mark.parametrize("world,log_n,w,lb", [(2, 12, 14, 1), (4, 12, 26, 1), (8, 12, 14, 1), (4, 11, 2, 2), (8, 13, 3, 1)])
def test_peer_push_and_root_ring_in_process_ranks(world, log_n, w, lb):
    import multi_stark_b200 as ms
    from multi_stark_b200._ffi import check
    from tests import _oracle as orc
    n, N = 1 << log_n, world
    H, nb, Ls = n << lb, n // world, (n << lb) // world
    wmax = -(-w // N)
    rng = np.random.default_rng(7 * world + w)
    m = orc.rand_matrix(rng, n, w)
    ctxs = [ms.GpuContext(0) for _ in range(N)]
    L = ctxs[0].L
    # the single-GPU commitment to compare with
    pcs0 = ms.GpuPcs(ctxs[0], lb)
    want_root, want_pd = pcs0.commit([m])
    want_lde = want_pd.read_rows(0)
    want_pd.free()
    peers, segs = [], []
    window = 1 << 24
    for r in range(N):
        p = C.c_void_p()
        check(L.msgpu_peers_create(ctxs[r].h, r, N, C.byref(p)))
        handle = (C.c_uint8 * 64)()
        check(L.msgpu_peers_segment_create(p, window, handle))
        peers.append(p)
    # Warm every context up with the shapes used below (NTT tables, arena segments, kernel attributes): a device allocation
    # between two launches keeps kernels of different streams from overlapping, and the flag barriers of the in-process ranks
    # must overlap. (Separate processes -- the real deployment -- do not share this constraint.)
    split = _col_split(w, N)
    for r in range(N):
        wd = max(split[r][1], 1)
        a = ctxs[r].upload(np.ascontiguousarray(m[:, :wd]))
        b = ctxs[r].malloc(H * wd * 8)
        check(L.msgpu_coset_lde_batch_bitrev_dev(ctxs[r].h, C.c_void_p(a), n, wd, lb, 7, C.c_void_p(b)))
        sh = ctxs[r].upload(np.ascontiguousarray(want_lde[:Ls]))
        sh2 = ctxs[r].malloc(Ls * w * 8)
        rr = ctxs[r].upload(np.ascontiguousarray(m[:nb]))
        _, pdw = ms.GpuPcs(ctxs[r], lb).commit_ldes([(sh, Ls, w)])
        pdw.free()
        for q in (a, b, sh, sh2, rr):
            ctxs[r].free(q)
        ctxs[r].sync()
    bases = (C.c_void_p * N)(*[L.msgpu_peers_ptr(peers[r], 0, 0, r) for r in range(N)])
    for r in range(N):
        check(L.msgpu_peers_segment_open_local(peers[r], bases))
    try:
        # identical allocation sequences on every rank -> identical (segment, offset)
        blocks = []
        for r in range(N):
            seg, off = C.c_uint32(), C.c_uint64()
            check(L.msgpu_peers_alloc(peers[r], n * wmax * 8, C.byref(seg), C.byref(off)))
            col = (seg.value, off.value)
            check(L.msgpu_peers_alloc(peers[r], H * wmax * 8, C.byref(seg), C.byref(off)))
            blocks.append((col, (seg.value, off.value)))
        assert all(b == blocks[0] for b in blocks)
        (cseg, coff), (lseg, loff) = blocks[0]
        # phase 1: upload the row block, push it into every owner's column block, barrier
        row_dev = []
        for r in range(N):
            d = ctxs[r].upload(np.ascontiguousarray(m[r * nb:(r + 1) * nb]))
            row_dev.append(d)
            check(L.msgpu_peers_pack_push(peers[r], C.c_void_p(d), nb, w, cseg, coff))
            check(L.msgpu_peers_barrier(peers[r]))
        # phase 2: column-local LDE into the LDE column block, barrier
        for r in range(N):
            wd = split[r][1]
            if wd:
                check(L.msgpu_coset_lde_batch_bitrev_dev(ctxs[r].h, C.c_void_p(L.msgpu_peers_ptr(peers[r], cseg, coff, r)), n, wd, lb, 7,
                                                         C.c_void_p(L.msgpu_peers_ptr(peers[r], lseg, loff, r))))
            check(L.msgpu_peers_barrier(peers[r]))
        # phase 3: the leaf pass assembles rank r's row shard from every rank's LDE column block; subtree root -> ring; barrier
        pds, shards, gathered = [], [], []
        for r in range(N):
            shard = ctxs[r].malloc(Ls * w * 8)
            shards.append(shard)
            blks = [(L.msgpu_peers_ptr(peers[r], lseg, loff, e) + r * Ls * split[e][1] * 8, split[e][1]) for e in range(N)]
            root_r, pd = ms.GpuPcs(ctxs[r], lb).commit_ldes_blocks([(shard, Ls, w, blks)])
            pds.append(pd)
            dg, nd = C.c_void_p(), C.c_uint64()
            check(L.msgpu_pdata_digests(pd.h, C.byref(dg), C.byref(nd)))
            g = C.c_void_p()
            check(L.msgpu_peers_put_root(peers[r], C.c_void_p(dg.value + (nd.value - 1) * 32), C.byref(g)))
            gathered.append(g)
            check(L.msgpu_peers_barrier(peers[r]))
        # phase 4: the top levels over the gathered subtree roots, on every rank
        roots = []
        for r in range(N):
            hh = (C.c_uint64 * 1)(N)
            pp = (C.c_void_p * 1)(gathered[r].value)
            top = C.c_void_p()
            root = np.zeros(32, dtype=np.uint8)
            check(L.msgpu_tree_from_digests(ctxs[r].h, 1, hh, pp, C.byref(top), root.ctypes.data_as(C.c_void_p)))
            L.msgpu_pdata_free(top)
            roots.append(bytes(root))
        # The ranks of this test share one device and one process: their flag barriers only complete if the kernels of the N
        # streams overlap. A barrier that timed out says the box serialised them (nothing about the code under test): skip.
        timed_out = [r for r in range(N) if L.msgpu_peers_check(peers[r]) != 0]
        if timed_out:
            pytest.skip("in-process ranks %s could not overlap their barrier kernels on this device" % timed_out)
        for r in range(N):
            assert roots[r] == bytes(want_root), "rank %d: root differs from the single-GPU commitment" % r
            got = ctxs[r].download(shards[r], (Ls, w))
            assert np.array_equal(got, want_lde[r * Ls:(r + 1) * Ls]), "rank %d: row shard differs from the single-GPU LDE" % r
        for r in range(N):
            pds[r].free()
            ctxs[r].free(shards[r])
            ctxs[r].free(row_dev[r])
            check(L.msgpu_peers_free_block(peers[r], cseg, coff))
            check(L.msgpu_peers_free_block(peers[r], lseg, loff))
    finally:
        for r in range(N):
            ctxs[r].sync()
        for r in range(N):
            L.msgpu_peers_destroy(peers[r])
        for c in ctxs:
            c.close()
