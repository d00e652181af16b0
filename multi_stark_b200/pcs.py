"""Host-side mirror of the reference's DFT / PCS / MMCS objects over libmsgpu.

Names and argument meaning follow the trait methods the reference calls (SURVEY.md section 8b):
  GpuDft.dft_batch / coset_lde_batch            <- TwoAdicSubgroupDft (src/prover.rs:440,650,716)
  GpuPcs.commit / commit_ldes / get_evaluations_on_domain / natural_domain_for_degree
                                                 <- Pcs (src/prover.rs:346-351,419,454-468,526)
  GpuMmcs.commit / open_batch / verify-free      <- Mmcs (src/types.rs:82-84,199-207)
Matrices are numpy uint64 arrays of canonical Goldilocks values, shape (rows, cols)."""
import ctypes as C

import numpy as np

from . import _ffi
from ._ffi import check

GENERATOR = 7


def _as_matrix(m):
    a = np.ascontiguousarray(m, dtype=np.uint64)
    if a.ndim != 2:
        raise ValueError("matrix must be 2-D (rows, cols)")
    return a


class GpuContext:
    """One CUDA device + stream. `stream` may be an existing cudaStream_t handle (int), e.g.
    torch.cuda.current_stream().cuda_stream, so that the caller's CUDA events bracket our launches."""

    def __init__(self, device=0, stream=None):
        self.L = _ffi.lib()
        h = C.c_void_p()
        check(self.L.msgpu_ctx_create(int(device), C.c_void_p(stream) if stream else None, C.byref(h)))
        self.h = h
        self.device = device
        self._pinned = []

    def close(self):
        if getattr(self, "h", None):
            for p in self._pinned:
                self.L.msgpu_host_free(p)
            self._pinned = []
            self.L.msgpu_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        check(self.L.msgpu_sync(self.h))

    @property
    def launches(self):
        return int(self.L.msgpu_launch_count(self.h))

    @property
    def stream(self):
        return self.L.msgpu_stream(self.h)

    def profile_begin(self):
        check(self.L.msgpu_profile_begin(self.h))

    def profile_end(self):
        import json
        buf = C.create_string_buffer(1 << 16)
        check(self.L.msgpu_profile_end(self.h, buf, len(buf)))
        return json.loads(buf.value.decode())

    # raw device buffers (uint64 elements)
    def malloc(self, nbytes):
        p = C.c_void_p()
        check(self.L.msgpu_malloc(self.h, nbytes, C.byref(p)))
        return p.value

    def free(self, ptr):
        check(self.L.msgpu_free(self.h, C.c_void_p(ptr)))

    def measure_int_peak(self):
        """msgpu_measure_int_peak: {"alu", "imad", "mixed"} in G thread-instructions / s."""
        out = (C.c_double * 3)()
        check(self.L.msgpu_measure_int_peak(self.h, out))
        return {"alu": out[0], "imad": out[1], "mixed": out[2]}

    def pinned_empty(self, shape, dtype=np.uint64):
        """numpy array over page-locked host memory (msgpu_host_alloc): H2D copies from it run at full PCIe rate.
        The memory lives until the context is closed."""
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        check(self.L.msgpu_host_alloc(max(n, 8), C.byref(p)))
        self._pinned.append(p)
        buf = (C.c_uint8 * max(n, 8)).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def pinned_copy(self, arr):
        out = self.pinned_empty(arr.shape, arr.dtype)
        out[...] = arr
        return out

    def blake3_hash(self, data):
        """msgpu_blake3_hash: BLAKE3-256 of a host byte string, hashed on the device (the transcript's long flushes)."""
        buf = np.frombuffer(bytes(data), dtype=np.uint8) if len(data) else np.zeros(1, dtype=np.uint8)
        out = np.zeros(32, dtype=np.uint8)
        check(self.L.msgpu_blake3_hash(self.h, buf.ctypes.data_as(C.c_void_p), len(data), out.ctypes.data_as(C.c_void_p)))
        return bytes(out)

    def upload_canonical(self, arr):
        """msgpu_upload_canonical: H2D copy that rejects values >= p."""
        a = np.ascontiguousarray(arr, dtype=np.uint64)
        p = self.malloc(max(a.nbytes, 8))
        try:
            check(self.L.msgpu_upload_canonical(self.h, C.c_void_p(p), a.ctypes.data_as(C.c_void_p), a.size))
        except Exception:
            self.free(p)
            raise
        return p

    def upload(self, arr):
        a = np.ascontiguousarray(arr)
        p = self.malloc(max(a.nbytes, 8))
        if a.nbytes:
            check(self.L.msgpu_memcpy_h2d(self.h, C.c_void_p(p), a.ctypes.data_as(C.c_void_p), a.nbytes))
        return p

    def download(self, ptr, shape, dtype=np.uint64):
        out = np.empty(shape, dtype=dtype)
        if out.nbytes:
            check(self.L.msgpu_memcpy_d2h(self.h, out.ctypes.data_as(C.c_void_p), C.c_void_p(ptr), out.nbytes))
        return out


class GpuDft:
    """`TwoAdicSubgroupDft<Goldilocks>` slot (reference `type Dft`, src/types.rs:200)."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.L = ctx.L

    def _call(self, fn, m, out_rows, *extra):
        a = _as_matrix(m)
        out = np.empty((out_rows, a.shape[1]), dtype=np.uint64)
        check(fn(self.ctx.h, a.ctypes.data_as(C.c_void_p), a.shape[0], a.shape[1], *extra, out.ctypes.data_as(C.c_void_p)))
        return out

    def dft_batch(self, m):
        return self._call(self.L.msgpu_dft_batch, m, len(m))

    def dft_batch_bitrev(self, m):
        """dft_batch(m).bit_reverse_rows() (src/prover.rs:650,716)."""
        return self._call(self.L.msgpu_dft_batch_bitrev, m, len(m))

    def idft_batch(self, m):
        return self._call(self.L.msgpu_idft_batch, m, len(m))

    def coset_lde_batch_bitrev(self, m, added_bits, shift=GENERATOR):
        """coset_lde_batch(m, added_bits, shift).bit_reverse_rows() (src/prover.rs:681-692)."""
        return self._call(self.L.msgpu_coset_lde_batch_bitrev, m, len(m) << added_bits, added_bits, shift)

    def lde_from_shifted_coefficients(self, m, added_bits):
        """src/prover.rs:709-717."""
        return self._call(self.L.msgpu_lde_from_shifted_coefficients, m, len(m) << added_bits, added_bits)


class ProverData:
    """Device-resident `ProverData`: committed matrices (bit-reversed rows) + digest layers."""

    def __init__(self, ctx, handle, root):
        self.ctx = ctx
        self.L = ctx.L
        self.h = handle
        self.root = root

    def free(self):
        if getattr(self, "h", None):
            self.L.msgpu_pdata_free(self.h)
            self.h = None

    def __del__(self):
        try:
            if self.ctx.h:
                self.free()
        except Exception:
            pass

    @property
    def num_matrices(self):
        return int(self.L.msgpu_pdata_num_matrices(self.h))

    def matrix_info(self, idx):
        p = C.c_void_p()
        r = C.c_uint64()
        c = C.c_uint64()
        check(self.L.msgpu_pdata_matrix(self.h, idx, C.byref(p), C.byref(r), C.byref(c)))
        return p.value, int(r.value), int(c.value)

    def read_rows(self, idx, row0=0, nrows=None):
        _, rows, cols = self.matrix_info(idx)
        if nrows is None:
            nrows = rows - row0
        out = np.empty((nrows, cols), dtype=np.uint64)
        check(self.L.msgpu_pdata_read_rows(self.ctx.h, self.h, idx, row0, nrows, out.ctypes.data_as(C.c_void_p)))
        return out

    def layers(self):
        out = []
        for i in range(int(self.L.msgpu_pdata_num_layers(self.h))):
            ln = int(self.L.msgpu_pdata_layer_len(self.h, i))
            buf = np.empty((ln, 32), dtype=np.uint8)
            check(self.L.msgpu_pdata_read_layer(self.ctx.h, self.h, i, buf.ctypes.data_as(C.c_void_p)))
            out.append(buf)
        return out

    def open_batch(self, indices):
        """Mmcs::open_batch for many indices: returns (opened[n_idx, sum widths], proofs[n_idx, depth, 32])."""
        idx = np.ascontiguousarray(indices, dtype=np.uint64)
        infos = [self.matrix_info(i) for i in range(self.num_matrices)]
        tw = sum(c for _, _, c in infos)
        depth = max(r for _, r, _ in infos).bit_length() - 1
        opened = np.zeros((len(idx), tw), dtype=np.uint64)
        proofs = np.zeros((len(idx), depth, 32), dtype=np.uint8)
        check(self.L.msgpu_open_batch(self.ctx.h, self.h, idx.ctypes.data_as(C.c_void_p), len(idx),
                                      opened.ctypes.data_as(C.c_void_p), proofs.ctypes.data_as(C.c_void_p)))
        return opened, proofs


def _mat_args(mats):
    n = len(mats)
    ptrs = (C.c_void_p * n)(*[m.ctypes.data for m in mats])
    hs = (C.c_uint64 * n)(*[m.shape[0] for m in mats])
    ws = (C.c_uint64 * n)(*[m.shape[1] for m in mats])
    return ptrs, hs, ws


class GpuMmcs:
    """`MerkleTreeMmcs<..Blake3..>` slot (reference `type Mmcs`, src/types.rs:82-84; `new_mmcs` :202-207)."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.L = ctx.L

    def commit(self, mats):
        mats = [_as_matrix(m) for m in mats]
        ptrs, hs, ws = _mat_args(mats)
        h = C.c_void_p()
        root = np.zeros(32, dtype=np.uint8)
        check(self.L.msgpu_mmcs_commit(self.ctx.h, ptrs, hs, ws, len(mats), C.byref(h), root.ctypes.data_as(C.c_void_p)))
        return root, ProverData(self.ctx, h, root)


class GpuPcs:
    """`TwoAdicFriPcs<Val, Dft, Mmcs, ExtMmcs>` slot (reference `type Pcs`, src/types.rs:85;
    `new_pcs` :209-223), commitment side."""

    ZK = False  # reference asserts !Pcs::ZK before commit_ldes (src/prover.rs:522-525)

    def __init__(self, ctx, log_blowup, cap_height=0):
        if cap_height != 0:
            raise ValueError("cap_height must be 0 (the only value the reference uses)")
        self.ctx = ctx
        self.L = ctx.L
        self.log_blowup = log_blowup

    @staticmethod
    def natural_domain_for_degree(degree):
        """(log_n, shift) of the two-adic coset H_n with shift 1."""
        assert degree & (degree - 1) == 0
        return degree.bit_length() - 1, 1

    def commit(self, evaluations):
        """`evaluations`: list of matrices over their natural domains. Returns (root, ProverData)."""
        mats = [_as_matrix(m) for m in evaluations]
        ptrs, hs, ws = _mat_args(mats)
        h = C.c_void_p()
        root = np.zeros(32, dtype=np.uint8)
        check(self.L.msgpu_commit(self.ctx.h, ptrs, hs, ws, len(mats), self.log_blowup, C.byref(h),
                                  root.ctypes.data_as(C.c_void_p)))
        return root, ProverData(self.ctx, h, root)

    def upload_begin(self, evaluations):
        """`msgpu_upload_begin`: start the host-to-device copies of the matrices on the context's copy stream and return at
        once; pass the handle to commit_upload. The host arrays (pinned memory for a real overlap) must stay alive until then.
        Calling upload_begin for commitment k + 1 BEFORE commit_upload of commitment k puts the next transfer under this
        commitment's kernels."""
        mats = [_as_matrix(m) for m in evaluations]
        ptrs, hs, ws = _mat_args(mats)
        up = C.c_void_p()
        check(self.L.msgpu_upload_begin(self.ctx.h, ptrs, hs, ws, len(mats), C.byref(up)))
        return (up, mats)

    def commit_upload(self, handle, verify_canonical=True):
        """`msgpu_commit_upload`: Pcs::commit of the matrices handed to upload_begin. Returns (root, ProverData)."""
        up, _keep = handle
        h = C.c_void_p()
        root = np.zeros(32, dtype=np.uint8)
        check(self.L.msgpu_commit_upload(up, self.log_blowup, 1 if verify_canonical else 0, None, 0, C.byref(h),
                                         root.ctypes.data_as(C.c_void_p)))
        return root, ProverData(self.ctx, h, root)

    def upload_free(self, handle):
        self.L.msgpu_upload_free(handle[0])

    def commit_dev(self, ptrs_shapes):
        """Same with device-resident inputs: list of (device_ptr, rows, cols)."""
        n = len(ptrs_shapes)
        ptrs = (C.c_void_p * n)(*[p for p, _, _ in ptrs_shapes])
        hs = (C.c_uint64 * n)(*[r for _, r, _ in ptrs_shapes])
        ws = (C.c_uint64 * n)(*[c for _, _, c in ptrs_shapes])
        h = C.c_void_p()
        root = np.zeros(32, dtype=np.uint8)
        check(self.L.msgpu_commit_dev(self.ctx.h, ptrs, hs, ws, n, self.log_blowup, C.byref(h),
                                      root.ctypes.data_as(C.c_void_p)))
        return root, ProverData(self.ctx, h, root)

    def commit_ldes(self, ptrs_shapes, take_ownership=False):
        """Pcs::commit_ldes (src/prover.rs:526) on device-resident LDEs: list of (device_ptr, rows, cols)."""
        n = len(ptrs_shapes)
        ptrs = (C.c_void_p * n)(*[p for p, _, _ in ptrs_shapes])
        hs = (C.c_uint64 * n)(*[r for _, r, _ in ptrs_shapes])
        ws = (C.c_uint64 * n)(*[c for _, _, c in ptrs_shapes])
        h = C.c_void_p()
        root = np.zeros(32, dtype=np.uint8)
        check(self.L.msgpu_commit_ldes_dev(self.ctx.h, ptrs, hs, ws, n, 1 if take_ownership else 0, C.byref(h),
                                           root.ctypes.data_as(C.c_void_p)))
        return root, ProverData(self.ctx, h, root)

    def commit_ldes_blocks(self, mats):
        """`commit_ldes` where some LDEs still exist as COLUMN BLOCKS (msgpu_commit_ldes_blocks_dev): mats = list of
        (dst_device_ptr, rows, cols, blocks) with blocks = None (the matrix is already at dst) or a list of
        (block_device_ptr, block_cols) -- dense rows x block_cols matrices in column order, possibly in another GPU's memory.
        Such a matrix is written to dst by the pass that hashes its rows. Returns (root, ProverData)."""
        n = len(mats)
        nb = max([len(b) for _, _, _, b in mats if b] or [0])
        ptrs = (C.c_void_p * n)(*[p for p, _, _, _ in mats])
        hs = (C.c_uint64 * n)(*[r for _, r, _, _ in mats])
        ws = (C.c_uint64 * n)(*[c for _, _, c, _ in mats])
        bp = (C.c_void_p * max(n * nb, 1))()
        bw = (C.c_uint64 * max(n * nb, 1))()
        for i, (_, _, _, blocks) in enumerate(mats):
            for b, (ptr, cols) in enumerate(blocks or []):
                bp[i * nb + b] = ptr
                bw[i * nb + b] = cols
        h = C.c_void_p()
        root = np.zeros(32, dtype=np.uint8)
        check(self.L.msgpu_commit_ldes_blocks_dev(self.ctx.h, ptrs, hs, ws, n, nb, bp if nb else None, bw if nb else None, 0, C.byref(h),
                                                  root.ctypes.data_as(C.c_void_p)))
        return root, ProverData(self.ctx, h, root)

    def get_evaluations_on_domain(self, pdata, idx, log_quotient_size):
        """View of the committed LDE on the coset GENERATOR * H_{2^log_quotient_size}: the first
        2^log_quotient_size stored rows, bit-reversed (src/prover.rs:454-468; SURVEY A.3 item 3).
        Returns (device_ptr, rows, cols); no copy."""
        ptr, rows, cols = pdata.matrix_info(idx)
        nq = 1 << log_quotient_size
        if nq > rows:
            raise ValueError("quotient domain larger than the committed LDE (needs quotient_degree <= blowup)")
        return ptr, nq, cols


class Challenger:
    """The reference's transcript object (`config.initialise_challenger()`, src/types.rs:118-130,152-154) for standalone
    PCS use as in examples/pcs_example.rs:77-79."""

    def __init__(self, log_blowup=1, log_final_poly_len=0, max_log_arity=1, num_queries=100, commit_pow_bits=0, query_pow_bits=0):
        self.H = _ffi.host_lib()
        self.params = dict(log_blowup=log_blowup, log_final_poly_len=log_final_poly_len, max_log_arity=max_log_arity,
                           num_queries=num_queries, commit_pow_bits=commit_pow_bits, query_pow_bits=query_pow_bits)
        self.h = self.H.msh_challenger_create(log_blowup, log_final_poly_len, max_log_arity, num_queries, commit_pow_bits,
                                              query_pow_bits)

    def observe(self, commitment):
        d = np.frombuffer(bytes(commitment), dtype=np.uint8).copy()
        assert d.size == 32
        self.H.msh_challenger_observe_digest(self.h, d.ctypes.data_as(C.c_void_p))

    def observe_values(self, values):
        v = np.ascontiguousarray(values, dtype=np.uint64)
        self.H.msh_challenger_observe_values(self.h, v.ctypes.data_as(C.c_void_p), v.size)

    def sample_algebra_element(self):
        out = np.zeros(2, dtype=np.uint64)
        self.H.msh_challenger_sample_ext(self.h, out.ctypes.data_as(C.c_void_p))
        return (int(out[0]), int(out[1]))

    def close(self):
        if getattr(self, "h", None):
            self.H.msh_challenger_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def pcs_open(ctx, rounds, challenger):
    """`Pcs::open(rounds, &mut challenger)` (src/prover.rs:580, examples/pcs_example.rs:85-90).
    rounds: list of (ProverData, points) with points[m] = list of extension points (c0, c1) for matrix m.
    Returns (bytes of opened values + FRI proof, per-phase ms)."""
    H = _ffi.host_lib()
    n = len(rounds)
    pds = (C.c_void_p * n)(*[pd.h for pd, _ in rounds])
    npts, pts = [], []
    for pd, points in rounds:
        assert len(points) == pd.num_matrices
        for mp in points:
            npts.append(len(mp))
            for z in mp:
                pts += [int(z[0]), int(z[1])]
    npts_a = np.array(npts, dtype=np.uint64)
    pts_a = np.array(pts if pts else [0], dtype=np.uint64)
    out, ln = C.c_void_p(), C.c_uint64()
    ms5 = (C.c_double * 5)()
    rc = H.msh_pcs_open(ctx.h, challenger.h, n, pds, npts_a.ctypes.data_as(_ffi.c_u64p), pts_a.ctypes.data_as(_ffi.c_u64p),
                        C.byref(out), C.byref(ln), ms5)
    if rc != 0:
        raise _ffi.host_error(rc)
    data = C.string_at(out.value, ln.value)
    H.msh_bytes_free(out)
    return data, dict(zip(["evaluate", "reduce", "commit_phase", "final_poly", "queries"], ms5))
